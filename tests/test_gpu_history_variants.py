"""Every instantiation of the history kernel launches with a shared-memory pad above the 48 KB a
kernel gets without the dynamic shared-memory attribute (option history_smem_pad), and the pad
changes no history. For each tally configuration, with and without the fast divisions, the
counts, the bank after every timestep and the per-particle counters are bit-identical to the
unpadded run, and the energy tally and the flux agree to 1e-10 per cell (atomic order)."""
import numpy as np
import pytest

from neutral_b200.decks import build_problem
from neutral_b200.host import NB200_BAD_OPTION, Simulation
from test_gpu_parity import TALLY_RTOL

pytestmark = pytest.mark.gpu

PAD = 65536
B = 4


def _config(kind, e0):
    """Simulation keyword arguments and options of one tally configuration."""
    edges = np.geomspace(1.0e-3, 2.0 * e0, 9)
    return {
        "plain": ({}, {}),
        "prereduce": ({}, dict(tally_prereduce=1)),
        "batched": (dict(tally_batches=B), {}),
        "flux": (dict(flux_tally=True), {}),
        "batched_flux": (dict(flux_tally=True, tally_batches=B), {}),
        "group_flux": (dict(flux_groups=edges), {}),
        "batched_group_flux": (dict(flux_groups=edges, tally_batches=B,
                                    group_flux_batches=True), {}),
    }[kind]


KINDS = ["plain", "prereduce", "batched", "flux", "batched_flux", "group_flux",
         "batched_group_flux"]
# prereduce has one variant, with the fast divisions
VARIANTS = [(k, f) for k in KINDS for f in (1, 0) if not (k == "prereduce" and f == 0)]


@pytest.fixture
def set_options(gpu_lib):
    """Sets process-wide options; every option set is restored to its old value afterwards."""
    old = {}

    def set_(**kw):
        for k, v in kw.items():
            prev = gpu_lib.nb200_set_option(k.encode(), v)
            assert prev != NB200_BAD_OPTION, k
            old.setdefault(k, prev)

    yield set_
    for k, v in old.items():
        gpu_lib.nb200_set_option(k.encode(), v)


def _close(got, want):
    """Relative 1e-10 above an absolute floor of the smallest normal double, as the group flux
    tests compare."""
    return bool(np.all(np.abs(got - want) <= TALLY_RTOL * np.maximum(np.abs(got), np.abs(want)) +
                       np.finfo(np.float64).tiny))


def _run(prob, kw):
    sim = Simulation(prob, **kw)
    sim.inject()
    counts, banks = [], []
    for tt in range(1, prob.deck.iterations + 1):
        r = sim.step(tt)
        counts.append((r.facets, r.collisions, r.processed, r.census, r.deaths))
        banks.append(sim.bank_to_host())
    out = dict(counts=counts, banks=banks, counters=sim.counters_to_host(),
               tally=sim.tally_to_host(),
               flux=sim.flux.download() if sim.flux is not None else None)
    sim.free()
    return out


@pytest.mark.parametrize("kind,fast_div", VARIANTS)
def test_smem_pad_above_48k(gpu_lib, set_options, kind, fast_div):
    prob = build_problem("csp_small")
    kw, opts = _config(kind, prob.deck.initial_energy)
    set_options(fast_div=fast_div, **opts)
    set_options(history_smem_pad=0)
    want = _run(prob, kw)
    set_options(history_smem_pad=PAD)
    got = _run(prob, kw)
    assert got["counts"] == want["counts"]
    assert sum(r[1] for r in got["counts"]) > 0
    for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
        diff = a.bit_equal(b)
        assert sum(diff.values()) == 0, (tt, diff)
    assert np.array_equal(got["counters"], want["counters"])
    assert np.count_nonzero(want["tally"]) > 0
    assert _close(got["tally"], want["tally"])
    if want["flux"] is not None:
        assert np.count_nonzero(want["flux"]) > 0
        assert _close(got["flux"], want["flux"])
