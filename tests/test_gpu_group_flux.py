"""The energy-group flux tally on the GPU (nb200_bank_set_group_flux_tally): attaching a group
flux changes no history and no energy deposit; every group equals the reference's after every
timestep (the oracle port's timestep with a group-resolved flux output,
tests/group_flux_reference.c) for edges covering every energy, a log grid, narrow groups that
most scatters leave, and edges that leave energies out; summed over covering groups it is the
plain flux; nothing outside the array is written; a group-flux bank steps beside plain-flux and
no-flux banks; detach, replacement and deallocate_data; and every refusal with its message."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import SMALL_DECKS
from flux_reference import flux_reference
from group_flux_reference import group_flux_reference
from neutral_b200.decks import build_problem
from neutral_b200.host import NB200_BAD_OPTION, DeviceArray, Simulation, _soa_p
from test_gpu_parity import DEFAULTS, MODES, TALLY_RTOL, tally_close
from test_group_flux_cpu import COVERING, edge_sets
from variants import VARIANTS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem(name):
    return VARIANTS[name]() if name in VARIANTS else build_problem(name)


def _set_mode(lib, name):
    for k, v in MODES[name].items():
        assert lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION


def _restore(lib):
    for k, v in DEFAULTS.items():
        lib.nb200_set_option(k.encode(), v)


@pytest.fixture(params=["pipeline", "pipeline-ieee-div"])
def kernel_mode(request, gpu_lib):
    _set_mode(gpu_lib, request.param)
    yield request.param
    _restore(gpu_lib)


def _reference(port, prob, edges, start=1):
    """The group flux after every timestep, (G, ncells) each, from the port's injected bank;
    timesteps before `start` deposit nothing."""
    d = prob.deck
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    gflux = np.zeros((edges.size - 1) * d.nx * d.ny)
    out = []
    for tt in range(1, d.iterations + 1):
        kw = dict(gflux=gflux, edges=edges) if tt >= start else {}
        group_flux_reference().step(prob, bank, tt, tally, **kw)
        out.append(gflux.reshape(edges.size - 1, -1).copy())
    return out


def _groups_close(got, want):
    """Every group against the reference with the flux tests' relative tolerance, above an
    absolute floor of the smallest normal double. Below it a deposit keeps only a subnormal's
    absolute precision: on absorb_scaled_csp (p_absorb = 0.75) weights underflow through
    hundreds of absorptions, and a low-energy group of a cell can hold nothing but subnormal
    deposits. There the kernel's flush of a summed collision flux and the reference's deposit of
    every segment round apart by some hundred subnormal ulps, which no relative tolerance
    admits."""
    a, b = np.ravel(got), np.ravel(want)
    return bool(np.all(np.abs(a - b) <= TALLY_RTOL * np.maximum(np.abs(a), np.abs(b)) +
                       np.finfo(np.float64).tiny))


def _run(prob, pipelined=False, edges=None, flux=False, ref=None):
    """Per-timestep counts, bank after every timestep (step by step) or at the end (pipelined),
    per-particle counters, the energy tally and the group flux (or plain flux). With `ref` (the
    reference's group flux per timestep), the group flux is checked after every timestep."""
    sim = Simulation(prob, flux_groups=edges, flux_tally=flux)
    sim.inject()
    d = prob.deck
    counts, banks = [], []
    if pipelined:
        counts = [(r.facets, r.collisions, r.processed, r.census, r.deaths)
                  for r in sim.run_pipelined(depth=3)]
        banks.append(sim.bank_to_host())
        if ref is not None:
            assert _groups_close(sim.group_flux_to_host(), ref[-1])
    else:
        for tt in range(1, d.iterations + 1):
            r = sim.step(tt)
            counts.append((r.facets, r.collisions, r.processed, r.census, r.deaths))
            banks.append(sim.bank_to_host())
            if ref is not None:
                assert _groups_close(sim.group_flux_to_host(), ref[tt - 1]), tt
    out = dict(counts=counts, banks=banks, counters=sim.counters_to_host(),
               tally=sim.tally_to_host())
    if edges is not None:
        out["gflux"] = sim.group_flux_to_host().reshape(len(edges) - 1, -1)
    if flux:
        out["flux"] = sim.flux_to_host().ravel()
    sim.free()
    return out


def _same_histories(got, want):
    assert got["counts"] == want["counts"]
    for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
        diff = a.bit_equal(b)
        assert sum(diff.values()) == 0, (tt, diff)
    assert np.array_equal(got["counters"], want["counters"])
    assert tally_close(got["tally"], want["tally"])


@pytest.mark.parametrize("name", SMALL_DECKS + list(VARIANTS))
def test_histories_unchanged_and_groups_match_the_reference(gpu_lib, port, kernel_mode, name):
    """Bit-identical histories (counts, per-particle counters, all bank fields) and an energy
    tally within 1e-10 with a group flux attached; every group equals the reference's after
    every timestep, step by step and pipelined, for the four edge sets; over the covering sets
    the groups sum to a plain-flux run's flux."""
    prob = _problem(name)
    sets = edge_sets(prob.deck.initial_energy)
    refs = {key: _reference(port, prob, edges) for key, edges in sets.items()}
    for pipelined in (False, True):
        base = _run(prob, pipelined)
        plain = _run(prob, pipelined, flux=True)["flux"] if pipelined else None
        for key, edges in sets.items():
            got = _run(prob, pipelined, edges=edges, ref=refs[key])
            _same_histories(got, base)
            if key in COVERING:
                assert np.count_nonzero(got["gflux"]) > 0, key
                if plain is not None:
                    assert _groups_close(got["gflux"].sum(axis=0), plain), key


@pytest.mark.parametrize("name", ["csp_small", "mixed_small"])
def test_without_the_step_graph(gpu_lib, port, name):
    """The same with the timestep's calls issued one by one (step_graph=0)."""
    _set_mode(gpu_lib, "pipeline-calls")
    try:
        prob = _problem(name)
        base = _run(prob)
        for key in ("log8", "narrow32"):
            edges = edge_sets(prob.deck.initial_energy)[key]
            _same_histories(_run(prob, edges=edges, ref=_reference(port, prob, edges)), base)
    finally:
        _restore(gpu_lib)


def test_stream_lands_in_the_group_of_the_initial_energy(gpu_lib):
    """stream_small: all flux in the group holding 1e6 eV, the other groups exactly 0, and every
    timestep sums to v(E0) dt (as the plain flux does)."""
    prob = build_problem("stream_small")
    d = prob.deck
    edges = np.geomspace(1.0e-3, 1.0e8, 12)
    g0 = int(np.searchsorted(edges, d.initial_energy, side="right") - 1)
    sim = Simulation(prob, flux_groups=edges)
    plain = Simulation(prob, flux_tally=True)
    sim.inject()
    plain.inject()
    for tt in range(1, d.iterations + 1):
        before, pbefore = sim.group_flux_to_host().sum(), plain.flux_to_host().sum()
        sim.step(tt)
        plain.step(tt)
        s, ps = sim.group_flux_to_host().sum() - before, plain.flux_to_host().sum() - pbefore
        assert abs(s - ps) <= 1e-12 * ps, (tt, s, ps)
    g = sim.group_flux_to_host()
    assert tally_close(g[g0].ravel(), plain.flux_to_host().ravel())
    assert not np.any(np.delete(g, g0, axis=0))
    sim.free()
    plain.free()


GUARD = 1024  # doubles of sentinel on either side of the attached array


def test_nothing_outside_the_array_is_written(gpu_lib, port):
    """The array is attached inside a larger allocation whose guard cells hold a sentinel: after
    the deck, for narrow groups and for edges leaving energies out, the guards are untouched and
    the inside equals the reference."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    d = prob.deck
    ncells = d.nx * d.ny
    sentinel = np.float64(-1.2345e-300)
    for key in ("narrow32", "gaps", "log8"):
        edges = edge_sets(d.initial_energy)[key]
        G = edges.size - 1
        buf = DeviceArray(G * ncells + 2 * GUARD)
        host = np.zeros(G * ncells + 2 * GUARD)
        host[:GUARD] = host[-GUARD:] = sentinel
        buf.upload(host)
        sim = Simulation(prob)
        sim.inject()
        assert lib.nb200_bank_set_group_flux_tally(sim.bank, buf.ptr + 8 * GUARD, ncells,
                                                   edges.ctypes.data, G) == 0
        sim.run_pipelined()
        got = buf.download()
        assert np.array_equal(got[:GUARD].view(np.uint64), host[:GUARD].view(np.uint64)), key
        assert np.array_equal(got[-GUARD:].view(np.uint64), host[-GUARD:].view(np.uint64)), key
        assert _groups_close(got[GUARD:-GUARD].reshape(G, -1), _reference(port, prob, edges)[-1])
        sim.free()
        buf.free()


def test_group_plain_and_no_flux_banks_alternate(gpu_lib, port):
    """A group-flux bank, a plain-flux bank and a bank without flux, stepped in turn on one device
    (the step graph switches kernels every timestep): all three histories unchanged, each flux
    right."""
    prob = build_problem("csp_small", iterations=5)
    d = prob.deck
    edges = edge_sets(d.initial_energy)["narrow32"]
    ref = _reference(port, prob, edges)
    base = _run(prob)
    plain_ref = _run(prob, flux=True)["flux"]
    sims = [Simulation(prob, flux_groups=edges), Simulation(prob, flux_tally=True),
            Simulation(prob)]
    for s in sims:
        s.inject()
    for tt in range(1, d.iterations + 1):
        for s in sims:
            r = s.step(tt)
            assert (r.facets, r.collisions) == base["counts"][tt - 1][:2]
            assert sum(s.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
        assert _groups_close(sims[0].group_flux_to_host(), ref[tt - 1]), tt
    assert tally_close(sims[1].flux_to_host().ravel(), plain_ref)
    for s in sims:
        assert tally_close(s.tally_to_host(), base["tally"])
        s.free()


def _set_groups(lib, sim, arr, edges):
    if arr is None:
        return lib.nb200_bank_set_group_flux_tally(sim.bank, None, 0, None, 0)
    e = np.ascontiguousarray(edges, dtype=np.float64)
    return lib.nb200_bank_set_group_flux_tally(sim.bank, arr.ptr, arr.n // (e.size - 1),
                                               e.ctypes.data, e.size - 1)


def test_detach_replace_and_deallocate(gpu_lib, port):
    """After a null attach (through either call) the array stays bitwise untouched and the bank
    continues bit-identical; the plain call replaces a group flux and the group call a plain
    flux, each array then receiving exactly the later timesteps; deallocate_data detaches."""
    lib = gpu_lib
    prob = build_problem("csp_small", iterations=6)
    d = prob.deck
    n = d.nx * d.ny
    edges = edge_sets(d.initial_energy)["log8"]
    G = edges.size - 1
    base = _run(prob)
    ref = _reference(port, prob, edges)
    ref_from_5 = _reference(port, prob, edges, start=5)
    pb = port.inject(prob)
    ptally, plain_3_4 = np.zeros(n), np.zeros(n)
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, pb, tt, ptally, flux=plain_3_4 if tt in (3, 4) else None)

    sim = Simulation(prob, flux_groups=edges)
    sim.inject()
    sim.step(1)
    assert _groups_close(sim.group_flux_to_host(), ref[0])
    assert lib.nb200_bank_set_flux_tally(sim.bank, None, 0) == 0  # detach through the plain call
    frozen = sim.flux.download()
    plain = DeviceArray(n)
    again = DeviceArray(G * n)
    for tt in range(2, d.iterations + 1):
        if tt == 3:  # a plain flux from step 3 on
            assert lib.nb200_bank_set_flux_tally(sim.bank, plain.ptr, n) == 0
        if tt == 5:  # replaced by a group flux from step 5 on
            assert _set_groups(lib, sim, again, edges) == 0
        sim.step(tt)
        assert np.array_equal(sim.flux.download().view(np.uint64), frozen.view(np.uint64)), tt
        assert sum(sim.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
    assert tally_close(plain.download(), plain_3_4)
    assert _groups_close(again.download().reshape(G, -1), ref_from_5[-1])
    assert _set_groups(lib, sim, None, None) == 0  # detach through the group call
    frozen_again = again.download()
    sim.free()
    assert np.array_equal(again.download().view(np.uint64), frozen_again.view(np.uint64))
    plain.free()
    again.free()

    sim = Simulation(prob, flux_groups=edges)
    sim.inject()
    sim.step(1)
    gpu_lib.deallocate_data(sim.flux.ptr)
    sim.flux.ptr = None
    fresh = DeviceArray(sim.flux.n)
    sim.step(2)
    assert not np.any(fresh.download())
    fresh.free()
    sim.flux = None
    sim.free()


def test_refusals(gpu_lib):
    """Every refusal returns its code and says why; with a group flux attached the bank refuses
    pipeline=0 and tally_prereduce=1."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    n = prob.deck.nx * prob.deck.ny
    edges = np.array([1.0, 100.0, 1.0e4, 1.0e5])
    G = edges.size - 1

    def refused(rc, word, code=-3):
        assert rc == code, (rc, word)
        assert word.encode() in lib.nb200_last_error(), lib.nb200_last_error()

    def call(sim_bank, ptr, ncells, e=edges, g=G):
        e = np.ascontiguousarray(e, dtype=np.float64)
        return lib.nb200_bank_set_group_flux_tally(sim_bank, ptr, ncells, e.ctypes.data, g)

    flux = DeviceArray(G * n)
    junk = (C.c_double * 4)()
    not_a_bank = C.cast(C.addressof(junk), _soa_p)
    refused(call(not_a_bank, flux.ptr, n), "not a bank handle")

    sim = Simulation(prob)
    sim.inject()
    refused(call(sim.bank, flux.ptr, n, g=0), "ngroups")
    refused(call(sim.bank, flux.ptr, n, e=np.arange(258.0), g=257), "ngroups")
    refused(call(sim.bank, flux.ptr, n, e=[1.0, 1.0, 2.0, 3.0]), "strictly increasing")
    refused(call(sim.bank, flux.ptr, n, e=[1.0, np.nan, 2.0, 3.0]), "finite")
    sim.step(1, defer=True)
    refused(call(sim.bank, flux.ptr, n), "enqueued", code=-4)
    sim.step_finish()
    lib.nb200_bank_set_option(sim.bank, b"defer_finish", 0)
    host = np.zeros(G * n)
    refused(call(sim.bank, host.ctypes.data, n), "not device memory")
    refused(call(sim.bank, flux.ptr, 0), "cells")
    refused(call(sim.bank, flux.ptr, (1 << 31) // 2, e=np.arange(4.0) + 1.0), "2^31")
    for name, value in ((b"pipeline", 0), (b"tally_prereduce", 1)):
        prev = lib.nb200_bank_set_option(sim.bank, name, value)
        refused(call(sim.bank, flux.ptr, n), "pipeline=1 and tally_prereduce=0")
        lib.nb200_bank_set_option(sim.bank, name, prev)
    assert call(sim.bank, flux.ptr, n) == 0
    assert lib.nb200_bank_set_option(sim.bank, b"pipeline", 0) == NB200_BAD_OPTION
    assert b"flux tally" in lib.nb200_last_error()
    assert lib.nb200_bank_set_option(sim.bank, b"tally_prereduce", 1) == NB200_BAD_OPTION
    assert lib.nb200_bank_set_option(sim.bank, b"fast_div", 0) != NB200_BAD_OPTION
    lib.nb200_bank_set_option(sim.bank, b"fast_div", 1)
    sim.free()

    batched = Simulation(prob, tally_batches=4)
    batched.inject()
    refused(call(batched.bank, flux.ptr, n), "tally_batches")
    batched.free()

    blob = (C.c_char * 256)()
    assert lib.nb200_mp_init(2, 0, n, blob) == 0
    try:
        grouped = Simulation(prob)
        grouped.inject()
        refused(call(grouped.bank, flux.ptr, n), "multi-process group")
        grouped.free()
    finally:
        lib.nb200_mp_finalize()

    if lib.nb200_device_count() >= 2:
        sharded = Simulation(prob, ngpus=2)
        sharded.inject()
        refused(call(sharded.bank, flux.ptr, n), "several GPUs")
        sharded.free()
    flux.free()


_TERMINATES = """
import sys
sys.path.insert(0, {root!r})
import numpy as np
from neutral_b200.decks import build_problem
from neutral_b200.host import Simulation
edges = np.array([1.0, 100.0, 2.0e4])
sim = Simulation(build_problem("csp_small"), flux_groups=edges)
sim.inject()
assert sim.lib.nb200_bank_set_group_flux_tally(sim.bank, sim.flux.ptr, 128 * 127,
                                               edges.ctypes.data, 2) == 0
sim.step(1)
print("stepped")
"""


def test_enqueue_terminates_on_another_mesh(gpu_lib):
    """A mesh of another size than the attached array's ncells ends the process with the
    message."""
    res = subprocess.run([sys.executable, "-c", _TERMINATES.format(root=ROOT)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode != 0
    assert "stepped" not in res.stdout
    assert "the bank's flux tally has" in res.stderr, res.stderr


def test_full_csp_sixteen_groups(gpu_lib):
    """The full csp deck with 16 logarithmic groups covering every energy: summed over the
    groups, the group flux equals a plain-flux run's flux to 1e-10 per cell."""
    prob = build_problem("csp")
    edges = np.geomspace(1.0e-3, 2.0 * prob.deck.initial_energy, 17)
    plain = Simulation(prob, per_particle_counters=False, flux_tally=True)
    plain.inject()
    plain.run_pipelined()
    want = plain.flux_to_host().ravel()
    plain.free()
    sim = Simulation(prob, per_particle_counters=False, flux_groups=edges)
    sim.inject()
    sim.run_pipelined()
    got = sim.group_flux_to_host().reshape(16, -1)
    sim.free()
    assert np.count_nonzero(want) > 0
    assert np.count_nonzero(got.sum(axis=1)) >= 8  # the spectrum spreads over the groups
    assert _groups_close(got.sum(axis=0), want)
