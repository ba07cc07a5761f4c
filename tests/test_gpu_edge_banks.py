"""The crafted edge-case banks (tests/edge_banks.py) on the GPU, loaded with
Simulation.load_bank: in every kernel mode of test_gpu_parity.MODES every timestep meets the
parity bar against the oracle port (exact counts and per-particle counters, all 11 fields bit
for bit, tally within 1e-10 per cell); the flux tally matches its reference; tally batches move
deposits, never histories; the host-buffer flavour matches the port; and the vacuum flights equal
the exact ray reference."""
import numpy as np
import pytest

import edge_banks as eb
from flux_reference import flux_reference
from neutral_b200.bank import ALL_FIELDS, HostBank
from neutral_b200.decks import shard_range
from neutral_b200.host import NB200_BAD_OPTION, Simulation, solve_transport_2d_host
from test_gpu_parity import DEFAULTS, MODES, tally_close

pytestmark = pytest.mark.gpu

CASES = eb.all_cases()
IDS = [c.id for c in CASES]
MIXED = [c for c in CASES if c.label == "mixed"]
VACUUM = [c for c in CASES if c.problem == "vacuum" and c.label != "dead"]


def _set_mode(lib, name):
    for k, v in MODES[name].items():
        assert lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION


@pytest.fixture(params=list(MODES))
def mode(request, gpu_lib):
    _set_mode(gpu_lib, request.param)
    yield request.param
    for k, v in DEFAULTS.items():
        gpu_lib.nb200_set_option(k.encode(), v)


@pytest.fixture(params=["pipeline", "pipeline-ieee-div"])
def flux_mode(request, gpu_lib):
    _set_mode(gpu_lib, request.param)
    yield request.param
    for k, v in DEFAULTS.items():
        gpu_lib.nb200_set_option(k.encode(), v)


def differing(case, got: HostBank, want: HostBank) -> dict:
    """{field: sorted categories of the slots whose bits differ} (empty when bit-identical)."""
    out = {}
    for k in ALL_FIELDS:
        a, b = got.arrays[k], want.arrays[k]
        bad = a.view(np.uint64) != b.view(np.uint64) if a.dtype == np.float64 else a != b
        if np.any(bad):
            out[k] = sorted(set(case.tags[bad]))
    return out


def counter_diff(case, got, want) -> list:
    return sorted(set(case.tags[np.any(got != want, axis=0)]))


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_every_step_matches_the_port(gpu_lib, port, case, mode):
    d = case.prob.deck
    sim = Simulation(case.prob)
    sim.load_bank(case.bank)
    bank = case.bank.copy()
    tally = np.zeros(d.nx * d.ny)
    ctr = np.zeros((3, len(bank)), dtype=np.uint64)
    for tt in range(1, d.iterations + 1):
        want = port.step(case.prob, bank, tt, tally, counters=ctr)
        r = sim.step(tt)
        assert (r.facets, r.collisions, r.processed) == want, f"step {tt}"
        assert differing(case, sim.bank_to_host(), bank) == {}, f"step {tt}"
        assert counter_diff(case, sim.counters_to_host(), ctr) == [], f"step {tt}"
        assert tally_close(sim.tally_to_host(), tally), f"step {tt}: tally"
    sim.free()


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_flux_matches_its_reference(gpu_lib, case, flux_mode):
    d = case.prob.deck
    sim = Simulation(case.prob, flux_tally=True)
    sim.load_bank(case.bank)
    bank = case.bank.copy()
    tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        want = flux_reference().step(case.prob, bank, tt, tally, flux=flux)
        r = sim.step(tt)
        assert (r.facets, r.collisions, r.processed) == want, f"step {tt}"
        assert differing(case, sim.bank_to_host(), bank) == {}, f"step {tt}"
        assert tally_close(sim.flux_to_host().ravel(), flux), f"step {tt}: flux"
    assert tally_close(sim.tally_to_host(), tally)
    sim.free()


@pytest.mark.parametrize("case", MIXED, ids=[c.id for c in MIXED])
def test_tally_batches_leave_histories_alone(gpu_lib, port, case):
    """tally_batches = 3: the bank after every timestep equals the port's, and every batch
    equals the port run on its particle range (with the whole bank's normalisation)."""
    d = case.prob.deck
    B = 3
    sim = Simulation(case.prob, tally_batches=B)
    sim.load_bank(case.bank)
    whole = case.bank.copy()
    t_whole = np.zeros(d.nx * d.ny)
    ranges = [shard_range(d.nparticles, b, B) for b in range(B)]
    parts = [case.bank.slice(f, n) for f, n in ranges]
    tallies = [np.zeros(d.nx * d.ny) for _ in range(B)]
    for tt in range(1, d.iterations + 1):
        want = port.step(case.prob, whole, tt, t_whole)
        for b, (f, n) in enumerate(ranges):
            port.step(case.prob, parts[b], tt, tallies[b], pid0=f, ntotal=d.nparticles)
        r = sim.step(tt)
        assert (r.facets, r.collisions, r.processed) == want, f"step {tt}"
        assert differing(case, sim.bank_to_host(), whole) == {}, f"step {tt}"
        got = sim.tally_batches_to_host().reshape(B, -1)
        for b in range(B):
            assert tally_close(got[b], tallies[b]), (tt, b)
    assert tally_close(sim.tally_to_host(), t_whole)
    sim.free()


@pytest.mark.parametrize("case", MIXED, ids=[c.id for c in MIXED])
def test_host_flavour_matches_the_port(gpu_lib, port, case):
    d = case.prob.deck
    bank = case.bank.copy()
    aos = case.bank.to_aos()
    t_port, t_gpu = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    c_port = np.zeros((3, len(bank)), dtype=np.uint64)
    c_gpu = np.zeros((3, len(bank)), dtype=np.uint64)
    for tt in range(1, d.iterations + 1):
        pf, pc, _ = port.step(case.prob, bank, tt, t_port, counters=c_port)
        assert solve_transport_2d_host(case.prob, aos, tt, t_gpu, counters=c_gpu) == (pf, pc)
        assert differing(case, HostBank.from_aos(aos), bank) == {}, f"step {tt}"
        assert counter_diff(case, c_gpu, c_port) == [], f"step {tt}"
        assert tally_close(t_gpu, t_port), f"step {tt}"


@pytest.mark.parametrize("case", VACUUM, ids=[c.id for c in VACUUM])
def test_gpu_flies_the_exact_rays(gpu_lib, case, flux_mode):
    """The exact ray reference of test_edge_banks_cpu applied to the GPU's own results."""
    run = eb.exact_run(case)
    sim = Simulation(case.prob, flux_tally=True)
    sim.load_bank(case.bank)
    prev = np.zeros(len(case.bank), dtype=np.uint64)
    for t in range(case.prob.deck.iterations):
        sim.step(t + 1)
        facets = sim.counters_to_host()[0]
        assert eb.exact_mismatches(case.prob, run, t, sim.bank_to_host(), facets - prev) == [], t
        prev = facets
    assert eb.flux_matches_exact(case.prob, sim.flux_to_host().ravel(), run.flux)
    sim.free()
