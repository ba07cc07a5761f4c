"""Parity of the CUDA path (through the C-ABI) against the oracle port and the committed golden
vectors of the reference build (whole runs and step by step). Bars (BASELINE.json north_star):
per-particle event counts and every particle field bit-exact; tally within 1e-10 relative per
cell (atomic summation order)."""
import hashlib
import os

import numpy as np
import pytest

from conftest import SMALL_DECKS
from neutral_b200.bank import ALL_FIELDS, HostBank
from neutral_b200.decks import build_problem
from neutral_b200.host import NB200_BAD_OPTION, Simulation, solve_transport_2d_host
from recorded import field_hashes, reference_run

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TALLY_RTOL = 1e-10


def tally_close(a, b, rtol=TALLY_RTOL):
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b))))


def _hashes(bank):
    return [hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
            for k in ALL_FIELDS]


MODES = {
    "pipeline": dict(pipeline=1, fast_div=1, tile_shift=8, length_bins=512),   # the default
    "pipeline-ieee-div": dict(pipeline=1, fast_div=0, tile_shift=2, length_bins=16),
    # ... staging on the main stream, occupancy probe's shared-memory padding
    "pipeline-class-only": dict(pipeline=1, fast_div=1, tile_shift=-1, length_bins=1,
                                stage_overlap=0, history_smem_pad=4096),
    "pipeline-prereduce": dict(pipeline=1, fast_div=1, tile_shift=9, length_bins=512,
                               tally_prereduce=1),
    "direct": dict(pipeline=0, fast_div=0, tile_shift=9, length_bins=512),
    # the timestep's ~23 driver calls issued one by one instead of recorded into a CUDA graph
    # and submitted as one launch (the default since round 2)
    # half of the collision class dispatched behind the first 40 % of the streamer CTAs
    # (whatever the colliders' share of the bank), on a sort without the spatial key
    "pipeline-stagger": dict(pipeline=1, fast_div=1, tile_shift=-1, length_bins=512,
                             stagger_at=40, stagger_share=50, stagger_min=0),
    "pipeline-calls": dict(pipeline=1, fast_div=1, tile_shift=8, length_bins=512, step_graph=0),
}


DEFAULTS = dict(MODES["pipeline"], tally_prereduce=0, stage_overlap=1, history_smem_pad=0,
                step_graph=1, stagger_at=0, stagger_share=50, stagger_min=35)


@pytest.fixture(params=list(MODES))
def mode(request, gpu_lib):
    """Every kernel configuration must meet the same parity bar."""
    opts = MODES[request.param]
    for k, v in opts.items():
        assert gpu_lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION
    yield request.param
    for k, v in DEFAULTS.items():
        gpu_lib.nb200_set_option(k.encode(), v)


@pytest.mark.parametrize("deck", SMALL_DECKS)
def test_device_flavour_matches_oracle_every_step(gpu_lib, port, deck, mode):
    prob = build_problem(deck)
    d = prob.deck
    sim = Simulation(prob)
    sim.inject()
    bank = port.inject(prob)
    assert sum(sim.bank_to_host().bit_equal(bank).values()) == 0, "inject_particles differs"
    tally = np.zeros(d.nx * d.ny)
    ctr = np.zeros((3, len(bank)), dtype=np.uint64)
    for tt in range(1, d.iterations + 1):
        pf, pc, pp = port.step(prob, bank, tt, tally, counters=ctr)
        r = sim.step(tt)
        assert (r.facets, r.collisions, r.processed) == (pf, pc, pp), f"step {tt}"
        diff = sim.bank_to_host().bit_equal(bank)
        assert sum(diff.values()) == 0, f"step {tt}: {diff}"
        assert np.array_equal(sim.counters_to_host(), ctr), f"step {tt}: per-particle counts"
        assert tally_close(sim.tally_to_host(), tally), f"step {tt}: tally"
    sim.free()


@pytest.mark.parametrize("deck", SMALL_DECKS)
def test_device_flavour_matches_golden(gpu_lib, deck, mode):
    g = np.load(os.path.join(GOLDEN, f"{deck}.npz"))
    prob = build_problem(deck)
    sim = Simulation(prob)
    sim.inject()
    assert _hashes(sim.bank_to_host()) == list(g["inject_hashes"])
    counts = []
    for tt in range(1, prob.deck.iterations + 1):
        r = sim.step(tt)
        counts.append((r.facets, r.collisions, r.processed))
        if tt == 1:
            assert _hashes(sim.bank_to_host()) == list(g["step1_hashes"])
    assert np.array_equal(np.array(counts, dtype=np.uint64), g["counts"])
    final = sim.bank_to_host()
    assert _hashes(final) == list(g["final_hashes"])
    for k in ALL_FIELDS:
        assert final.arrays[k][:256].tobytes() == np.ascontiguousarray(g["sample"][k]).tobytes()
    assert np.array_equal(sim.counters_to_host(), g["particle_counters"])
    assert tally_close(sim.tally_to_host(), g["tally"])
    sim.free()


@pytest.mark.parametrize("deck", ["mixed_small", "csp_small"])
def test_host_flavour_is_a_drop_in_for_omp3(gpu_lib, port, deck):
    """Same call, same host arrays: nb200_solve_transport_2d_host against the reference omp3
    run recorded in tests/golden/steps.json, timestep by timestep."""
    prob = build_problem(deck)
    d = prob.deck
    want = reference_run(deck)
    aos_gpu = port.inject(prob).to_aos()
    assert field_hashes(HostBank.from_aos(aos_gpu)) == want["hashes"][0]
    t_gpu = np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        got = solve_transport_2d_host(prob, aos_gpu, tt, t_gpu)
        assert list(got) == want["counts"][tt - 1]
        assert field_hashes(HostBank.from_aos(aos_gpu)) == want["hashes"][tt]
        assert tally_close(np.array([t_gpu.sum()]), np.array([want["tally_sums"][tt - 1]]))
    assert tally_close(np.load(os.path.join(GOLDEN, f"{deck}.npz"))["tally"], t_gpu)


def test_host_flavour_matches_oracle(gpu_lib, port):
    prob = build_problem("split_small")
    d = prob.deck
    bank = port.inject(prob)
    aos = bank.to_aos()
    t_port, t_gpu = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    ctr_port = np.zeros((3, len(bank)), dtype=np.uint64)
    ctr_gpu = np.zeros((3, len(bank)), dtype=np.uint64)
    pf, pc, _ = port.step(prob, bank, 1, t_port, counters=ctr_port)
    assert solve_transport_2d_host(prob, aos, 1, t_gpu, counters=ctr_gpu) == (pf, pc)
    assert sum(HostBank.from_aos(aos).bit_equal(bank).values()) == 0
    assert np.array_equal(ctr_port, ctr_gpu)
    assert tally_close(t_port, t_gpu)


@pytest.mark.parametrize("nranks", [2, 3])
def test_shards_replay_the_whole_bank(gpu_lib, nranks):
    """Particle sharding (global RNG keys): shards reproduce their slice bit for bit and the
    shard tallies add up to the single-GPU tally."""
    prob = build_problem("mixed_small")
    d = prob.deck
    whole = Simulation(prob)
    whole.inject()
    res_whole = whole.run()
    bank_whole, tally_whole = whole.bank_to_host(), whole.tally_to_host()
    ctr_whole = whole.counters_to_host()
    whole.free()
    t_sum = np.zeros_like(tally_whole)
    ev = np.zeros((d.iterations, 2), dtype=np.int64)
    for r in range(nranks):
        sim = Simulation(prob, rank=r, nranks=nranks)
        sim.inject()
        res = sim.run()
        part = sim.bank_to_host()
        assert sum(bank_whole.slice(sim.pid0, sim.count).bit_equal(part).values()) == 0
        assert np.array_equal(ctr_whole[:, sim.pid0:sim.pid0 + sim.count], sim.counters_to_host())
        t_sum += sim.tally_to_host()
        ev += np.array([(x.facets, x.collisions) for x in res])
        sim.free()
    assert np.array_equal(ev, np.array([(x.facets, x.collisions) for x in res_whole]))
    assert tally_close(t_sum, tally_whole)


def test_edge_cases(gpu_lib, port):
    """Empty bank, fully dead bank, ragged (non multiple of the block size) bank."""
    prob = build_problem("scatter_small")
    d = prob.deck
    sim = Simulation(prob)
    sim.inject()
    r1 = sim.step(1)
    assert r1.processed == d.nparticles and r1.deaths == d.nparticles  # everyone dies
    r2 = sim.step(2)                                                   # nothing left to do
    assert (r2.facets, r2.collisions, r2.processed) == (0, 0, 0)
    sim.free()
    prob = build_problem("stream_small", nparticles=37)
    sim = Simulation(prob)
    sim.inject()
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny if False else prob.deck.nx * prob.deck.ny)
    pf, pc, pp = port.step(prob, bank, 1, tally)
    r = sim.step(1)
    assert (r.facets, r.collisions, r.processed) == (pf, pc, pp)
    assert sum(sim.bank_to_host().bit_equal(bank).values()) == 0
    sim.free()


def test_deferred_step_and_async_fold(gpu_lib, port):
    """solve_transport_2d under defer_finish + nb200_solve_finish, and the multi-GPU engine's
    three-buffer / side-stream fold, give the single-call result: exact counts, bit-equal
    bank, tally within tolerance (the fold only changes the summation order)."""
    import torch
    from neutral_b200.multi import GpuShardEngine

    prob = build_problem("csp_small")
    d = prob.deck
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    want = [port.step(prob, bank, tt, tally) for tt in range(1, d.iterations + 1)]
    sim = Simulation(prob, per_particle_counters=False)
    sim.inject()
    eng = GpuShardEngine(sim, d.nx * d.ny)
    got = []
    for i in range(d.iterations):
        k = i % eng.nbuffers
        eng.acquire(k)
        eng.step_begin(i + 1, k)
        eng.fold_async(k, None)  # queued behind the transport on the side stream
        r = eng.step_end()
        got.append((r.facets, r.collisions, r.processed))
    eng.drain()
    torch.cuda.synchronize()
    assert got == want
    assert sum(sim.bank_to_host().bit_equal(bank).values()) == 0
    assert tally_close(sim.tally_to_host(), tally)
    assert all(not bool(t.any()) for t in eng.delta), "delta buffers must end up cleared"
    sim.free()


@pytest.mark.parametrize("deck", ["csp_small", "split_small"])
def test_device_inject_equals_host_inject(gpu_lib, port, deck):
    """inject_particles on the device (default), on the host with libm (device_inject=0) and
    the oracle port, whose bank is pinned by tests/golden/steps.json, all produce the same
    bank, bit for bit - whole and as shards (global RNG keys)."""
    prob = build_problem(deck, nparticles=50_000)
    want = port.inject(prob)
    assert field_hashes(want) == reference_run(f"{deck}@50000")["hashes"][0]
    for device_inject in (1, 0):
        gpu_lib.nb200_set_option(b"device_inject", device_inject)
        try:
            sim = Simulation(prob, per_particle_counters=False)
            sim.inject()
            assert sum(sim.bank_to_host().bit_equal(want).values()) == 0, device_inject
            sim.free()
            for r in range(3):
                part = Simulation(prob, rank=r, nranks=3, per_particle_counters=False)
                part.inject()
                got = part.bank_to_host()
                assert sum(want.slice(part.pid0, part.count).bit_equal(got).values()) == 0
                part.free()
        finally:
            gpu_lib.nb200_set_option(b"device_inject", 1)
