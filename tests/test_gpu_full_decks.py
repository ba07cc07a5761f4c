"""The BASELINE.json decks at full size on the GPU (4000 x 4000 mesh, 1e6 / 1e7 particles).

The oracle cannot replay these in seconds, so the checks are (i) the aggregate event counts
the UNMODIFIED reference omp3 build printed for the same decks (SURVEY.md 2.2 / BASELINE.md 3,
measured with the reference binary, `Facets` / `Collisions` / `Particles` lines of
main.c:118-125 and omp3/neutral.c:205) - exact; (ii) the reference's own golden tally sums of
problems/neutral.tests through `validate`'s 1e-3 criterion (omp3/neutral.c:549) and the tally
sums the reference build produced, to 1e-10; (iii) size-independent invariants: every processed
particle ends the step in exactly one census or death, dead particles are never processed
again, the tally only grows."""
import numpy as np
import pytest

from neutral_b200.decks import build_problem
from neutral_b200.host import Simulation

pytestmark = pytest.mark.gpu

# deck -> (facets, collisions, `Particles` line of the last timestep, tally sum) of the
# reference run
REFERENCE_RUNS = {
    "stream": (7_044_482_122, 0, 1_000_000, 5.760059926484883e-24),
    "csp": (6_197_618_387, 216_380_159, 795_597, 1.121829757714269e+07),
    "split": (557_455_972, 510_991_328, 1_000_000, 4.139740922510341e+06),
    "scatter": (4_918, 6_987_255_492, 0, 3.413271914237598e-02),
}
NEUTRAL_TESTS = {"scatter": 3.411662060900e-02, "stream": 5.760064605960129e-24,
                 "csp": 1.121870290714e+07}


@pytest.mark.parametrize("deck", list(REFERENCE_RUNS))
def test_full_deck_matches_the_reference_run(gpu_lib, deck):
    facets, collisions, last_processed, tally_sum = REFERENCE_RUNS[deck]
    prob = build_problem(deck)
    d = prob.deck
    sim = Simulation(prob, per_particle_counters=False)
    sim.inject()
    live = d.nparticles
    tot_f = tot_c = 0
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        assert r.processed == live, f"step {tt}: dead particles must not be processed"
        assert r.census + r.deaths == r.processed, f"step {tt}: one census or death each"
        live -= r.deaths
        tot_f += r.facets
        tot_c += r.collisions
    assert (tot_f, tot_c) == (facets, collisions)
    assert r.processed == last_processed
    tally = sim.tally_to_host()
    assert np.all(tally >= 0.0)
    got = float(np.sum(tally))
    assert got > 0.0
    assert abs(got - tally_sum) <= 1e-10 * tally_sum
    if deck in NEUTRAL_TESTS:  # validate()'s criterion, omp3/neutral.c:549
        assert abs(got - NEUTRAL_TESTS[deck]) / NEUTRAL_TESTS[deck] < 1e-3
    bank = sim.bank_to_host()
    assert int(np.count_nonzero(bank.dead == 0)) == live
    assert np.all((bank.cellx >= 0) & (bank.cellx < d.nx) & (bank.celly >= 0) & (bank.celly < d.ny))
    sim.free()


def test_full_deck_shards_add_up(gpu_lib):
    """split at full size as 2 shards: counts add up exactly, tallies to 1e-10 per cell."""
    prob = build_problem("split")
    whole = Simulation(prob, per_particle_counters=False)
    whole.inject()
    rw = whole.step(1)
    tw = whole.tally_to_host()
    whole.free()
    f = c = 0
    ts = np.zeros_like(tw)
    for r in range(2):
        sim = Simulation(prob, rank=r, nranks=2, per_particle_counters=False)
        sim.inject()
        res = sim.step(1)
        f += res.facets
        c += res.collisions
        ts += sim.tally_to_host()
        sim.free()
    assert (f, c) == (rw.facets, rw.collisions)
    assert np.all(np.abs(ts - tw) <= 1e-10 * np.maximum(np.abs(ts), np.abs(tw)))


def _golden_full():
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_decks.json")
    with open(path) as f:
        return json.load(f)


@pytest.mark.parametrize("deck", ["split", "csp", "stream", "scatter"])
def test_full_deck_bank_is_bit_identical_to_the_reference(gpu_lib, deck):
    """Full-size parity against fixtures generated from the UNMODIFIED reference library
    (tests/golden/make_golden_full.py): per-timestep counts exact, the injected bank and the
    final bank bit-identical in all 11 fields (sha256 per field, 1e6 / 1e7 particles), the tally
    through its total and a 64 x 64 block-sum image (1e-10: atomic summation order; observed 1e-15)."""
    import hashlib

    from neutral_b200.bank import ALL_FIELDS
    g = _golden_full()
    if deck not in g:
        pytest.skip(f"no full-size fixture for {deck}")
    g = g[deck]
    prob = build_problem(deck)
    d = prob.deck
    assert (d.nparticles, [d.nx, d.ny], d.iterations) == (g["nparticles"], g["mesh"],
                                                          g["iterations"])

    def hashes(bank):
        return {k: hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
                for k in ALL_FIELDS}

    sim = Simulation(prob, per_particle_counters=False)
    sim.inject()
    assert hashes(sim.bank_to_host()) == g["inject_hashes"]
    counts = []
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        counts.append([r.facets, r.collisions])
    assert counts == g["counts"]
    bank = sim.bank_to_host()
    assert hashes(bank) == g["final_hashes"]
    assert int(np.count_nonzero(bank.dead == 0)) == g["live"]
    tally = sim.tally_to_host()
    assert abs(float(tally.sum()) - g["tally_sum"]) <= 1e-10 * g["tally_sum"]
    blocks = 64
    by, bx = d.ny // blocks, d.nx // blocks
    img = tally.reshape(d.ny, d.nx)[:by * blocks, :bx * blocks] \
        .reshape(blocks, by, blocks, bx).sum(axis=(1, 3)).ravel()
    want = np.array(g["tally_block_sums"])
    assert np.all(np.abs(img - want) <= 1e-10 * np.maximum(np.abs(img), np.abs(want)))
    sim.free()


@pytest.mark.parametrize("deck", ["csp", "split"])
def test_full_deck_tally_per_cell_against_the_reference_library(gpu_lib, deck):
    """north_star's tally bar at FULL size (BASELINE.json: "within a stated relative tolerance
    of 1e-10 per cell"): the final tally of the deck's reference run, recorded on a fixed,
    seeded sample of its non-zero cells (tests/golden/tally_samples.npz, from the oracle port's
    replay of the run that matches the reference library's counts, bank and block sums), is
    compared cell by cell with the pipelined run - together with the number of non-zero cells,
    the per-timestep counts and every field of the final bank."""
    import hashlib

    from neutral_b200.bank import ALL_FIELDS
    from recorded import tally_matches_sample
    g = _golden_full()[deck]
    prob = build_problem(deck)
    sim = Simulation(prob, per_particle_counters=False)
    sim.inject()
    got = [[r.facets, r.collisions] for r in sim.run_pipelined()]
    assert got == g["counts"]
    bank = sim.bank_to_host()
    assert {k: hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
            for k in ALL_FIELDS} == g["final_hashes"]
    assert tally_matches_sample(sim.tally_to_host(), deck, 1e-10)
    sim.free()
