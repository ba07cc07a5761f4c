"""Pins the oracle port against the committed golden vectors of the UNMODIFIED reference omp3
build (tests/golden/make_golden.py, make_golden_steps.py) - bit-exact particle state, exact
counts, tally to 1e-12."""
import hashlib
import os

import numpy as np
import pytest

from conftest import SMALL_DECKS
from neutral_b200.bank import ALL_FIELDS
from neutral_b200.decks import build_problem, shard_range
from recorded import field_hashes, reference_run

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _hashes(bank):
    return [hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
            for k in ALL_FIELDS]


def _run_port(port, prob, pid0=0, count=None, counters=True):
    d = prob.deck
    bank = port.inject(prob, pid0, count)
    tally = np.zeros(d.nx * d.ny)
    ctr = np.zeros((3, len(bank)), dtype=np.uint64) if counters else None
    counts, step1 = [], None
    for tt in range(1, d.iterations + 1):
        counts.append(port.step(prob, bank, tt, tally, pid0=pid0, counters=ctr))
        if tt == 1:
            step1 = bank.copy()
    return bank, tally, ctr, counts, step1


@pytest.mark.parametrize("deck", SMALL_DECKS)
def test_port_matches_golden(port, deck):
    g = np.load(os.path.join(GOLDEN, f"{deck}.npz"))
    prob = build_problem(deck)
    assert _hashes(port.inject(prob)) == list(g["inject_hashes"])
    bank, tally, ctr, counts, step1 = _run_port(port, prob)
    assert np.array_equal(np.array(counts, dtype=np.uint64), g["counts"])
    assert _hashes(step1) == list(g["step1_hashes"])
    assert _hashes(bank) == list(g["final_hashes"])
    for k in ALL_FIELDS:  # field-wise: the AoS padding bytes are not part of the state
        assert bank.arrays[k][:256].tobytes() == np.ascontiguousarray(g["sample"][k]).tobytes(), k
    assert np.array_equal(ctr, g["particle_counters"])
    ref_t = g["tally"]
    assert np.all(np.abs(tally - ref_t) <= 1e-12 * np.maximum(np.abs(tally), np.abs(ref_t)))


@pytest.mark.parametrize("deck", SMALL_DECKS)
def test_port_matches_reference_build(port, deck):
    """Every timestep against the reference run recorded in tests/golden/steps.json: exact
    counts, every particle field bit for bit, the tally's sum; the final tally cell by cell to
    1e-12."""
    prob = build_problem(deck)
    d = prob.deck
    want = reference_run(deck)
    bank = port.inject(prob)
    assert field_hashes(bank) == want["hashes"][0]
    t_port = np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        pf, pc, _ = port.step(prob, bank, tt, t_port)
        assert [pf, pc] == want["counts"][tt - 1]
        assert field_hashes(bank) == want["hashes"][tt]
        assert abs(t_port.sum() - want["tally_sums"][tt - 1]) <= 1e-12 * abs(t_port.sum())
    t_ref = np.load(os.path.join(GOLDEN, f"{deck}.npz"))["tally"]
    assert np.all(np.abs(t_ref - t_port) <= 1e-12 * np.maximum(np.abs(t_ref), np.abs(t_port)))


def test_golden_totals_are_consistent():
    """Per-particle counters sum to the reference's aggregate counts."""
    for deck in SMALL_DECKS:
        g = np.load(os.path.join(GOLDEN, f"{deck}.npz"))
        assert g["particle_counters"][0].sum() == g["counts"][:, 0].sum()
        assert g["particle_counters"][1].sum() == g["counts"][:, 1].sum()


@pytest.mark.parametrize("nranks", [2, 3])
def test_sharded_histories_replay_identically(port, nranks):
    """Histories depend on the global pid only: any contiguous shard reproduces its slice
    of the whole-bank run bit for bit, and the shard tallies add up (SURVEY.md 8e)."""
    prob = build_problem("mixed_small")
    d = prob.deck
    whole, t_whole, c_whole, counts_whole, _ = _run_port(port, prob)
    t_sum = np.zeros_like(t_whole)
    totals = np.zeros((d.iterations, 3), dtype=np.int64)
    for r in range(nranks):
        first, count = shard_range(d.nparticles, r, nranks)
        part, t_part, c_part, counts, _ = _run_port(port, prob, first, count)
        assert sum(whole.slice(first, count).bit_equal(part).values()) == 0
        assert np.array_equal(c_whole[:, first:first + count], c_part)
        t_sum += t_part
        totals += np.array(counts)
    assert np.array_equal(totals, np.array(counts_whole))
    assert np.all(np.abs(t_sum - t_whole) <= 1e-10 * np.maximum(np.abs(t_sum), np.abs(t_whole)))


def test_shard_range_partitions():
    for n in (0, 1, 7, 1000, 10**6 + 3):
        for g in (1, 2, 3, 4, 8):
            pos = 0
            for r in range(g):
                first, count = shard_range(n, r, g)
                assert first == pos and count >= 0
                pos += count
            assert pos == n
