"""The pieces of the sharded-tally tests that need no GPU (tests/collective_cases.py): the owned
slices of every mesh, the schedule model, the rank-order emulator against hand-made deltas whose
sum depends on the order, and the precondition of the deterministic banks, checked with the
oracle port one particle at a time."""
import numpy as np
import pytest

from collective_cases import (MESHES, SCHEDULES, exact_bank, group_events, layout,
                              mesh_problem, rank_order_looks, summation_bound_violations,
                              timesteps, windows)
from edge_banks import contract_violations
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.multi import owned_slice_layout


@pytest.mark.parametrize("ncells,nranks,want", [
    # even chunk, odd last slice
    (9999, 2, [(0, 5000), (5000, 4999)]),
    (9999, 3, [(0, 3334), (3334, 3334), (6668, 3331)]),
    # a one-cell slice and an empty one
    (9, 4, [(0, 4), (4, 4), (8, 1), (12, 0)]),
    # a slice longer than one pass of k_gather_owned (296 x 256 threads x 2 cells = 151 552)
    # and of k_fold_plain (75 776); odd last slice
    (305909, 2, [(0, 152956), (152956, 152953)]),
    # the decks
    (16384, 3, [(0, 5462), (5462, 5462), (10924, 5460)]),
    (6400, 8, [(0, 800), (800, 800), (1600, 800), (2400, 800), (3200, 800), (4000, 800),
               (4800, 800), (5600, 800)]),
    (9999, 8, [(0, 1250)] + [(1250 * r, 1250) for r in range(1, 7)] + [(8750, 1249)]),
    (9, 5, [(0, 2), (2, 2), (4, 2), (6, 2), (8, 1)]),
    (9, 8, [(0, 2), (2, 2), (4, 2), (6, 2), (8, 1), (10, 0), (12, 0), (14, 0)]),
])
def test_owned_slice_layouts(ncells, nranks, want):
    chunk, padded = owned_slice_layout(ncells, nranks)
    assert chunk % 2 == 0 and padded == chunk * nranks and padded >= ncells
    assert layout(ncells, nranks) == want
    assert sum(c for _, c in want) == ncells


def test_mesh_sizes():
    assert {k: nx * ny for k, (nx, ny) in MESHES.items()} == \
        {"m9999": 9999, "m9": 9, "m305909": 305909}
    chunk, _ = owned_slice_layout(305909, 2)
    assert chunk > 296 * 256 * 2 and chunk > 296 * 256


@pytest.mark.parametrize("schedule,every", [(s, e) for s in SCHEDULES for e in (0, 1, 2)
                                             if not (s.startswith("pipe") and e == 0)])
def test_schedules_wrap_the_delta_buffers(schedule, every):
    """Every schedule makes at least 4 reductions (3 delta buffers rotate), runs an odd number
    of timesteps, and every timestep lands in exactly one window. (The pipelined schedules are
    for reduce_every >= 1: on demand they reduce twice.)"""
    ev = group_events(SCHEDULES[schedule], every)
    ws = windows(ev)
    steps = [tt for tt, _ in timesteps(SCHEDULES[schedule])]
    assert len(ws) >= 4, ws
    assert len(steps) % 2 == 1
    assert sorted(tt for w in ws for tt in w) == steps
    if every:
        assert all(len(w) <= every for w in ws)


def test_schedule_model_windows():
    ev = group_events(SCHEDULES["looks"], 2)
    assert windows(ev) == [(1,), (2, 3), (4,), (5,)]
    # the second look after timestep 1 finds nothing new: no reduction, no gather
    assert ev[:5] == [("reduce", (1,)), ("gather", "A"), ("look", "A"), ("look", "A"),
                      ("reduce", (2, 3))]
    ev = group_events(SCHEDULES["second_tally"], 0)
    assert ev == [("reduce", (1,)), ("gather", "A"), ("look", "A"),
                  ("reduce", (2, 3)), ("gather", "A"),          # the switch to B flushes A
                  ("look", "A"), ("reduce", (4,)), ("gather", "B"), ("look", "B"),
                  ("look", "B"), ("reduce", (5,)), ("gather", "A"), ("look", "A")]
    assert windows(group_events(SCHEDULES["pipe4"], 1)) == [(t,) for t in range(1, 8)]


def test_rank_order_emulator_on_order_sensitive_deltas():
    """Three ranks, one cell: 1 + 2^-53 + 2^-53 is 1 summed from rank 0 up and 1 + 2^-52 in
    any order that adds the two small terms first; a second window and a look show that the
    owned value is kept across reductions and zeroed by a gather."""
    u = 2.0 ** -53
    d = [{(1,): np.array([1.0, -0.0]), (2,): np.array([3.0, 0.0])},
         {(1,): np.array([u, 5e-324]), (2,): np.array([u, 0.0])},
         {(1,): np.array([u, 5e-324]), (2,): np.array([u, 1e300])}]
    ev = [("reduce", (1,)), ("gather", "A"), ("look", "A"), ("reduce", (2,)), ("look", "A"),
          ("gather", "A"), ("look", "A")]
    looks = rank_order_looks(ev, d, 2)
    assert looks[0].tolist() == [1.0, 1e-323]
    assert looks[1].tolist() == [1.0, 1e-323]          # reduced, not yet gathered
    # owned after window 2: ((0 + 3) + u) + u = 3 (ties to even twice)
    assert looks[2].tolist() == [4.0, 1e300 + 1e-323]
    rev = rank_order_looks(ev, d[::-1], 2)
    assert rev[0][0] == 1.0 + 2.0 ** -52 != looks[0][0]
    # the ordered sum is not the exact one either: fsum would say 1 + 2^-52
    assert summation_bound_violations(ev, d, looks, 2) == []
    assert summation_bound_violations(ev, d, [x + 1e-9 for x in looks], 2) != []


EXACT = [("m9999", 2), ("m9999", 3), ("m9", 4), ("m305909", 2), ("m9999", 5), ("m9999", 8),
         ("m9", 8)]


@pytest.mark.parametrize("mesh,nranks", EXACT)
def test_exact_bank_precondition(port, mesh, nranks):
    """Within every shard, the cells each particle deposits into over the longest schedule are
    disjoint from every other particle's (the port, one particle at a time); the whole bank
    records no collision; the bank is valid input (edge_banks.contract_violations)."""
    steps = max(max(tt for tt, _ in timesteps(s)) for s in SCHEDULES.values())
    prob = mesh_problem(mesh, nranks * MESHES[mesh][1], steps, exact=True)
    d = prob.deck
    bank = exact_bank(prob, nranks)
    assert contract_violations(prob, bank) == []
    # the ranks' energies and weights differ
    for k in ("energy", "weight"):
        means = [bank.arrays[k][slice(*_range(d.nparticles, r, nranks))].mean()
                 for r in range(nranks)]
        assert len(set(means)) == nranks
    whole = exact_bank(prob, nranks)
    tally = np.zeros(d.nx * d.ny)
    for tt in range(1, steps + 1):
        f, c, p = port.step(prob, whole, tt, tally)
        assert c == 0 and p == d.nparticles and f > 0
    assert contract_violations(prob, whole) == []
    for r in range(nranks):
        pid0, count = shard_range(d.nparticles, r, nranks)
        owner = np.full(d.nx * d.ny, -1)
        for j in range(count):
            one = bank.slice(pid0 + j, 1)
            mine = np.zeros(d.nx * d.ny)
            for tt in range(1, steps + 1):
                port.step(prob, one, tt, mine, pid0=pid0 + j, ntotal=d.nparticles)
            cells = np.flatnonzero(mine)
            assert cells.size and np.all(owner[cells] == -1), (r, j)
            owner[cells] = j
    # every cell is reached (the last slice's cells included)
    assert np.all(tally > 0.0)


def _range(n, r, nranks):
    pid0, count = shard_range(n, r, nranks)
    return pid0, pid0 + count


def test_deck_cases_build():
    prob = build_problem("csp_small", iterations=7)
    assert prob.deck.iterations == 7 and prob.deck.nx * prob.deck.ny == 16384
