"""Meshes, banks, schedules and references for the tests of the sharded tally collective
(TEST INFRASTRUCTURE).

A sharded run combines its tally in ``csrc/group.cu`` and ``capi.cu`` (``group_layout``,
``group_reduce``, ``group_flush``): every rank deposits into a private buffer, a reduction adds
slice r of every rank's buffer, in rank order, to the slice rank r owns, and a look at the tally
adds every owned slice into it and clears them. The meshes here are chosen for the slices they
produce (odd last slices, a one-cell slice and an empty one, slices longer than one pass of the
kernels' grids), the schedules for the state they drive the protocol through (repeated looks,
rotating delta buffers, pipelined timesteps, a second tally pointer).

:func:`exact_bank` builds a bank whose tally is deterministic: within one shard no two particles
ever deposit into the same cell, so each rank's buffer receives every cell's deposits in one
thread's program order. :class:`GroupModel` restates when the library reduces and gathers, and
:func:`rank_order_looks` what the peer-memory flavour then computes, addition by addition, so the
library's tally can be held to it bit for bit.

Plain numpy; nothing here runs a kernel.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Sequence, Tuple

import numpy as np

from neutral_b200.bank import HostBank
from neutral_b200.decks import Deck, Problem, build_problem, shard_range
from neutral_b200.multi import owned_slice_layout

#: name -> (nx, ny). The slice shapes they give are pinned in tests/test_collective_cpu.py
MESHES = {
    "m9999": (99, 101),      # N = 2: 5000 + 4999 cells; N = 3: 3334 + 3334 + 3331
    "m9": (3, 3),            # N = 4: chunk 4, slices of 4, 4, 1 and 0 cells
    "m305909": (601, 509),   # N = 2: chunk 152 956, more than one pass of the gather's grid
}

DT = 1.0e-7
E_EXACT = 1.0e6           # ~1.4 mesh widths per timestep: a particle sweeps its whole row
RHO_EXACT = 1.0e-9        # the port records no collision on any exact bank here


def mesh_problem(mesh: str, nparticles: int, iterations: int, exact: bool) -> Problem:
    """The unit square on one of MESHES. ``exact``: uniform density RHO_EXACT (for
    :func:`exact_bank`); otherwise a thin medium with a denser box (mixed_small's densities),
    source over the whole mesh so that every cell sees deposits."""
    nx, ny = MESHES[mesh]
    problems = [(RHO_EXACT, 0.0, 0.0, 1.0, 1.0)] if exact else \
        [(1.0e-30, 0.0, 0.0, 1.0, 1.0), (1.0, 0.25, 0.25, 0.5, 0.5), (6.0, 0.45, 0.45, 0.1, 0.1)]
    deck = Deck(path=f"{mesh}.params", nx=nx, ny=ny, dt=DT, iterations=iterations,
                nparticles=nparticles, initial_energy=1.0e5, source=(0.0, 0.0, 1.0, 1.0),
                problems=problems)
    return build_problem(deck)


def exact_bank(prob: Problem, nranks: int, seed: int = 0) -> HostBank:
    """nranks shards of ny particles each: particle j of every shard sits in row j and flies
    along +-x (omega_y = +0.0), so it never leaves its row and no two particles of one shard
    share a cell. Energy and weight differ per rank (scaled by 1 + r and 1 / (1 + 2r)) and per
    particle, so that the ranks' deltas of one cell differ in magnitude and their sum depends on
    the order of the additions."""
    d = prob.deck
    n = nranks * d.ny
    assert d.nparticles == n
    ex, ey = prob.edgex, prob.edgey
    rng = np.random.default_rng(seed + 1000 * nranks + d.nx)
    bank = HostBank.empty(n)
    for r in range(nranks):
        pid0, count = shard_range(n, r, nranks)
        assert count == d.ny
        for j in range(count):
            i = pid0 + j
            cx = int(rng.integers(d.nx))
            bank.x[i] = ex[cx] + (0.2 + 0.6 * rng.random()) * (ex[cx + 1] - ex[cx])
            bank.y[i] = ey[j] + 0.5 * (ey[j + 1] - ey[j])
            bank.omega_x[i] = 1.0 if rng.random() < 0.5 else -1.0
            bank.omega_y[i] = 0.0
            bank.energy[i] = E_EXACT * (1 + r) * (0.75 + 0.5 * rng.random())
            bank.weight[i] = (0.5 + rng.random()) / (1 + 2 * r)
            bank.dt_to_census[i], bank.mfp_to_collision[i] = d.dt, 0.0
            bank.cellx[i], bank.celly[i], bank.dead[i] = cx, j, 0
    return bank


# ---------------------------------------------------------------------------- schedules --
# ("step", tt, tally) | ("look", tally) | ("pipe", first_tt, count, depth): timesteps into
# tally "A" enqueued `depth` deep (Simulation.run_pipelined). Tally "B" is a second pointer.

SCHEDULES: Dict[str, List[tuple]] = {
    # a look after timestep 1, twice in a row, then between timesteps and at the end
    "looks": [("step", 1, "A"), ("look", "A"), ("look", "A"), ("step", 2, "A"), ("step", 3, "A"),
              ("look", "A"), ("step", 4, "A"), ("look", "A"), ("step", 5, "A"), ("look", "A")],
    # timestep 4 into a second tally: A keeps exactly timesteps 1-3 (switching flushes A), B
    # gets timestep 4 alone, and switching back flushes B
    "second_tally": [("step", 1, "A"), ("look", "A"), ("step", 2, "A"), ("step", 3, "A"),
                     ("step", 4, "B"), ("look", "A"), ("look", "B"), ("step", 5, "A"),
                     ("look", "B"), ("look", "A")],
    "pipe3": [("step", 1, "A"), ("look", "A"), ("pipe", 2, 6, 3), ("look", "A")],
    "pipe4": [("step", 1, "A"), ("look", "A"), ("pipe", 2, 6, 4), ("look", "A")],
}


def timesteps(schedule: Sequence[tuple]) -> List[Tuple[int, str]]:
    """(tt, tally) of every timestep, in order."""
    out = []
    for op in schedule:
        if op[0] == "step":
            out.append((op[1], op[2]))
        elif op[0] == "pipe":
            out += [(tt, "A") for tt in range(op[1], op[1] + op[2])]
    return out


class GroupModel:
    """When the library's group reduces and gathers (capi.cu: enqueue_step, group_flush).
    A timestep into another tally than the group's flushes the old one first; a window of
    timesteps is reduced when it holds `reduce_every` timesteps (0: never by itself) or when the
    tally is looked at; a look at a tally with nothing new since the last look does nothing."""

    def __init__(self, reduce_every: int):
        self.every = reduce_every
        self.window: List[int] = []
        self.target = None
        self.dirty = False
        self.events: List[tuple] = []

    def step(self, tt: int, tally: str) -> None:
        if tally != self.target:
            self.flush()
            self.target = tally
        self.window.append(tt)
        self.dirty = True
        if self.every > 0 and len(self.window) >= self.every:
            self.events.append(("reduce", tuple(self.window)))
            self.window = []

    def look(self, tally: str) -> None:
        if tally == self.target:
            self.flush()
        self.events.append(("look", tally))

    def flush(self) -> None:
        if not self.dirty or self.target is None:
            return
        if self.window:
            self.events.append(("reduce", tuple(self.window)))
            self.window = []
        self.events.append(("gather", self.target))
        self.dirty = False


def group_events(schedule: Sequence[tuple], reduce_every: int) -> List[tuple]:
    """("reduce", window) / ("gather", tally) / ("look", tally) of a schedule, in order."""
    m = GroupModel(reduce_every)
    for op in schedule:
        if op[0] == "look":
            m.look(op[1])
        else:
            for tt, tally in timesteps([op]):
                m.step(tt, tally)
    return m.events


def windows(events: Sequence[tuple]) -> List[Tuple[int, ...]]:
    return [ev[1] for ev in events if ev[0] == "reduce"]


def rank_order_looks(events: Sequence[tuple], deltas: Sequence[Dict[tuple, np.ndarray]],
                     ncells: int) -> List[np.ndarray]:
    """The tally at every look of the peer-memory flavour, in float64, addition by addition
    (group.cu): a reduction adds (((0 + delta_0) + delta_1) + ... + delta_{N-1}) to the owned
    value of every cell; a gather adds the owned value to the tally and zeroes it.
    ``deltas[r][window]`` is rank r's buffer after the timesteps of that window."""
    owned = np.zeros(ncells)
    tallies = {"A": np.zeros(ncells), "B": np.zeros(ncells)}
    looks = []
    for ev in events:
        if ev[0] == "reduce":
            s = np.zeros(ncells)
            for per_rank in deltas:
                s = s + per_rank[ev[1]]
            owned = owned + s
        elif ev[0] == "gather":
            tallies[ev[1]] = tallies[ev[1]] + owned
            owned = np.zeros(ncells)
        else:
            looks.append(tallies[ev[1]].copy())
    return looks


def summation_bound_violations(events: Sequence[tuple], deltas: Sequence[Dict[tuple, np.ndarray]],
                               got_looks: Sequence[np.ndarray], ncells: int) -> List[str]:
    """For a flavour that sums in an order of its own (NCCL): at every look, per cell,
    |got - fsum(terms)| <= k 2^-53 sum|terms|, where the terms are every rank's delta of every
    window gathered into that tally and k counts the additions that reached the cell (ranks
    times windows, plus the gathers)."""
    terms: Dict[str, list] = {"A": [], "B": []}
    gathers = {"A": 0, "B": 0}
    pending: list = []
    bad = []
    li = 0
    for ev in events:
        if ev[0] == "reduce":
            pending += [per_rank[ev[1]] for per_rank in deltas]
        elif ev[0] == "gather":
            terms[ev[1]] += pending
            gathers[ev[1]] += 1
            pending = []
        else:
            got = got_looks[li]
            li += 1
            ts = terms[ev[1]]
            if not ts:
                if np.any(got != 0.0):
                    bad.append(f"look {li - 1}: nonzero tally before any gather")
                continue
            stack = np.stack(ts)
            k = len(ts) + gathers[ev[1]]
            for i in np.flatnonzero(np.any(stack != 0.0, axis=0) | (got != 0.0)):
                col = stack[:, i]
                exact = math.fsum(col)
                if abs(got[i] - exact) > k * 2.0 ** -53 * float(np.sum(np.abs(col))):
                    bad.append(f"look {li - 1} cell {i}: {got[i]!r} vs fsum {exact!r}")
                    break
    return bad


# -------------------------------------------------------------------------------- cases --


@dataclass(frozen=True)
class Case:
    """One run of a sharded bank: a mesh (MESHES) or a small deck, an injected bank of
    `nparticles` or an exact_bank, the group options and a schedule. `offset` places the
    caller's tallies `offset` doubles past a 256-byte aligned allocation."""
    mesh: str
    bank: str                 # "inject" | "exact"
    reduce_every: int
    reduce_ctas: int
    schedule: str
    nparticles: int = 0       # inject on a mesh: particles (a deck: its own count)
    offset: int = 0
    collective: int = 1

    @property
    def id(self) -> str:
        s = f"{self.mesh}-{self.bank}-every{self.reduce_every}-ctas{self.reduce_ctas}-{self.schedule}"
        if self.offset:
            s += f"-off{self.offset}"
        if not self.collective:
            s += "-nccl"
        return s

    @property
    def iterations(self) -> int:
        return max(tt for tt, _ in timesteps(SCHEDULES[self.schedule]))

    def problem(self, nranks: int) -> Problem:
        if self.mesh in MESHES:
            n = nranks * MESHES[self.mesh][1] if self.bank == "exact" else self.nparticles
            return mesh_problem(self.mesh, n, self.iterations, self.bank == "exact")
        return build_problem(self.mesh, iterations=self.iterations)

    def host_bank(self, prob: Problem, nranks: int, port) -> HostBank:
        """The whole bank (all shards, injection order)."""
        return exact_bank(prob, nranks) if self.bank == "exact" else port.inject(prob)


def layout(ncells: int, nranks: int) -> List[Tuple[int, int]]:
    """(begin, count) of every owned slice (empty ones included) of group_layout."""
    chunk, _ = owned_slice_layout(ncells, nranks)
    out = []
    for r in range(nranks):
        begin = r * chunk
        out.append((begin, max(0, min(begin + chunk, ncells) - begin)))
    return out
