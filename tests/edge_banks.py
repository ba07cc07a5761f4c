"""Crafted problems and particle banks for the edges of the history kernel (TEST INFRASTRUCTURE).

Injected banks only ever hold random angles, the deck's energy and weight 1, and the decks'
densities are at least 1e-30 with the reference's cross-section table. The banks built here reach
what those never do: direction components that are exactly zero, exact corner ties, positions on
cell edges, energies on table keys and at MIN_ENERGY_OF_INTEREST, energies and cross sections
outside the range of the kernel's branch-free division cores, extreme weights, densities of +0.0,
denormals and 1e+-80, and cross-section tables of 2 entries or with thousands of keys in one
bucket of the staged lookup.

Every particle carries a category tag (``Case.tags``), so that a failure names what kind of
particle went wrong. :func:`cases` returns, for one problem, a mixed bank of every category
(shuffled, with a ragged count, so that the categories share sort classes and warps) and one bank
per category. :func:`contract_violations` lists what a problem and bank must not contain: inputs
on which the reference itself has no defined result (see the notes there).

Plain numpy; nothing here runs a kernel.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from fractions import Fraction
from typing import Dict, List, Tuple

import numpy as np

from neutral_b200.bank import HostBank
from neutral_b200.decks import Deck, Problem, build_problem, cross_section_table, mesh_edges, \
    source_box

# neutral_data.h:17-24, as the oracle port and the kernel write them
EV_TO_J = 1.60217646e-19
AVOGADROS = 6.02214085774e23
BARNS = 1.0e-28
PARTICLE_MASS = 1.674927471213e-27
MOLAR_MASS = 1.0e-2
MIN_ENERGY = 1.0
OPEN_BOUND_CORRECTION = 1.0e-13

#: the range in which the kernel's division, reciprocal and root cores are the IEEE result
#: (fm_safe in nb_fastmath.cuh): 2^-255 <= |v| < 2^257
FM_LO, FM_HI = 2.0 ** -255, 2.0 ** 257

STEPS = 3
PROBLEMS = ("edges", "extreme", "tables", "vacuum")

# the 48 x 40 mesh of square cells 1/8 wide: every edge, centre and half-cell offset is exact
NX, NY, DX = 48, 40, 0.125
E0 = 1.0e6                    # energy of the particles whose energy is not what is tested
DT = 1.0e-7                   # a particle of E0 flies ~1.38 mesh units (11 cells) per timestep
RHO_BACKGROUND = 1.0e-30
RHO_DENSE = 100.0             # a 1 eV particle collides about twice per timestep
DENSE_BLOCK = (8, 20, 4, 20)  # cells [x0, x1) x [y0, y1): straddles the 16-cell tile borders
ZERO_BLOCK = (28, 48, 12, 36)  # contains the whole 16x16 tile (2, 1) and straddles its borders
RHO_EXTREME = (0.0, 5e-324, 1.0e-80, 1.0e80)
# the vacuum's path per timestep, in mesh units: no end point falls within 1e-9 of an edge
VACUUM_PATH = 3.3


def speed_of(e: float) -> float:
    return math.sqrt((2.0 * e * EV_TO_J) / PARTICLE_MASS)


def macroscopic_total(rho: float, sig_s: float, sig_a: float) -> float:
    """Sigma_s + Sigma_a with the reference's operation order (omp3/neutral.c:112-116)."""
    nd = (rho * AVOGADROS) / MOLAR_MASS
    return (nd * sig_s) * BARNS + (nd * sig_a) * BARNS


# ------------------------------------------------------------------------------- tables --


def extreme_table() -> Tuple[Tuple[np.ndarray, np.ndarray], Tuple[np.ndarray, np.ndarray]]:
    """(elastic, capture) on one geometric grid from 1e-90 eV to 1e8 eV, with smooth positive
    values of different bits (no half shortcut), sigma_t between 2 and 6 barns."""
    keys = np.geomspace(1.0e-90, 1.0e8, 4001)
    lk = np.log(keys)
    sig_s = 2.0 + np.sin(lk / 7.0)
    sig_a = 1.5 + 0.5 * np.cos(lk / 11.0)
    return (keys, np.ascontiguousarray(sig_s)), (keys.copy(), np.ascontiguousarray(sig_a))


#: keys of the crowded elastic table: the interval every bank energy of `tables` lies in
CROWD_CENTRE = 1.0e4
CROWD_KEYS = 10_000


def crowded_table() -> Tuple[Tuple[np.ndarray, np.ndarray], Tuple[np.ndarray, np.ndarray]]:
    """(elastic, capture) of `tables`: an elastic table of ~10 200 keys, 10 000 of them within
    1e-9 of CROWD_CENTRE (a few of the 8192 buckets of the staged lookup hold them all), and a
    capture table of 2 entries, both zero (p_absorb = 0: nobody is absorbed)."""
    far = np.geomspace(1.0e-20, 1.0e8, 201)
    crowd = CROWD_CENTRE * (1.0 + np.arange(CROWD_KEYS) * 1.0e-13)
    keys = np.unique(np.concatenate([far, crowd]))
    sig_s = 3.0 + np.sin(np.log(keys)) + np.clip(1.0e9 * (keys / CROWD_CENTRE - 1.0), 0.0, 1.0)
    capture = (np.array([keys[0], keys[-1]]), np.zeros(2))
    return (np.ascontiguousarray(keys), np.ascontiguousarray(sig_s)), capture


# ----------------------------------------------------------------------------- problems --


def _block(rho, block, value):
    x0, x1, y0, y1 = block
    rho[y0:y1, x0:x1] = value


def _density(name: str) -> np.ndarray:
    rho = np.full((NY, NX), RHO_BACKGROUND)
    if name == "edges":
        _block(rho, DENSE_BLOCK, RHO_DENSE)
        _block(rho, ZERO_BLOCK, 0.0)
    elif name == "extreme":
        # four vertical bands, one per extreme density; the background stays in the left
        # columns and between the bands
        for i, r in enumerate(RHO_EXTREME):
            _block(rho, (8 + 10 * i, 16 + 10 * i, 0, NY), r)
    elif name == "vacuum":
        rho[:] = 0.0
    return rho


def make_problem(name: str, nparticles: int) -> Problem:
    """One of PROBLEMS, for a bank of `nparticles` particles (the tally's normalisation)."""
    if name == "tables":
        base = build_problem("csp_small", nparticles=nparticles, iterations=STEPS)
        s, a = crowded_table()
        return Problem(deck=base.deck, edgex=base.edgex, edgey=base.edgey,
                       density=base.density, source=base.source, cs_scatter=s, cs_absorb=a)
    dt = DT if name != "vacuum" else VACUUM_PATH / speed_of(E0)
    deck = Deck(path=f"{name}.params", nx=NX, ny=NY, dt=dt, iterations=STEPS,
                nparticles=nparticles, initial_energy=E0, source=(0.0, 0.0, 1.0, 1.0),
                width=NX * DX, height=NY * DX)
    edgex, edgey = mesh_edges(deck)
    if name == "extreme":
        s, a = extreme_table()
    else:
        s, a = cross_section_table(), cross_section_table()
    return Problem(deck=deck, edgex=edgex, edgey=edgey,
                   density=np.ascontiguousarray(_density(name)),
                   source=source_box(deck, edgex, edgey), cs_scatter=s, cs_absorb=a)


# -------------------------------------------------------------------------------- banks --

C45 = math.sqrt(0.5)
GENERIC_ANGLES = (0.3, 1.9, 3.5, 5.1, 2.6)


@dataclass
class Case:
    """A problem, a bank for it (slot = pid) and the category of every slot."""
    problem: str
    label: str
    prob: Problem
    bank: HostBank
    tags: np.ndarray

    @property
    def id(self) -> str:
        return f"{self.problem}-{self.label}"


class _Builder:
    def __init__(self, prob: Problem):
        self.prob = prob
        self.rows: List[tuple] = []

    def centre(self, cx, cy):
        return (float(self.prob.edgex[cx]) + 0.5 * (self.prob.edgex[cx + 1] - self.prob.edgex[cx]),
                float(self.prob.edgey[cy]) + 0.5 * (self.prob.edgey[cy + 1] - self.prob.edgey[cy]))

    def add(self, tag, cx, cy, ox, oy, e=E0, w=1.0, x=None, y=None, dead=0):
        px, py = self.centre(cx, cy)
        self.rows.append((tag, px if x is None else x, py if y is None else y, ox, oy, e, w,
                          cx, cy, dead))

    def generic(self, tag, cells, e=E0, w=1.0, angles=GENERIC_ANGLES):
        for (cx, cy) in cells:
            for th in angles:
                self.add(tag, cx, cy, math.cos(th), math.sin(th), e, w)


AXIS_DIRS = ((1.0, 0.0), (-1.0, 0.0), (0.0, 1.0), (0.0, -1.0))
CORNER_DIRS = ((C45, C45), (-C45, -C45), (C45, -C45), (-C45, C45))


def _geometry(b: _Builder, interior, nx, ny):
    """axis-parallel, corner-tie and on-edge particles (energy E0, weight 1)."""
    boundary = [(0, ny // 2), (nx - 1, ny // 3), (nx // 2, 0), (nx // 3, ny - 1)]
    corners = [(0, 0), (nx - 1, 0), (0, ny - 1), (nx - 1, ny - 1)]
    for cell in interior + boundary + corners:
        for ox, oy in AXIS_DIRS:
            b.add("axis_boundary" if cell in boundary + corners else "axis", *cell, ox, oy)
    for cell in interior + boundary + corners:
        for ox, oy in CORNER_DIRS:
            b.add("corner_tie", *cell, ox, oy)
    ex, ey = b.prob.edgex, b.prob.edgey
    for (cx, cy) in interior + corners:
        _, yc = b.centre(cx, cy)
        xc, _ = b.centre(cx, cy)
        for th in GENERIC_ANGLES:
            ox, oy = math.cos(th), math.sin(th)
            b.add("on_edge", cx, cy, ox, oy, x=float(ex[cx + 1]))  # far x edge
            b.add("on_edge", cx, cy, ox, oy, x=float(ex[cx]))      # near x edge
            b.add("on_edge", cx, cy, ox, oy, y=float(ey[cy + 1]))
            b.add("on_edge", cx, cy, ox, oy, y=float(ey[cy]))
        # axis-parallel along the axis of the edge it sits on (a zero component with the
        # position on that axis's far edge has no defined result, see contract_violations)
        for ox in (1.0, -1.0):
            b.add("on_edge", cx, cy, ox, 0.0, x=float(ex[cx + 1]), y=yc)
            b.add("on_edge", cx, cy, ox, 0.0, x=float(ex[cx]), y=yc)
        for oy in (1.0, -1.0):
            b.add("on_edge", cx, cy, 0.0, oy, x=xc, y=float(ey[cy + 1]))
            b.add("on_edge", cx, cy, 0.0, oy, x=xc, y=float(ey[cy]))
        # the far corner itself
        b.add("on_edge", cx, cy, C45, C45, x=float(ex[cx + 1]), y=float(ey[cy + 1]))
        b.add("on_edge", cx, cy, -C45, C45, x=float(ex[cx]), y=float(ey[cy + 1]))


def _dead(b: _Builder, cells):
    for i, (cx, cy) in enumerate(cells):
        b.add("dead", cx, cy, math.cos(i + 0.5), math.sin(i + 0.5), dead=1)


def _edges(b: _Builder):
    keys = b.prob.cs_scatter[0]
    # interior cells: background, dense (on both sides of a tile border) and zero density
    interior = [(5, 30), (15, 10), (16, 10), (40, 24), (31, 20)]
    _geometry(b, interior, NX, NY)
    # energies on keys: mid-table keys in the dense block (they collide) and in the background;
    # the first key only where nothing collides (a scatter would leave the table)
    rng = np.random.default_rng(5)
    for k in rng.choice(np.arange(20000, len(keys) - 1), 12, replace=False):
        b.generic("on_key", [(14, 8)], e=float(keys[k]), angles=(0.7,))
        b.generic("on_key", [(3, 33)], e=float(keys[k]), angles=(2.2,))
    b.generic("first_key", [(40, 24), (38, 20)], e=float(keys[0]))
    b.generic("last_key", [(14, 14), (3, 3)], e=float(keys[-1]))
    b.generic("last_key", [(14, 14), (3, 3)], e=float(np.nextafter(keys[-1], 0.0)))
    # MIN_ENERGY_OF_INTEREST exactly (an absorption does not end the history) and one ulp below
    one_cells = [(10, 6), (12, 9), (17, 12), (19, 18), (9, 17)]
    b.generic("one_ev", one_cells, e=1.0)
    b.generic("below_one_ev", one_cells, e=float(np.nextafter(1.0, 0.0)))
    # weights: zero and the smallest denormal everywhere; 1e300 slow and away from the dense
    # block (its deposits stay finite)
    b.generic("weight", [(14, 8), (3, 33), (40, 24)], w=0.0)
    b.generic("weight", [(14, 8), (3, 33), (40, 24)], w=5e-324)
    b.generic("weight", [(3, 33), (40, 24)], e=100.0, w=1.0e300)
    _dead(b, [(5, 5), (14, 8), (40, 24), (0, 0), (47, 39)] * 3)


def _extreme(b: _Builder):
    (keys, _), _ = extreme_table()
    band = [(12 + 10 * i, 20) for i in range(len(RHO_EXTREME))]  # one cell per extreme band
    b.generic("extreme_cells", band + [(12 + 10 * i, 0) for i in range(len(RHO_EXTREME))])
    # energies below 2^-255: they collide (and scatter) in the 1e80 band
    for e in (1.0e-80, 2.0 ** -280, 3.0e-88):
        b.generic("tiny_energy", [band[3], (band[3][0] + 1, 30), band[2], band[0]], e=e)
    for k in (0, 1, 2000, len(keys) - 2, len(keys) - 1):
        b.generic("on_key", [band[0], band[2]], e=float(keys[k]), angles=(1.1, 4.4))
    b.generic("weight", [band[0], band[1], band[2]], w=5e-324)
    b.generic("weight", [band[0], band[2]], e=100.0, w=1.0e300)
    _geometry(b, [band[0], band[1], band[2], band[3], (3, 20)], NX, NY)
    _dead(b, band * 4)


def _tables(b: _Builder):
    (keys, _), _ = crowded_table()
    crowd = np.flatnonzero(np.abs(keys - CROWD_CENTRE) < 1.0e-3)
    nx, ny = b.prob.deck.nx, b.prob.deck.ny
    bg, dense = [(20, 100), (110, 30)], [(55, 60), (70, 74)]
    rng = np.random.default_rng(9)
    for k in rng.choice(crowd[1:-1], 16, replace=False):
        for e in (keys[k], np.nextafter(keys[k], 0.0), np.nextafter(keys[k], np.inf),
                  0.5 * (keys[k] + keys[k + 1])):
            b.generic("crowded_key", [bg[k % 2], dense[k % 2]], e=float(e), angles=(0.4, 3.9))
    for k in (crowd[0], crowd[-1]):
        b.generic("crowded_key", bg + dense, e=float(keys[k]))
    b.generic("generic", bg + dense, e=1.0e5)
    _geometry(b, [(64, 64), (20, 100)], nx, ny)
    _dead(b, dense * 5)


def _vacuum(b: _Builder):
    _geometry(b, [(5, 30), (15, 10), (16, 16), (40, 24), (31, 20)], NX, NY)
    _dead(b, [(5, 5), (40, 24)] * 4)


_BUILDERS = {"edges": _edges, "extreme": _extreme, "tables": _tables, "vacuum": _vacuum}


def _bank(rows, dt) -> Tuple[HostBank, np.ndarray]:
    bank = HostBank.empty(len(rows))
    for i, (tag, x, y, ox, oy, e, w, cx, cy, dead) in enumerate(rows):
        bank.x[i], bank.y[i] = x, y
        bank.omega_x[i], bank.omega_y[i] = ox, oy
        bank.energy[i], bank.weight[i] = e, w
        bank.dt_to_census[i], bank.mfp_to_collision[i] = dt, 0.0
        bank.cellx[i], bank.celly[i], bank.dead[i] = cx, cy, dead
    return bank, np.array([r[0] for r in rows])


def cases(name: str) -> List[Case]:
    """The mixed bank of problem `name` (label "mixed") and one bank per category."""
    b = _Builder(make_problem(name, 1))
    _BUILDERS[name](b)
    rows = list(b.rows)
    # the mixed bank: every category, shuffled, topped up with generic particles of the first
    # interior cell to a count that is not a multiple of a warp or of a history CTA
    filler = rows[0][1:]
    while len(rows) % 32 == 0:
        rows.append(("generic",) + filler)
    order = np.random.default_rng(17).permutation(len(rows))
    out = []
    groups: Dict[str, list] = {"mixed": [rows[i] for i in order]}
    for r in b.rows:
        groups.setdefault(r[0], []).append(r)
    for label, rs in groups.items():
        prob = make_problem(name, len(rs))
        bank, tags = _bank(rs, prob.deck.dt)
        out.append(Case(name, label, prob, bank, tags))
    return out


def all_cases() -> List[Case]:
    return [c for name in PROBLEMS for c in cases(name)]


# ------------------------------------------------------------------------------ contract --


def contract_violations(prob: Problem, bank: HostBank) -> List[str]:
    """What a problem and bank must not contain; an empty list for valid input.

    * a -0.0 direction component: the reference's arithmetic then gives tx = -inf and a facet
      of length -inf, a NaN position, dt_to_census = +inf and a loop that never ends. Valid
      histories never produce one: reflections negate non-zero components, and a scatter's
      exact-zero sum is +0.0;
    * a zero direction component with the position on that axis's far edge: 0 * inf makes the
      facet distance NaN and the particle jumps to its census point through every edge;
    * a cell out of range, or a position outside its cell's closed interval (the device reads
      out of bounds: banks are not validated on upload);
    * NaN, infinite or negative values, a density of -0.0;
    * an energy outside [first key, last key] of either table (undefined in the reference; the
      port and the kernel clamp). Energies only decrease, so a final bank inside the tables
      shows that the whole run stayed inside;
    * tables that are both zero at one energy (NaN heating, NaN tally), and keys that do not
      increase strictly.
    """
    bad = []
    d = prob.deck
    ex, ey, rho = prob.edgex, prob.edgey, prob.density
    if not (np.all(np.isfinite(rho)) and np.all(rho >= 0.0) and not np.any(np.signbit(rho))):
        bad.append("density not finite, negative or -0.0")
    lo, hi = -math.inf, math.inf
    union = []
    for keys, vals in (prob.cs_scatter, prob.cs_absorb):
        if len(keys) < 2 or not np.all(np.diff(keys) > 0.0):
            bad.append("keys not strictly increasing")
        if not (np.all(np.isfinite(vals)) and np.all(vals >= 0.0)):
            bad.append("cross section not finite or negative")
        lo, hi = max(lo, float(keys[0])), min(hi, float(keys[-1]))
        union.append(keys)
    # sigma_s + sigma_a is piecewise linear between the keys of both tables
    knots = np.unique(np.concatenate(union))
    knots = knots[(knots >= lo) & (knots <= hi)]
    tot = np.interp(knots, *prob.cs_scatter) + np.interp(knots, *prob.cs_absorb)
    if np.any(tot <= 0.0):
        bad.append("both tables zero at one energy")
    live = bank.dead == 0
    if not np.all((bank.dead == 0) | (bank.dead == 1)):
        bad.append("dead not 0/1")
    for k in ("x", "y", "omega_x", "omega_y", "energy", "weight"):
        if not np.all(np.isfinite(bank.arrays[k][live])):
            bad.append(f"{k} not finite")
    if np.any(bank.weight[live] < 0.0) or np.any(np.signbit(bank.weight[live])):
        bad.append("negative weight")
    for k in ("omega_x", "omega_y"):
        o = bank.arrays[k][live]
        if np.any((o == 0.0) & np.signbit(o)):
            bad.append(f"{k} is -0.0")
    e = bank.energy[live]
    if np.any(e < lo) or np.any(e > hi):
        bad.append("energy outside the tables")
    cx, cy = bank.cellx, bank.celly
    if np.any((cx < 0) | (cx >= d.nx) | (cy < 0) | (cy >= d.ny)):
        bad.append("cell out of range")
        return bad
    x, y = bank.x, bank.y
    inside = (x >= ex[cx]) & (x <= ex[cx + 1]) & (y >= ey[cy]) & (y <= ey[cy + 1])
    if not np.all(inside[live]):
        bad.append("position outside its cell")
    nan_x = (bank.omega_x == 0.0) & (x == ex[cx + 1])
    nan_y = (bank.omega_y == 0.0) & (y == ey[cy + 1])
    if np.any((nan_x | nan_y)[live]):
        bad.append("zero direction component on that axis's far edge")
    return bad


# ------------------------------------------------------------------- exact ray reference --


@dataclass
class Flight:
    """One timestep of a particle that cannot collide, in exact rational arithmetic."""
    x: Fraction
    y: Fraction
    ox: float
    oy: float
    cx: int
    cy: int
    facets: int = 0
    ties: int = 0         # crossings of two edges at one point
    reflections: int = 0


def _target(edges, c, o) -> Fraction:
    # omp3/neutral.c:442-450: the far edge for o >= 0, else the near edge pulled in by
    # OPEN_BOUND_CORRECTION (the float subtraction, as the reference computes it)
    return Fraction(float(edges[c + 1])) if o >= 0.0 else \
        Fraction(float(edges[c]) - OPEN_BOUND_CORRECTION)


def exact_step(prob: Problem, f: Flight, path: Fraction, chords: Dict[Tuple[int, int], Fraction],
               margins: List[Fraction]) -> None:
    """Flies `path` (v * dt) from the state `f`, in place: straight lines at the direction
    (ox, oy) - read as exact rationals - cut by the edge targets, reflections at the walls.
    Adds the length flown in every cell to `chords` and the distance of the end point from the
    nearest target to `margins`."""
    d = prob.deck
    ex, ey = prob.edgex, prob.edgey
    left = path
    while True:
        tx = (_target(ex, f.cx, f.ox) - f.x) / Fraction(f.ox) if f.ox != 0.0 else None
        ty = (_target(ey, f.cy, f.oy) - f.y) / Fraction(f.oy) if f.oy != 0.0 else None
        t = min(v for v in (tx, ty) if v is not None)
        if t >= left:
            margins.append(t - left)
            f.x += left * Fraction(f.ox)
            f.y += left * Fraction(f.oy)
            chords[(f.cx, f.cy)] = chords.get((f.cx, f.cy), Fraction(0)) + left
            return
        chords[(f.cx, f.cy)] = chords.get((f.cx, f.cy), Fraction(0)) + t
        left -= t
        f.x += t * Fraction(f.ox)
        f.y += t * Fraction(f.oy)
        if tx == t and ty == t:
            f.ties += 1
        # the port takes the y facet of a tie first; both cross at the same point
        for axis in ("y", "x"):
            if (ty if axis == "y" else tx) != t:
                continue
            f.facets += 1
            o = f.oy if axis == "y" else f.ox
            c = f.cy if axis == "y" else f.cx
            n = d.ny if axis == "y" else d.nx
            cn = c + (1 if o > 0.0 else -1)
            if cn < 0 or cn >= n:
                f.reflections += 1
                if axis == "y":
                    f.oy = -f.oy
                else:
                    f.ox = -f.ox
            elif axis == "y":
                f.cy = cn
            else:
                f.cx = cn


def ray_traceable(bank: HostBank, tags: np.ndarray) -> np.ndarray:
    """Slots whose flights the exact reference covers in `vacuum`: live axis-parallel, corner-tie
    and on-edge particles (every vacuum category but the dead)."""
    return (bank.dead == 0) & np.isin(tags, ["axis", "axis_boundary", "corner_tie", "on_edge",
                                             "generic"])


@dataclass
class ExactRun:
    """The exact reference of a vacuum bank over STEPS timesteps: per timestep the state of
    every traced slot, and the flux w * chord / N per cell summed over the run."""
    slots: np.ndarray
    steps: List[List[Flight]]          # [timestep][index into slots] after that timestep
    facets: np.ndarray                 # (STEPS, len(slots)) facets of each timestep
    flux: np.ndarray                   # (ny * nx) float of the exact sum
    margin: Fraction                   # least distance of an end point from its next target


def exact_run(case: Case) -> ExactRun:
    prob, bank = case.prob, case.bank
    d = prob.deck
    assert not np.any(prob.density), "the exact reference is for a bank that cannot collide"
    slots = np.flatnonzero(ray_traceable(bank, case.tags))
    flights = [Flight(Fraction(float(bank.x[i])), Fraction(float(bank.y[i])),
                      float(bank.omega_x[i]), float(bank.omega_y[i]),
                      int(bank.cellx[i]), int(bank.celly[i])) for i in slots]
    flux = {}
    margins: List[Fraction] = []
    steps, facets = [], np.zeros((d.iterations, len(slots)), dtype=np.uint64)
    for t in range(d.iterations):
        for j, (i, f) in enumerate(zip(slots, flights)):
            chords: Dict[Tuple[int, int], Fraction] = {}
            before = f.facets
            path = Fraction(speed_of(float(bank.energy[i]))) * Fraction(d.dt)
            exact_step(prob, f, path, chords, margins)
            facets[t, j] = f.facets - before
            w = Fraction(float(bank.weight[i]))
            for cell, c in chords.items():
                flux[cell] = flux.get(cell, Fraction(0)) + c * w
        steps.append([Flight(**f.__dict__) for f in flights])
    out = np.zeros(d.nx * d.ny)
    for (cx, cy), v in flux.items():
        out[cy * d.nx + cx] = float(v / d.nparticles)
    return ExactRun(slots, steps, facets, out, min(margins) if margins else Fraction(1))


def _bits(v) -> int:
    return int(np.float64(v).view(np.uint64))


def exact_mismatches(prob: Problem, run: ExactRun, t: int, bank: HostBank,
                     facets: np.ndarray) -> List[str]:
    """Where the bank after timestep t (0-based) and its facets of that timestep (per slot)
    differ from the exact flights: facet counts exactly, cells and direction bits exactly,
    positions within 1e-12 of the box size."""
    box = max(float(prob.edgex[-1] - prob.edgex[0]), float(prob.edgey[-1] - prob.edgey[0]))
    bad = []
    for j, i in enumerate(run.slots):
        f = run.steps[t][j]
        got = (int(facets[i]), int(bank.cellx[i]), int(bank.celly[i]))
        if got != (int(run.facets[t, j]), f.cx, f.cy):
            bad.append(f"slot {i}: facets/cell {got} != {(int(run.facets[t, j]), f.cx, f.cy)}")
        if _bits(bank.omega_x[i]) != _bits(f.ox) or _bits(bank.omega_y[i]) != _bits(f.oy):
            bad.append(f"slot {i}: direction")
        if abs(Fraction(float(bank.x[i])) - f.x) > Fraction(1e-12) * Fraction(box) or \
                abs(Fraction(float(bank.y[i])) - f.y) > Fraction(1e-12) * Fraction(box):
            bad.append(f"slot {i}: position ({bank.x[i]}, {bank.y[i]}) vs "
                       f"({float(f.x)}, {float(f.y)})")
    return bad


def flux_matches_exact(prob: Problem, got: np.ndarray, want: np.ndarray) -> bool:
    """Per cell within 1e-12 relative of the exact chord sum; a cell the exact ray only grazes
    (a corner passage, the 1e-13 of the open-bound correction) is held to 1e-12 of the flux of
    one cell width."""
    dx = float(prob.edgex[1] - prob.edgex[0])
    floor = dx / prob.deck.nparticles
    return bool(np.all(np.abs(got - want) <= 1e-12 * np.maximum(np.abs(want), floor)))
