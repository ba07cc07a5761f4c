"""The crafted edge-case banks (tests/edge_banks.py) without a device: every input obeys the
contract of valid banks, the oracle port runs every problem and bank to finite results, every
category reaches the branch it was built for (witnessed from the inputs and the port's counters
and banks), and in `vacuum` the port's flights equal an exact rational ray reference."""
import math

import numpy as np
import pytest

import edge_banks as eb
from flux_reference import flux_reference

CASES = eb.all_cases()
IDS = [c.id for c in CASES]
VACUUM = [c for c in CASES if c.problem == "vacuum" and c.label != "dead"]

_RUNS = {}


def port_run(port, case):
    """The port (through the flux reference, which replays it bit for bit) over STEPS
    timesteps: banks and per-particle counters after every timestep, tally and flux."""
    if case.id not in _RUNS:
        d = case.prob.deck
        bank = case.bank.copy()
        tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
        ctr = np.zeros((3, len(bank)), dtype=np.uint64)
        banks, ctrs, counts = [], [], []
        for tt in range(1, d.iterations + 1):
            counts.append(flux_reference().step(case.prob, bank, tt, tally, counters=ctr,
                                                flux=flux))
            banks.append(bank.copy())
            ctrs.append(ctr.copy())
        _RUNS[case.id] = dict(banks=banks, counters=ctrs, counts=counts, tally=tally, flux=flux)
    return _RUNS[case.id]


def by_id(ident):
    return CASES[IDS.index(ident)]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_inputs_obey_the_contract(case):
    assert eb.contract_violations(case.prob, case.bank) == []
    assert len(case.bank) == case.prob.deck.nparticles
    if case.label == "mixed":
        assert len(case.bank) % 32 != 0, "the mixed bank has a ragged count"
        assert len(set(case.tags)) >= 5
        assert 0 < np.count_nonzero(case.bank.dead) < len(case.bank)
    else:
        assert set(case.tags) <= {case.label}


def test_the_contract_check_sees_every_violation():
    case = by_id("edges-mixed")
    live = int(np.flatnonzero(case.bank.dead == 0)[0])

    def bad(**changes):
        bank = case.bank.copy()
        for k, v in changes.items():
            bank.arrays[k][live] = v
        return eb.contract_violations(case.prob, bank)

    assert bad(omega_y=-0.0) == ["omega_y is -0.0"]
    assert bad(cellx=eb.NX) == ["cell out of range"]
    assert bad(x=float(case.prob.edgex[case.bank.cellx[live] + 1]) + 1e-9) == \
        ["position outside its cell"]
    assert bad(energy=math.nan) and bad(weight=-1.0) and bad(weight=math.inf)
    assert bad(energy=1.0e9) == ["energy outside the tables"]
    cx, cy = int(case.bank.cellx[live]), int(case.bank.celly[live])
    assert "zero direction component on that axis's far edge" in \
        bad(omega_x=1.0, omega_y=0.0, y=float(case.prob.edgey[cy + 1]),
            x=float(case.prob.edgex[cx]))
    prob = eb.make_problem("edges", len(case.bank))
    prob.density[0, 0] = -0.0
    assert eb.contract_violations(prob, case.bank) == ["density not finite, negative or -0.0"]
    prob = eb.make_problem("edges", len(case.bank))
    prob.cs_absorb[1][:] = 0.0
    prob.cs_scatter[1][5] = 0.0
    assert eb.contract_violations(prob, case.bank) == ["both tables zero at one energy"]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_port_runs_to_finite_results(port, case):
    r = port_run(port, case)
    for tt, bank in enumerate(r["banks"]):
        for k in ("x", "y", "omega_x", "omega_y", "energy", "weight", "dt_to_census"):
            assert np.all(np.isfinite(bank.arrays[k])), (tt, k)
        mfp = bank.mfp_to_collision
        assert not np.any(np.isnan(mfp) | (mfp == -np.inf)), tt
        # energies never rise, so a final bank inside the tables kept the whole run inside
        assert eb.contract_violations(case.prob, bank) == [], tt
    assert np.all(np.isfinite(r["tally"])) and np.all(np.isfinite(r["flux"]))
    live = case.bank.dead == 0
    assert r["counts"][0][2] == np.count_nonzero(live)
    dead = case.bank.dead == 1
    assert np.all(r["banks"][-1].dead[dead] == 1)
    for k in eb.HostBank.empty(0).arrays:
        assert np.array_equal(r["banks"][-1].arrays[k][dead], case.bank.arrays[k][dead])


# ---- witnesses: every category reaches its branch ------------------------------------------


def test_extreme_cross_sections_leave_the_core_range():
    """Sigma_t of the 1e-80 band lies below 2^-255 and that of the 1e80 band at or above 2^257
    at every energy of the table (kFlagDivBad stays set, every facet divides with the plain
    operator); in the +0.0 and 5e-324 bands 1 / Sigma_t is +inf."""
    prob = eb.make_problem("extreme", 1)
    (keys, s), (_, a) = prob.cs_scatter, prob.cs_absorb
    tot = {rho: [eb.macroscopic_total(rho, float(x), float(y)) for x, y in zip(s, a)]
           for rho in eb.RHO_EXTREME}
    assert max(tot[1.0e-80]) < eb.FM_LO and 1.0 / max(tot[1.0e-80]) >= eb.FM_HI
    assert min(tot[1.0e80]) >= eb.FM_HI and 1.0 / min(tot[1.0e80]) < eb.FM_LO
    for rho in (0.0, 5e-324):
        with np.errstate(divide="ignore"):
            assert all(np.float64(1.0) / np.float64(t) == np.inf for t in tot[rho])
    assert set(np.unique(prob.density)) == {eb.RHO_BACKGROUND, *eb.RHO_EXTREME}


def test_tiny_energies_collide_and_scatter(port):
    """Energies below 2^-255 (outside the scatter block's range: the fallback redraws and
    redoes the event on the plain path) collide in the 1e80 band and scatter at least once."""
    case = by_id("extreme-tiny_energy")
    r = port_run(port, case)
    assert np.all(case.bank.energy < eb.FM_LO)
    first = r["banks"][0]
    collided = r["counters"][0][1] > 0
    scattered = collided & (first.energy != case.bank.energy)
    assert np.count_nonzero(scattered) >= 5
    assert np.all(case.prob.density.ravel()[first.celly * eb.NX + first.cellx][scattered] == 1e80)
    # the normal energies of the 1e80 band take the fallback too (Sigma beyond 2^257)
    case = by_id("extreme-extreme_cells")
    r = port_run(port, case)
    in_band = case.prob.density.ravel()[case.bank.celly * eb.NX + case.bank.cellx] == 1e80
    assert np.all(r["counters"][0][1][in_band] > 100)


def test_one_ev_survives_an_absorption_and_one_ulp_below_dies(port):
    """p_absorb is exactly 1/2 (same tables), so a history that ends with weight 2^-k was
    absorbed k times. At exactly 1.0 eV `e < MIN_ENERGY_OF_INTEREST` is false: some histories
    die only at a second absorption. One ulp below, the first absorption ends every history."""
    one = port_run(port, by_id("edges-one_ev"))["banks"][-1]
    assert np.count_nonzero((one.dead == 1) & (one.weight <= 0.25)) >= 3
    below = by_id("edges-below_one_ev")
    b = port_run(port, below)["banks"][-1]
    assert np.all(b.dead == 1) and np.all(b.weight == 0.5)
    assert np.count_nonzero(b.energy == below.bank.energy) >= 3  # absorbed before any scatter


def test_energy_categories_sit_where_intended():
    keys = eb.make_problem("edges", 1).cs_scatter[0]
    case = by_id("edges-first_key")
    assert np.all(case.bank.energy == keys[0])
    assert np.all(case.prob.density.ravel()[case.bank.celly * eb.NX + case.bank.cellx] == 0.0)
    case = by_id("edges-last_key")
    assert set(case.bank.energy) == {keys[-1], np.nextafter(keys[-1], 0.0)}
    case = by_id("edges-on_key")
    assert np.all(np.isin(case.bank.energy, keys))
    (ck, _), _ = eb.crowded_table()
    case = by_id("tables-crowded_key")
    assert len(ck) > 8192 and np.count_nonzero(np.abs(ck - eb.CROWD_CENTRE) < 1e-5) == eb.CROWD_KEYS
    on = np.isin(case.bank.energy, ck)
    assert np.count_nonzero(on) >= 16 and np.count_nonzero(~on) >= 48
    w = by_id("edges-weight").bank.weight
    assert {0.0, 5e-324, 1e300} == set(w)


def test_edges_has_uniform_zero_tiles_and_crossings_at_tile_borders(port):
    prob = eb.make_problem("edges", 1)
    assert np.all(prob.density[16:32, 32:48] == 0.0) and not np.any(np.signbit(prob.density))
    x0, x1, y0, y1 = eb.DENSE_BLOCK
    assert x0 < 16 < x1 and y0 < 16 <= y1
    x0, x1, y0, y1 = eb.ZERO_BLOCK
    assert x0 < 32 and y0 < 16 and y1 > 32
    # particles starting in the zero block, with same-grid tables: Sigma_t = 0 there
    case = by_id("edges-on_edge")
    start = prob.density.ravel()[case.bank.celly * eb.NX + case.bank.cellx]
    assert np.count_nonzero(start == 0.0) >= 20
    assert np.count_nonzero(port_run(port, case)["counters"][-1][0]) > 0


# ---- the exact ray reference in `vacuum` ------------------------------------------------


@pytest.mark.parametrize("case", VACUUM, ids=[c.id for c in VACUUM])
def test_port_flies_the_exact_rays(port, case):
    """Facet counts exact, positions within 1e-12 of the box, flux within 1e-12 relative of the
    exact chords (w / N per unit length); every corner tie crosses two edges at one point and
    every axis-parallel boundary particle reflects."""
    run = eb.exact_run(case)
    assert run.margin > 1e-9, "an end point lies within 1e-9 of an edge"
    r = port_run(port, case)
    prev = np.zeros(len(case.bank), dtype=np.uint64)
    for t in range(case.prob.deck.iterations):
        facets = r["counters"][t][0] - prev
        prev = r["counters"][t][0]
        assert eb.exact_mismatches(case.prob, run, t, r["banks"][t], facets) == [], t
    assert eb.flux_matches_exact(case.prob, r["flux"], run.flux)
    last = run.steps[-1]
    tags = case.tags[run.slots]
    if case.label in ("corner_tie", "mixed"):
        # (c, c) and (-c, -c) from a cell centre of a square cell meet exact corners; the
        # mixed signs aim at an edge and at an edge pulled in by 1e-13
        ties = [f.ties > 0 for f, g in zip(last, tags) if g == "corner_tie"]
        assert sum(ties) >= len(ties) // 2
    if case.label in ("axis_boundary", "mixed"):
        assert all(f.reflections > 0 for f, g in zip(last, tags) if g == "axis_boundary")
