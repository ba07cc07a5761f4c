"""The track-length flux tally without a device. Its reference (tests/flux_reference.c: the oracle
port's timestep with a flux output) replays the unmodified port's histories and energy tally bit
for bit, sums to the distance travelled on a deck without
collisions, relates to the energy tally through the deposition's cross section and response,
and equals the chord lengths of an independent ray march; the C entry point refuses a handle
that is not a bank without needing a GPU."""
import ctypes as C

import numpy as np
import pytest

from neutral_b200.bank import HostBank, ParticleSoA
from flux_reference import flux_reference
from neutral_b200.decks import Deck, Problem, build_problem, cross_section_table, density_field, \
    mesh_edges, source_box

# neutral_data.h:17-24, as the oracle port and the kernel write them
EV_TO_J = 1.60217646e-19
AVOGADROS = 6.02214085774e23
BARNS = 1.0e-28
PARTICLE_MASS = 1.674927471213e-27
MASS_NO = 1.0e2
MOLAR_MASS = 1.0e-2


def speed_of(e):
    return np.sqrt((2.0 * e * EV_TO_J) / PARTICLE_MASS)


def rel_close(a, b, rtol):
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b))))


@pytest.fixture
def one_thread(port):
    """The tallies of the port and the reference are OpenMP atomics (one libgomp serves both): one thread makes their summation order, and so
    their bits, repeatable."""
    omp = port.lib
    omp.omp_get_max_threads.restype = C.c_int
    prev = omp.omp_get_max_threads()
    omp.omp_set_num_threads(1)
    yield
    omp.omp_set_num_threads(prev)


def port_run(port, prob, step, with_flux):
    d = prob.deck
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    flux = np.zeros(d.nx * d.ny) if with_flux else None
    counters = np.zeros((3, len(bank)), dtype=np.uint64)
    kw = dict(flux=flux) if with_flux is not None else {}
    counts = [step(prob, bank, tt, tally, counters=counters, **kw)
              for tt in range(1, d.iterations + 1)]
    return dict(bank=bank, tally=tally, flux=flux, counts=counts, counters=counters)


@pytest.mark.parametrize("name", ["csp_small", "mixed_small", "scatter_small", "split_small"])
def test_flux_reference_replays_the_port(port, one_thread, name):
    """(a) The reference without and with the flux array gives the counts, per-particle counters,
    bank and energy tally of the unmodified oracle port, bit for bit."""
    prob = build_problem(name)
    want = port_run(port, prob, port.step, None)
    for with_flux in (False, True):
        got = port_run(port, prob, flux_reference().step, with_flux)
        assert got["counts"] == want["counts"], with_flux
        assert np.array_equal(got["counters"], want["counters"]), with_flux
        assert sum(got["bank"].bit_equal(want["bank"]).values()) == 0, with_flux
        assert np.array_equal(got["tally"].view(np.uint64), want["tally"].view(np.uint64))
    assert np.count_nonzero(got["flux"]) > 0


def stream_expectations(port, prob):
    """On stream (no collisions, unit weights, one energy): the flux of a timestep sums to
    v(E0) dt, and energy = flux (sigma_t BARNS) response nd in every cell."""
    d = prob.deck
    e = d.initial_energy
    (sk, sv), (ak, av) = prob.cs_scatter, prob.cs_absorb
    sig_s, sig_a = port.cs_lookup(sk, sv, e), port.cs_lookup(ak, av, e)
    sig_t = sig_s + sig_a
    exit_scatter = e * ((MASS_NO * MASS_NO + MASS_NO + 1) / ((MASS_NO + 1) * (MASS_NO + 1)))
    response = e - (1.0 - sig_a / sig_t) * exit_scatter - (sig_a / sig_t) * 0.0
    nd = prob.density.ravel() * AVOGADROS / MOLAR_MASS
    return speed_of(e) * d.dt, (sig_t * BARNS) * response * nd


def check_stream(step_sums, want_sum, flux, tally, factor):
    for s in step_sums:
        assert abs(s - want_sum) <= 1e-12 * want_sum, (s, want_sum)
    assert rel_close(tally, flux * factor, 1e-12)
    assert np.all((flux == 0.0) == (tally == 0.0))


def test_reference_stream_sums_to_the_distance_travelled(port):
    """(b) on the flux reference."""
    prob = build_problem("stream_small")
    d = prob.deck
    want_sum, factor = stream_expectations(port, prob)
    bank = port.inject(prob)
    tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    sums = []
    for tt in range(1, d.iterations + 1):
        before = flux.sum()
        _, collisions, processed = flux_reference().step(prob, bank, tt, tally, flux=flux)
        assert collisions == 0 and processed == d.nparticles
        sums.append(flux.sum() - before)
    assert np.all(bank.weight == 1.0) and np.all(bank.energy == d.initial_energy)
    check_stream(sums, want_sum, flux, tally, factor)


# ---- one particle on a generic angle through a mesh it cannot collide in ----------------------
RAY_START = (1.3, 2.2)
RAY_ANGLE = 0.61   # radians: both direction components positive, no edge hit twice at once
RAY_LENGTH = 4.0   # per timestep, in the mesh's length unit; 2 steps stay inside the 10 x 10 mesh
RAY_STEPS = 2


def ray_problem() -> Problem:
    """A 10 x 10 mesh of unit cells, density 1e-30 (no collision in any timestep), one particle
    whose timestep covers RAY_LENGTH."""
    e0 = 1.0e6
    deck = Deck(path="one_ray.params", nx=10, ny=10, dt=RAY_LENGTH / float(speed_of(e0)),
                iterations=RAY_STEPS, nparticles=1, initial_energy=e0,
                source=(0.1, 0.1, 0.2, 0.2), problems=[(1.0e-30, 0.0, 0.0, 1.0, 1.0)],
                width=10.0, height=10.0)
    edgex, edgey = mesh_edges(deck)
    return Problem(deck=deck, edgex=edgex, edgey=edgey,
                   density=density_field(deck, edgex, edgey),
                   source=source_box(deck, edgex, edgey),
                   cs_scatter=cross_section_table(), cs_absorb=cross_section_table())


def ray_bank(prob) -> HostBank:
    bank = HostBank.empty(1)
    x, y = RAY_START
    bank.x[0], bank.y[0] = x, y
    bank.omega_x[0], bank.omega_y[0] = np.cos(RAY_ANGLE), np.sin(RAY_ANGLE)
    bank.energy[0], bank.weight[0] = prob.deck.initial_energy, 1.0
    bank.dt_to_census[0] = prob.deck.dt
    bank.cellx[0] = int(np.searchsorted(prob.edgex, x, side="right") - 1)
    bank.celly[0] = int(np.searchsorted(prob.edgey, y, side="right") - 1)
    return bank


def ray_march(prob, length) -> np.ndarray:
    """(ny * nx) chord length of the straight ray from RAY_START in every cell: the distances
    at which it crosses a grid line, sorted, cut the ray into segments, each inside one cell."""
    x0, y0 = RAY_START
    ox, oy = np.cos(RAY_ANGLE), np.sin(RAY_ANGLE)
    ts = [0.0, length]
    ts += [(e - x0) / ox for e in prob.edgex if 0.0 < (e - x0) / ox < length]
    ts += [(e - y0) / oy for e in prob.edgey if 0.0 < (e - y0) / oy < length]
    ts = np.sort(np.array(ts))
    out = np.zeros((prob.deck.ny, prob.deck.nx))
    for t0, t1 in zip(ts[:-1], ts[1:]):
        tm = 0.5 * (t0 + t1)
        cx = int(np.searchsorted(prob.edgex, x0 + tm * ox, side="right") - 1)
        cy = int(np.searchsorted(prob.edgey, y0 + tm * oy, side="right") - 1)
        out[cy, cx] += t1 - t0
    return out.ravel()


def check_chords(flux, prob):
    want = ray_march(prob, RAY_LENGTH * RAY_STEPS)
    assert np.count_nonzero(want) >= 10
    assert np.array_equal(flux != 0.0, want != 0.0)
    assert rel_close(flux, want, 1e-12), np.max(np.abs(flux - want))


def test_reference_chord_lengths():
    """(c) on the flux reference: per-cell flux = chord lengths of the ray (ntotal = 1)."""
    prob = ray_problem()
    d = prob.deck
    bank = ray_bank(prob)
    tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        f, c, p = flux_reference().step(prob, bank, tt, tally, flux=flux)
        assert c == 0 and p == 1
    assert bank.dead[0] == 0
    check_chords(flux, prob)


def test_set_flux_tally_refuses_a_non_bank_without_a_device(lib):
    """(d) the entry point checks its handle before it needs a GPU."""
    junk = (C.c_double * 16)()
    handle = C.cast(C.addressof(junk), C.POINTER(ParticleSoA))
    assert lib.nb200_bank_set_flux_tally(handle, C.addressof(junk), 16) == -3
    assert b"not a bank handle" in lib.nb200_last_error()
    assert lib.nb200_bank_set_flux_tally(None, None, 0) == -3
