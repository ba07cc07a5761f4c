"""The energy-group flux tally without a device. Its reference (tests/group_flux_reference.c: the
oracle port's timestep with a group-resolved flux output) replays the unmodified port's histories
and energy tally bit for bit, equals the plain flux reference with one group covering every
energy, and on a deck without collisions puts a timestep's whole distance travelled into the group
of the initial energy; the C entry point refuses a handle that is not a bank and bad energy edges
without needing a GPU."""
import ctypes as C

import numpy as np
import pytest

from flux_reference import flux_reference
from group_flux_reference import group_flux_reference
from neutral_b200.bank import ParticleSoA
from neutral_b200.decks import build_problem
from neutral_b200.host import NeutralB200Error, Simulation
from test_flux_tally_cpu import one_thread, port_run, rel_close, stream_expectations  # noqa: F401


def edge_sets(e0: float) -> dict:
    """The energy edges (eV) the tests run for a deck of initial energy e0. Energies only fall
    from e0, and a particle below 1 eV dies at its next absorption."""
    return {
        # (a) one group covering every energy
        "one": np.array([0.0, 2.0 * e0]),
        # (b) 8 logarithmic groups, covering every energy too
        "log8": np.geomspace(1.0e-3, 2.0 * e0, 9),
        # (c) 32 narrow groups just below e0: one elastic scatter (A = 100) loses up to 3.9 %, so
        # most scatters of the first few collisions change group
        "narrow32": np.linspace(0.97 * e0, e0 * (1.0 + 1.0e-6), 33),
        # (d) e0 itself above the last edge, everything below 0.5 e0 below the first
        "gaps": np.array([0.5 * e0, 0.9 * e0, 0.99 * e0]),
    }


COVERING = ("one", "log8")  # the edge sets under which no energy goes unscored


def group_run(port, prob, edges):
    """The group flux reference over the deck's timesteps from the port's injected bank: counts,
    counters, bank, tally and the (G, ncells) group flux."""
    d = prob.deck
    gflux = np.zeros((edges.size - 1) * d.nx * d.ny)

    def step(*args, **kw):
        return group_flux_reference().step(*args, gflux=gflux, edges=edges, **kw)

    out = port_run(port, prob, step, None)
    out["gflux"] = gflux.reshape(edges.size - 1, d.nx * d.ny)
    return out


@pytest.mark.parametrize("name", ["csp_small", "mixed_small", "scatter_small", "split_small"])
def test_group_reference_replays_the_port(port, one_thread, name):  # noqa: F811
    """The group flux reference gives the counts, per-particle counters, bank and energy tally
    of the unmodified oracle port, bit for bit, whatever the edges."""
    prob = build_problem(name)
    want = port_run(port, prob, port.step, None)
    for key in ("one", "narrow32"):
        got = group_run(port, prob, edge_sets(prob.deck.initial_energy)[key])
        assert got["counts"] == want["counts"], key
        assert np.array_equal(got["counters"], want["counters"]), key
        assert sum(got["bank"].bit_equal(want["bank"]).values()) == 0, key
        assert np.array_equal(got["tally"].view(np.uint64), want["tally"].view(np.uint64)), key
        assert np.count_nonzero(got["gflux"]) > 0, key


@pytest.mark.parametrize("name", ["csp_small", "mixed_small", "scatter_small", "split_small"])
def test_one_group_is_the_plain_flux(port, name):
    """With one group covering every energy the group flux equals tests/flux_reference.c's flux
    (1e-12 per cell: the plain reference sums consecutive collisions' segments before it
    scales them, this one deposits every segment on its own). Every covering edge set sums over
    the groups to the same flux."""
    prob = build_problem(name)
    d = prob.deck
    bank = port.inject(prob)
    tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, bank, tt, tally, flux=flux)
    assert np.count_nonzero(flux) > 0
    for key in COVERING:
        got = group_run(port, prob, edge_sets(d.initial_energy)[key])["gflux"]
        if key == "one":
            assert rel_close(got[0], flux, 1e-12), np.max(np.abs(got[0] - flux))
        assert rel_close(got.sum(axis=0), flux, 1e-12), key


def test_edges_that_leave_energies_out_score_less(port):
    """(c) and (d) on csp_small: a narrow band below e0 and edges that leave e0 itself out score
    a part of the covering flux, never more in a cell than the covering flux's share there."""
    prob = build_problem("csp_small")
    sets = edge_sets(prob.deck.initial_energy)
    total = group_run(port, prob, sets["one"])["gflux"][0]
    for key in ("narrow32", "gaps"):
        got = group_run(port, prob, sets[key])["gflux"]
        part = got.sum(axis=0)
        assert np.count_nonzero(got) > 0 and 0.0 < part.sum() < total.sum(), key
        assert np.all(part <= total * (1.0 + 1e-12)), key
        if key == "narrow32":
            # the groups that the first scatters land in all see flux
            assert np.count_nonzero(got.sum(axis=1)) >= 16


def test_stream_lands_in_the_group_of_the_initial_energy(port):
    """On stream_small (one energy, no collisions): all flux is in the group holding 1e6 eV, the
    other groups are exactly 0, and every timestep sums to v(E0) dt."""
    prob = build_problem("stream_small")
    d = prob.deck
    assert d.initial_energy == 1.0e6
    edges = np.geomspace(1.0e-3, 1.0e8, 12)
    g0 = int(np.searchsorted(edges, d.initial_energy, side="right") - 1)
    want_sum, _ = stream_expectations(port, prob)
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    gflux = np.zeros((edges.size - 1) * d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        before = gflux.sum()
        _, collisions, processed = group_flux_reference().step(prob, bank, tt, tally,
                                                               gflux=gflux, edges=edges)
        assert collisions == 0 and processed == d.nparticles
        s = gflux.sum() - before
        assert abs(s - want_sum) <= 1e-12 * want_sum, (tt, s, want_sum)
    g = gflux.reshape(edges.size - 1, -1)
    assert np.count_nonzero(g[g0]) > 0
    assert not np.any(np.delete(g, g0, axis=0))


def test_set_group_flux_tally_refuses_without_a_device(lib):
    """The entry point checks its handle and its edges before it needs a GPU."""
    junk = (C.c_double * 16)()
    handle = C.cast(C.addressof(junk), C.POINTER(ParticleSoA))
    good = np.array([1.0, 10.0, 100.0])

    def call(edges, ngroups, h=handle):
        e = None if edges is None else np.ascontiguousarray(edges, dtype=np.float64)
        return lib.nb200_bank_set_group_flux_tally(h, C.addressof(junk), 4,
                                                   None if e is None else e.ctypes.data, ngroups)

    assert call(good, 2) == -3
    assert b"not a bank handle" in lib.nb200_last_error()
    assert lib.nb200_bank_set_group_flux_tally(None, None, 0, None, 0) == -3
    assert b"not a bank handle" in lib.nb200_last_error()
    for ngroups in (0, -1, 257):
        assert call(np.arange(max(ngroups, 0) + 1, dtype=np.float64) + 1.0, ngroups) == -3
        assert b"ngroups" in lib.nb200_last_error(), ngroups
    assert call(None, 2) == -3
    assert b"no energy edges" in lib.nb200_last_error()
    for bad in ([1.0, np.nan, 100.0], [1.0, np.inf, 1e300], [-np.inf, 1.0, 2.0],
                [1.0, 10.0, 10.0], [100.0, 10.0, 1.0]):
        assert call(bad, 2) == -3, bad
        assert b"finite and strictly increasing" in lib.nb200_last_error(), bad
    assert call(np.arange(257, dtype=np.float64), 256) == -3  # 256 groups pass, the handle not
    assert b"not a bank handle" in lib.nb200_last_error()


def test_simulation_refuses_two_fluxes(lib):
    """flux_groups with flux_tally or tally_batches is refused before anything needs a GPU."""
    prob = build_problem("csp_small")
    for kw in (dict(flux_tally=True), dict(tally_batches=4)):
        with pytest.raises(NeutralB200Error, match="flux_groups"):
            Simulation(prob, flux_groups=[1.0, 2.0], **kw)
