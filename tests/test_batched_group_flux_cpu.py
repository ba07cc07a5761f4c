"""The batched group flux without a device: its three entry points refuse a handle that is not a
bank, and the attach call bad groups and edges, before they need a GPU; Simulation refuses the
combinations of group_flux_batches it cannot serve; and the premise the GPU tests rely on holds
for the reference: the group flux reference (tests/group_flux_reference.c) run on every batch's
particle range with the whole run's ntotal gives batch group fluxes that sum to the whole run's
group flux."""
import ctypes as C

import numpy as np
import pytest

from group_flux_reference import group_flux_reference
from neutral_b200.bank import ParticleSoA
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.host import EXPORTED_SYMBOLS, NeutralB200Error, Simulation
from test_flux_tally_cpu import rel_close
from test_group_flux_cpu import edge_sets


def test_entry_points_refuse_a_non_bank_without_a_device(lib):
    junk = (C.c_double * 16)()
    handle = C.cast(C.addressof(junk), C.POINTER(ParticleSoA))
    good = np.array([1.0, 10.0, 100.0])
    groups = np.zeros(2)
    total = C.c_double(0.0)
    calls = {
        "nb200_bank_set_batched_group_flux_tally":
            lambda h: lib.nb200_bank_set_batched_group_flux_tally(h, C.addressof(junk), 4,
                                                                  good.ctypes.data, 2),
        "nb200_bank_group_flux_batches":
            lambda h: lib.nb200_bank_group_flux_batches(h, C.addressof(junk), 4, 2),
        "nb200_bank_group_flux_relerr":
            lambda h: lib.nb200_bank_group_flux_relerr(h, C.addressof(junk), groups.ctypes.data,
                                                       C.byref(total)),
    }
    for name, call in calls.items():
        assert name in EXPORTED_SYMBOLS
        for h in (handle, None):
            assert call(h) == -3, name
            assert b"not a bank handle" in lib.nb200_last_error(), name
    assert lib.nb200_bank_set_batched_group_flux_tally(None, None, 0, None, 0) == -3
    assert b"not a bank handle" in lib.nb200_last_error()
    assert total.value == 0.0 and not np.any(groups)


def test_attach_refuses_bad_groups_and_edges_without_a_device(lib):
    """The groups and edges are checked first, on the host, as for the unbatched group flux."""
    junk = (C.c_double * 16)()
    handle = C.cast(C.addressof(junk), C.POINTER(ParticleSoA))

    def call(edges, ngroups):
        e = None if edges is None else np.ascontiguousarray(edges, dtype=np.float64)
        return lib.nb200_bank_set_batched_group_flux_tally(
            handle, C.addressof(junk), 4, None if e is None else e.ctypes.data, ngroups)

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
    assert b"nb200_bank_set_batched_group_flux_tally" in lib.nb200_last_error()


def test_simulation_refuses_what_it_cannot_batch(lib):
    """group_flux_batches needs flux_groups and tally_batches and excludes flux_tally; flux_groups
    with tally_batches still needs the flag. All refused before anything needs a GPU."""
    prob = build_problem("csp_small")
    edges = [1.0, 2.0]
    for kw in (dict(tally_batches=4), dict(flux_groups=edges),
               dict(flux_groups=edges, tally_batches=4, flux_tally=True)):
        with pytest.raises(NeutralB200Error, match="group_flux_batches"):
            Simulation(prob, group_flux_batches=True, **kw)
    with pytest.raises(NeutralB200Error, match="flux_groups.*group_flux_batches"):
        Simulation(prob, flux_groups=edges, tally_batches=4)


@pytest.mark.parametrize("B", [2, 7, 16])
def test_batch_references_sum_to_the_whole_run(port, B):
    """csp_small, 8 log groups and 32 narrow ones: the group flux reference on the particles of
    every batch [first_b, first_b + n_b), each with the whole run's ntotal, sums over the batches
    to the whole run's group flux (1e-12 per cell), after every timestep."""
    prob = build_problem("csp_small")
    d = prob.deck
    for key in ("log8", "narrow32"):
        edges = edge_sets(d.initial_energy)[key]
        size = (edges.size - 1) * d.nx * d.ny
        whole_bank = port.inject(prob)
        whole_tally, whole = np.zeros(d.nx * d.ny), np.zeros(size)
        ranges = [shard_range(d.nparticles, b, B) for b in range(B)]
        banks = [port.inject(prob, pid0=f, count=n) for f, n in ranges]
        tallies = [np.zeros(d.nx * d.ny) for _ in range(B)]
        fluxes = [np.zeros(size) for _ in range(B)]
        for tt in range(1, d.iterations + 1):
            group_flux_reference().step(prob, whole_bank, tt, whole_tally, gflux=whole,
                                        edges=edges)
            for b, (f, _) in enumerate(ranges):
                group_flux_reference().step(prob, banks[b], tt, tallies[b], pid0=f,
                                            ntotal=d.nparticles, gflux=fluxes[b], edges=edges)
            assert np.count_nonzero(whole) > 0
            assert all(np.count_nonzero(fl) > 0 for fl in fluxes), (key, tt)
            assert rel_close(sum(fluxes), whole, 1e-12), (key, tt)
