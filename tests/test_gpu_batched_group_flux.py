"""Group flux batches on the GPU (nb200_bank_set_batched_group_flux_tally): batching the group flux
moves deposits, never histories. Counts, per-particle counters and every bank field are
bit-identical to the unbatched run without flux; after a flush the energy tally and the group
flux equal an unbatched group-flux run's to 1e-10 per cell; every (batch, group) equals the group
flux reference run on the batch's particle range after every timestep; the relative errors per
cell, per group and of the total follow the estimator's formula; one covering group is the
batched flux; every flush path, attachment change and refusal behaves as the header says."""
import ctypes as C

import numpy as np
import pytest

from conftest import SMALL_DECKS
from group_flux_reference import group_flux_reference
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.host import NB200_BAD_OPTION, DeviceArray, Simulation, _soa_p
from test_flux_tally_cpu import stream_expectations
from test_gpu_parity import DEFAULTS, MODES, TALLY_RTOL, tally_close
from test_gpu_tally_batches import _rel_close, _relerr_numpy
from test_group_flux_cpu import edge_sets
from variants import VARIANTS

pytestmark = pytest.mark.gpu

BATCHES = (2, 7, 16)


def _problem(name):
    return VARIANTS[name]() if name in VARIANTS else build_problem(name)


def _set_mode(lib, name):
    for k, v in MODES[name].items():
        assert lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION


def _restore(lib):
    for k, v in DEFAULTS.items():
        lib.nb200_set_option(k.encode(), v)


@pytest.fixture(params=["pipeline", "pipeline-ieee-div"])
def kernel_mode(request, gpu_lib):
    _set_mode(gpu_lib, request.param)
    yield request.param
    _restore(gpu_lib)


def _peek(lib, arr):
    """The device array WITHOUT flushing: accumulated into a scratch buffer on the device."""
    scratch = DeviceArray(arr.n)
    assert lib.nb200_accumulate(scratch.ptr, arr.ptr, arr.n) == 0
    out = scratch.download()
    scratch.free()
    return out


def _groups_close(got, want):
    """The group flux tests' comparison: relative 1e-10 above an absolute floor of the smallest
    normal double (tests/test_gpu_group_flux.py says why)."""
    a, b = np.ravel(got), np.ravel(want)
    return bool(np.all(np.abs(a - b) <= TALLY_RTOL * np.maximum(np.abs(a), np.abs(b)) +
                       np.finfo(np.float64).tiny))


def _sim(prob, B=0, edges=None, flux=False, **kw):
    grouped = dict(flux_groups=edges, group_flux_batches=bool(B)) if edges is not None else {}
    return Simulation(prob, tally_batches=B, flux_tally=flux, **grouped, **kw)


def _run(prob, B=0, edges=None, pipelined=False, flux=False):
    """Per-timestep counts, bank after every timestep (step by step) or at the end (pipelined),
    per-particle counters, the flushed energy tally and group flux (or plain flux), and the
    exported batches."""
    sim = _sim(prob, B, edges, flux)
    sim.inject()
    counts, banks = [], []
    if pipelined:
        counts = [(r.facets, r.collisions, r.processed, r.census, r.deaths)
                  for r in sim.run_pipelined(depth=3)]
        banks.append(sim.bank_to_host())
    else:
        for tt in range(1, prob.deck.iterations + 1):
            r = sim.step(tt)
            counts.append((r.facets, r.collisions, r.processed, r.census, r.deaths))
            banks.append(sim.bank_to_host())
    out = dict(counts=counts, banks=banks, counters=sim.counters_to_host(),
               tally=sim.tally_to_host())
    if edges is not None:
        out["gflux"] = sim.group_flux_to_host().reshape(edges.size - 1, -1)
        if B:
            out["batches"] = sim.group_flux_batches_to_host()
    if flux:
        out["flux"] = sim.flux_to_host().ravel()
        if B:
            out["flux_batches"] = sim.flux_batches_to_host()
    sim.free()
    return out


def _same_histories(got, want, what):
    assert got["counts"] == want["counts"], what
    for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
        diff = a.bit_equal(b)
        assert sum(diff.values()) == 0, (what, tt, diff)
    assert np.array_equal(got["counters"], want["counters"]), what


def _check_batched(prob, pipelined, edges, what):
    d = prob.deck
    G = edges.size - 1
    base = _run(prob, pipelined=pipelined)
    want = _run(prob, edges=edges, pipelined=pipelined)
    assert np.count_nonzero(want["gflux"]) > 0
    for B in BATCHES:
        got = _run(prob, B, edges, pipelined)
        _same_histories(got, base, (what, B))
        assert tally_close(got["tally"], base["tally"]), (what, B)
        assert _groups_close(got["gflux"], want["gflux"]), (what, B)
        assert got["batches"].shape == (B, G, d.ny, d.nx)
        assert _groups_close(got["batches"].sum(axis=0).reshape(G, -1), want["gflux"]), (what, B)


@pytest.mark.parametrize("name", SMALL_DECKS + list(VARIANTS))
def test_histories_unchanged(gpu_lib, kernel_mode, name):
    """1: bit-identical histories against the unbatched run without flux; the energy tally, the
    flushed group flux and the sum of the exported batches within 1e-10 of an unbatched
    group-flux run, step by step and pipelined, B = 2, 7 and 16."""
    prob = _problem(name)
    edges = edge_sets(prob.deck.initial_energy)["log8"]
    for pipelined in (False, True):
        _check_batched(prob, pipelined, edges, (name, pipelined))


@pytest.mark.parametrize("name", ["csp_small", "mixed_small"])
def test_without_the_step_graph(gpu_lib, name):
    """1: the same with the timestep's calls issued one by one (step_graph=0), for narrow
    groups that most scatters leave."""
    _set_mode(gpu_lib, "pipeline-calls")
    try:
        prob = _problem(name)
        _check_batched(prob, False, edge_sets(prob.deck.initial_energy)["narrow32"], name)
    finally:
        _restore(gpu_lib)


@pytest.mark.parametrize("key", ["one", "log8", "narrow32", "gaps"])
@pytest.mark.parametrize("name", ["csp_small", "mixed_small"])
def test_every_batch_and_group_matches_the_reference(gpu_lib, port, name, key):
    """2: after every timestep, every group of every batch equals the group flux reference run
    on particles [first_b, first_b + n_b) with the whole run's ntotal; the energy batches equal
    the same runs' energy tallies (the group reference's energy tally is the oracle port's)."""
    prob = _problem(name)
    d = prob.deck
    edges = edge_sets(d.initial_energy)[key]
    G = edges.size - 1
    B = 7
    sim = _sim(prob, B, edges)
    sim.inject()
    ranges = [shard_range(d.nparticles, b, B) for b in range(B)]
    banks = [port.inject(prob, pid0=f, count=n) for f, n in ranges]
    tallies = [np.zeros(d.nx * d.ny) for _ in range(B)]
    fluxes = [np.zeros(G * d.nx * d.ny) for _ in range(B)]
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        facets = 0
        for b, (f, _) in enumerate(ranges):
            facets += group_flux_reference().step(prob, banks[b], tt, tallies[b], pid0=f,
                                                  ntotal=d.nparticles, gflux=fluxes[b],
                                                  edges=edges)[0]
        assert r.facets == facets, tt
        got = sim.group_flux_batches_to_host().reshape(B, G, -1)
        got_tally = sim.tally_batches_to_host().reshape(B, -1)
        for b in range(B):
            for g in range(G):
                assert _groups_close(got[b, g], fluxes[b].reshape(G, -1)[g]), (tt, b, g)
            assert tally_close(got_tally[b], tallies[b]), (tt, b)
    # every batch scores (edges that leave e0 out may score nothing in a batch's first timestep)
    assert all(np.count_nonzero(f) > 0 for f in fluxes), key
    sim.free()


def _stepped(prob, B, edges, steps=None, **kw):
    sim = _sim(prob, B, edges, **kw)
    sim.inject()
    for tt in range(1, (steps or prob.deck.iterations) + 1):
        sim.step(tt)
    return sim


@pytest.mark.parametrize("name", ["csp_small", "split_small"])
def test_statistics_match_the_formula(gpu_lib, name):
    """3: device R per group and cell, per group total and of the grand total equal the formula
    on the exported batches (1e-12); R is 0 where the mean is 0."""
    prob = build_problem(name)
    d = prob.deck
    B = 16
    edges = edge_sets(d.initial_energy)["log8"]
    G = edges.size - 1
    sim = _stepped(prob, B, edges)
    S = sim.group_flux_batches_to_host().reshape(B, G, -1)
    cell, groups, total = sim.group_flux_relative_error()
    sim.free()
    assert cell.shape == (G, d.ny, d.nx) and groups.shape == (G,)
    want = _relerr_numpy(list(S.reshape(B, -1)), d.nparticles)
    assert _rel_close(cell.ravel(), want, 1e-12)
    assert np.all(cell.ravel()[S.sum(axis=0).ravel() == 0.0] == 0.0)
    assert np.count_nonzero(cell) > 0
    want_groups = _relerr_numpy(list(S.sum(axis=2)), d.nparticles)
    assert _rel_close(groups, want_groups, 1e-12), (groups, want_groups)
    assert np.count_nonzero(groups) >= 2
    want_total = _relerr_numpy([np.array([S[b].sum()]) for b in range(B)], d.nparticles)[0]
    assert abs(total - want_total) <= 1e-12 * abs(want_total)
    assert 0.0 < total < 1.0
    print(f"{name}, {B} batches, {G} groups: R per group {np.array2string(groups, precision=3)}, "
          f"R of the total {total:.3e}")


@pytest.mark.parametrize("name", ["csp_small", "split_small", "mixed_small"])
def test_one_covering_group_is_the_batched_flux(gpu_lib, name):
    """4 and 3: with one group covering every energy the batches equal the batched flux's
    (nb200_bank_set_batched_flux_tally) to 1e-10 per cell, and R of the group total equals that
    batched flux's R of the total."""
    prob = build_problem(name)
    d = prob.deck
    B = 7
    edges = edge_sets(d.initial_energy)["one"]
    grouped = _stepped(prob, B, edges)
    plain = _stepped(prob, B, None, flux=True)
    got = grouped.group_flux_batches_to_host().reshape(B, -1)
    want = plain.flux_batches_to_host().reshape(B, -1)
    assert np.count_nonzero(want) > 0
    assert tally_close(got.ravel(), want.ravel())
    _, groups, total = grouped.group_flux_relative_error()
    _, want_total = plain.flux_relative_error()
    assert abs(groups[0] - want_total) <= 1e-9 * want_total, (groups[0], want_total)
    assert abs(total - want_total) <= 1e-9 * want_total, (total, want_total)
    grouped.free()
    plain.free()


def test_stream_batches_gain_their_share_in_the_group_of_e0(gpu_lib, port):
    """5: on stream every batch's group of E0 gains n_b v(E0) dt / N per timestep (1e-12), and
    every other group of every batch stays exactly 0."""
    prob = build_problem("stream_small")
    d = prob.deck
    B = 7
    edges = np.geomspace(1.0e-3, 1.0e8, 12)
    G = edges.size - 1
    g0 = int(np.searchsorted(edges, d.initial_energy, side="right") - 1)
    want_sum, _ = stream_expectations(port, prob)
    sim = _sim(prob, B, edges)
    sim.inject()
    nb = np.array([shard_range(d.nparticles, b, B)[1] for b in range(B)], dtype=np.float64)
    before = np.zeros(B)
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        assert r.collisions == 0 and r.processed == d.nparticles
        S = sim.group_flux_batches_to_host().reshape(B, G, -1)
        assert not np.any(np.delete(S, g0, axis=1)), tt
        now = S[:, g0].sum(axis=1)
        want = nb * want_sum / d.nparticles
        assert np.all(np.abs((now - before) - want) <= 1e-12 * want), (tt, now - before, want)
        before = now
    sim.free()


def test_every_flush_path(gpu_lib):
    """6: the attached array is untouched until something looks at it; then nb200_memcpy_d2h (of
    the whole array, and of a range inside the last group's slice only), copy_buffer(RECV),
    nb200_tally_sync (NULL and the array), nb200_bank_free and a detach through each of the
    four attach calls each bring it to the unbatched group flux."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    d = prob.deck
    n = d.nx * d.ny
    edges = edge_sets(d.initial_energy)["log8"]
    G = edges.size - 1
    ref = _run(prob, edges=edges)
    want, want_tally = ref["gflux"].ravel(), ref["tally"]
    assert np.count_nonzero(want[(G - 1) * n + n // 3:(G - 1) * n + 2 * n // 3]) > 0

    def by_memcpy(sim):
        return sim.flux.download()

    def by_memcpy_inside_the_last_group(sim):
        lo, hi = (G - 1) * n + n // 3, (G - 1) * n + 2 * n // 3
        part = np.zeros(hi - lo)
        assert lib.nb200_memcpy_d2h(part.ctypes.data, sim.flux.ptr + 8 * lo, 8 * part.size) == 0
        assert tally_close(part, want[lo:hi])
        return _peek(lib, sim.flux)

    def by_copy_buffer(sim):
        host = np.zeros(G * n)
        src, dst = C.c_void_p(sim.flux.ptr), C.c_void_p(host.ctypes.data)
        lib.copy_buffer(C.c_size_t(host.size), C.byref(src), C.byref(dst), C.c_int(0))
        return host

    def by_tally_sync_null(sim):
        assert lib.nb200_tally_sync(None) == 0
        return _peek(lib, sim.flux)

    def by_tally_sync_other(sim):  # the energy tally's sync leaves the group flux alone
        assert lib.nb200_tally_sync(sim.tally.ptr) == 0
        assert not np.any(_peek(lib, sim.flux))
        assert lib.nb200_tally_sync(sim.flux.ptr) == 0
        return _peek(lib, sim.flux)

    def by_bank_free(sim):
        assert lib.nb200_bank_free(sim.bank) == 0
        sim.bank = None
        return _peek(lib, sim.flux)

    def detach(call):
        def by_detach(sim):
            assert call(sim.bank) == 0
            return _peek(lib, sim.flux)
        by_detach.__name__ = f"by_detach_{call.__name__}"
        return by_detach

    def batched_group(bank):
        return lib.nb200_bank_set_batched_group_flux_tally(bank, None, 0, None, 0)

    def group(bank):
        return lib.nb200_bank_set_group_flux_tally(bank, None, 0, None, 0)

    def batched(bank):
        return lib.nb200_bank_set_batched_flux_tally(bank, None, 0)

    def plain(bank):
        return lib.nb200_bank_set_flux_tally(bank, None, 0)

    for flush in (by_memcpy, by_memcpy_inside_the_last_group, by_copy_buffer, by_tally_sync_null,
                  by_tally_sync_other, by_bank_free, detach(batched_group), detach(group),
                  detach(batched), detach(plain)):
        sim = _stepped(prob, 7, edges)
        assert not np.any(_peek(lib, sim.flux)), ("deposits reached the array unflushed", flush)
        assert _groups_close(flush(sim), want), flush.__name__
        assert tally_close(sim.tally_to_host(), want_tally), flush.__name__
        sim.free()


def test_memset_flushes_then_zeroes(gpu_lib):
    """6: after nb200_memset_d of the group flux array, later flushes add only the later
    timesteps; the batches still hold every timestep."""
    prob = build_problem("mixed_small")
    d = prob.deck
    edges = edge_sets(d.initial_energy)["log8"]
    k = 2
    got = {}
    for B in (0, 7):
        sim = _sim(prob, B, edges)
        sim.inject()
        for tt in range(1, d.iterations + 1):
            sim.step(tt)
            if tt == k:
                sim.flux.zero()
                if B:
                    assert not np.any(_peek(gpu_lib, sim.flux))
        got[B] = sim.group_flux_to_host().ravel()
        if B:
            got["batches"] = sim.group_flux_batches_to_host().sum(axis=0).ravel()
        sim.free()
    full = _run(prob, edges=edges)["gflux"].ravel()
    assert np.count_nonzero(got[0]) > 0
    # A flush adds S - F per cell, where S and F both have the size of the whole run's flux in
    # the cell: where the timesteps after the memset add little to a group of a cell (the group
    # of e0 early in a deck), the result keeps the absolute rounding of the whole run's value.
    a, b = got[7], got[0]
    err = np.abs(a - b) - TALLY_RTOL * np.maximum(np.abs(a), np.abs(b))
    assert np.all(err <= 1e-14 * np.abs(full) + np.finfo(np.float64).tiny), np.max(err / full)
    assert _groups_close(got["batches"], full)


def _reference_per_step(port, prob, edges):
    """The group flux each timestep adds, (G * ncells) per timestep, from the port's bank."""
    d = prob.deck
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    out = []
    for tt in range(1, d.iterations + 1):
        gflux = np.zeros((edges.size - 1) * d.nx * d.ny)
        group_flux_reference().step(prob, bank, tt, tally, gflux=gflux, edges=edges)
        out.append(gflux)
    return out


def test_replacement_by_each_other_attach_call(gpu_lib, port):
    """6: on a batched bank, nb200_bank_set_batched_flux_tally and the batched group call itself
    replace a batched group flux, and the batched group call replaces a batched flux: the old
    array receives the timesteps before the switch and then stays bitwise frozen, the new one
    receives exactly the later timesteps, histories are unchanged. The two unbatched calls refuse
    the batched bank and leave its attachment as it was."""
    lib = gpu_lib
    prob = build_problem("csp_small", iterations=4)
    d = prob.deck
    n = d.nx * d.ny
    edges = edge_sets(d.initial_energy)["log8"]
    G = edges.size - 1
    e = np.ascontiguousarray(edges)
    base = _run(prob)
    per_step = _reference_per_step(port, prob, edges)
    early, later = per_step[0] + per_step[1], per_step[2] + per_step[3]

    def plain_of(gflux):
        return gflux.reshape(G, -1).sum(axis=0)

    cases = {  # old kind, new array size, attach of the new array, what the new array receives
        "batched": (edges, n, lambda b, a: lib.nb200_bank_set_batched_flux_tally(b, a.ptr, n),
                    plain_of(later)),
        "batched_group": (edges, G * n, lambda b, a: lib.nb200_bank_set_batched_group_flux_tally(
            b, a.ptr, n, e.ctypes.data, G), later),
        "batched_group_over_batched": (None, G * n,
                                       lambda b, a: lib.nb200_bank_set_batched_group_flux_tally(
                                           b, a.ptr, n, e.ctypes.data, G), later),
    }
    for key, (old_edges, size, attach, want_new) in cases.items():
        sim = _sim(prob, 7, old_edges, flux=old_edges is None)
        sim.inject()
        sim.step(1)
        sim.step(2)
        new = DeviceArray(size)
        assert attach(sim.bank, new) == 0, key
        frozen = _peek(lib, sim.flux)
        want_old = early if old_edges is not None else plain_of(early)
        assert _groups_close(frozen, want_old), key
        for tt in (3, 4):
            sim.step(tt)
            assert sum(sim.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
        assert lib.nb200_tally_sync(None) == 0
        assert np.array_equal(_peek(lib, sim.flux).view(np.uint64), frozen.view(np.uint64)), key
        assert _groups_close(new.download(), want_new), key
        sim.free()
        new.free()

    sim = _sim(prob, 7, edges)
    sim.inject()
    sim.step(1)
    other = DeviceArray(G * n)
    assert lib.nb200_bank_set_flux_tally(sim.bank, other.ptr, n) == -3
    assert b"tally_batches" in lib.nb200_last_error()
    assert lib.nb200_bank_set_group_flux_tally(sim.bank, other.ptr, n, e.ctypes.data, G) == -3
    assert b"tally_batches" in lib.nb200_last_error()
    for tt in range(2, d.iterations + 1):
        sim.step(tt)
    assert _groups_close(sim.group_flux_to_host(), early + later)
    assert not np.any(other.download())
    sim.free()
    other.free()


def test_deallocated_array_is_detached(gpu_lib):
    """6: after deallocate_data of the attached array, a fresh array of the same size (often at
    the same address) stays zero through a timestep and every flush, and the read calls refuse."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    edges = edge_sets(prob.deck.initial_energy)["log8"]
    sim = _sim(prob, 7, edges)
    sim.inject()
    sim.step(1)
    lib.deallocate_data(sim.flux.ptr)
    sim.flux.ptr = None
    fresh = DeviceArray(sim.flux.n)
    assert lib.nb200_tally_sync(None) == 0
    sim.step(2)
    assert lib.nb200_tally_sync(None) == 0
    assert not np.any(fresh.download())
    assert lib.nb200_bank_group_flux_relerr(sim.bank, None, None, None) == -3
    assert b"batched group flux" in lib.nb200_last_error()
    fresh.free()
    sim.flux = None
    sim.free()


GUARD = 1024  # doubles of sentinel on either side of an array


def _guarded(size, sentinel):
    buf = DeviceArray(size + 2 * GUARD)
    host = np.zeros(size + 2 * GUARD)
    host[:GUARD] = host[-GUARD:] = sentinel
    buf.upload(host)
    return buf, host


def _guards_intact(got, host):
    return (np.array_equal(got[:GUARD].view(np.uint64), host[:GUARD].view(np.uint64)) and
            np.array_equal(got[-GUARD:].view(np.uint64), host[-GUARD:].view(np.uint64)))


def test_nothing_outside_the_arrays_is_written(gpu_lib, port):
    """7: the attached array, the export buffer and the relative-error buffer sit inside larger
    allocations whose guard cells hold a sentinel: after the deck, for narrow groups and for
    edges leaving energies out, the guards are untouched and the insides are right."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    d = prob.deck
    n = d.nx * d.ny
    B = 7
    sentinel = np.float64(-1.2345e-300)
    for key in ("narrow32", "gaps"):
        edges = edge_sets(d.initial_energy)[key]
        G = edges.size - 1
        want = sum(_reference_per_step(port, prob, edges))
        buf, host = _guarded(G * n, sentinel)
        out, out_host = _guarded(B * G * n, sentinel)
        rel, rel_host = _guarded(G * n, sentinel)
        sim = Simulation(prob, tally_batches=B)
        sim.inject()
        assert lib.nb200_bank_set_batched_group_flux_tally(sim.bank, buf.ptr + 8 * GUARD, n,
                                                           edges.ctypes.data, G) == 0
        sim.run_pipelined()
        assert lib.nb200_bank_group_flux_batches(sim.bank, out.ptr + 8 * GUARD, n, G) == B
        assert lib.nb200_bank_group_flux_relerr(sim.bank, rel.ptr + 8 * GUARD, None, None) == 0
        got, got_out, got_rel = buf.download(), out.download(), rel.download()
        for g, h in ((got, host), (got_out, out_host), (got_rel, rel_host)):
            assert _guards_intact(g, h), key
        assert _groups_close(got[GUARD:-GUARD], want), key
        assert _groups_close(got_out[GUARD:-GUARD].reshape(B, -1).sum(axis=0), want), key
        assert np.all(np.isfinite(got_rel[GUARD:-GUARD])) and np.any(got_rel[GUARD:-GUARD])
        sim.free()
        for a in (buf, out, rel):
            a.free()


@pytest.mark.parametrize("graph", ["pipeline", "pipeline-calls"])
def test_four_kinds_of_bank_alternate(gpu_lib, port, graph):
    """8: a batched-group-flux bank, a batched-flux bank, a group-flux bank and a plain bank,
    stepped in turn on one device (the step graph switches kernels every timestep), with and
    without the step graph: all histories unchanged, every flux right."""
    _set_mode(gpu_lib, graph)
    try:
        prob = build_problem("csp_small", iterations=5)
        d = prob.deck
        edges = edge_sets(d.initial_energy)["narrow32"]
        want = sum(_reference_per_step(port, prob, edges))
        base = _run(prob)
        plain_flux = _run(prob, flux=True)["flux"]
        sims = [_sim(prob, 7, edges), _sim(prob, 7, None, flux=True), _sim(prob, 0, edges),
                _sim(prob)]
        for s in sims:
            s.inject()
        for tt in range(1, d.iterations + 1):
            for s in sims:
                r = s.step(tt)
                assert (r.facets, r.collisions) == base["counts"][tt - 1][:2]
                assert sum(s.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
        assert _groups_close(sims[0].group_flux_to_host(), want)
        assert _groups_close(sims[2].group_flux_to_host(), want)
        assert tally_close(sims[1].flux_to_host().ravel(), plain_flux)
        for s in sims:
            assert tally_close(s.tally_to_host(), base["tally"])
            s.free()
    finally:
        _restore(gpu_lib)


def test_refusals(gpu_lib):
    """9: every refusal returns its code and says why."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    n = prob.deck.nx * prob.deck.ny
    edges = np.array([1.0, 100.0, 1.0e4, 1.0e5])
    G = edges.size - 1

    def refused(rc, word, code=-3):
        assert rc == code, (rc, word)
        assert word.encode() in lib.nb200_last_error(), lib.nb200_last_error()

    def call(bank, ptr, ncells, e=edges, g=G):
        e = np.ascontiguousarray(e, dtype=np.float64)
        return lib.nb200_bank_set_batched_group_flux_tally(bank, ptr, ncells, e.ctypes.data, g)

    flux = DeviceArray(G * n)
    junk = (C.c_double * 4)()
    not_a_bank = C.cast(C.addressof(junk), _soa_p)
    refused(call(not_a_bank, flux.ptr, n), "not a bank handle")
    refused(lib.nb200_bank_group_flux_batches(not_a_bank, flux.ptr, n, G), "not a bank handle")
    refused(lib.nb200_bank_group_flux_relerr(not_a_bank, flux.ptr, None, None),
            "not a bank handle")

    plain = Simulation(prob)
    plain.inject()
    refused(call(plain.bank, flux.ptr, n), "no tally_batches")
    refused(lib.nb200_bank_group_flux_relerr(plain.bank, None, None, None), "batched group flux")
    plain.free()

    B = 16
    sim = Simulation(prob, tally_batches=B)
    sim.inject()
    refused(call(sim.bank, flux.ptr, n, g=0), "ngroups")
    refused(call(sim.bank, flux.ptr, n, e=[1.0, 1.0, 2.0, 3.0]), "strictly increasing")
    sim.step(1, defer=True)
    refused(call(sim.bank, flux.ptr, n), "enqueued", code=-4)
    sim.step_finish()
    lib.nb200_bank_set_option(sim.bank, b"defer_finish", 0)
    # the unbatched group call still refuses a batched bank, and names the batched one
    refused(lib.nb200_bank_set_group_flux_tally(sim.bank, flux.ptr, n, edges.ctypes.data, G),
            "tally_batches")
    assert b"nb200_bank_set_batched_group_flux_tally" in lib.nb200_last_error()
    host = np.zeros(G * n)
    refused(call(sim.bank, host.ctypes.data, n), "not device memory")
    refused(call(sim.bank, flux.ptr, 0), "cells")
    # B * G * ncells >= 2^31 with B * ncells < 2^31: a large ncells on a small allocation
    refused(call(sim.bank, flux.ptr, (1 << 31) // (B * G) + 1), "2^31")
    for name, value in ((b"pipeline", 0), (b"tally_prereduce", 1)):
        prev = lib.nb200_set_option(name, value)  # process-wide: the bank refuses it for itself
        try:
            refused(call(sim.bank, flux.ptr, n), "pipeline=1 and tally_prereduce=0")
        finally:
            lib.nb200_set_option(name, prev)
    assert call(sim.bank, flux.ptr, n) == 0
    refused(lib.nb200_bank_group_flux_batches(sim.bank, flux.ptr, n, G), "no timestep")
    refused(lib.nb200_bank_group_flux_relerr(sim.bank, None, None, None), "no timestep")
    assert lib.nb200_bank_set_option(sim.bank, b"pipeline", 0) == NB200_BAD_OPTION
    assert lib.nb200_bank_set_option(sim.bank, b"tally_prereduce", 1) == NB200_BAD_OPTION
    sim.step(2)
    out = DeviceArray(B * G * n)
    refused(lib.nb200_bank_group_flux_batches(sim.bank, out.ptr, n - 1, G), "cells")
    refused(lib.nb200_bank_group_flux_batches(sim.bank, out.ptr, n, G + 1), "groups")
    refused(lib.nb200_bank_group_flux_batches(sim.bank, None, n, G), "cells")
    assert lib.nb200_bank_group_flux_batches(sim.bank, out.ptr, n, G) == B
    # the batched flux's read calls refuse a group attachment and name the group calls
    for rc in (lib.nb200_bank_flux_batches(sim.bank, out.ptr, n),
               lib.nb200_bank_flux_relerr(sim.bank, None, None)):
        refused(rc, "group flux")
        assert b"nb200_bank_group_flux_batches" in lib.nb200_last_error()
        assert b"nb200_bank_group_flux_relerr" in lib.nb200_last_error()
    groups = np.zeros(G)
    total = C.c_double(-1.0)
    assert lib.nb200_bank_group_flux_relerr(sim.bank, None, groups.ctypes.data,
                                            C.byref(total)) == 0
    assert np.all(np.isfinite(groups)) and np.isfinite(total.value) and total.value >= 0.0
    sim.free()
    out.free()

    blob = (C.c_char * 256)()
    assert lib.nb200_mp_init(2, 0, n, blob) == 0
    try:
        grouped = Simulation(prob)
        grouped.inject()
        refused(call(grouped.bank, flux.ptr, n), "multi-process group")
        grouped.free()
    finally:
        lib.nb200_mp_finalize()

    if lib.nb200_device_count() >= 2:
        import torch
        with torch.cuda.device(1):
            other = torch.zeros(G * n, dtype=torch.float64, device="cuda:1")
        sim = Simulation(prob, tally_batches=4)
        sim.inject()
        refused(call(sim.bank, other.data_ptr(), n), "not device memory")
        sim.free()
        sharded = Simulation(prob, ngpus=2)
        sharded.inject()
        refused(call(sharded.bank, flux.ptr, n), "several GPUs")
        sharded.free()
    flux.free()


def test_full_size_csp_16_batches_8_groups(gpu_lib):
    """10: csp at full size, B = 16, G = 8 log groups covering every energy (B * G * ncells =
    2.05e9 < 2^31; a slab of about 17 GB): counts and energy tally total of the reference run,
    the flushed group flux summed over the groups equal to a plain-flux run's flux (1e-10 per
    cell), finite R per group."""
    from test_gpu_full_decks import _golden_full
    g = _golden_full()["csp"]
    prob = build_problem("csp")
    d = prob.deck
    edges = np.geomspace(1.0e-3, 2.0 * d.initial_energy, 9)
    plain = Simulation(prob, per_particle_counters=False, flux_tally=True)
    plain.inject()
    plain.run_pipelined()
    want = plain.flux_to_host().ravel()
    plain.free()
    sim = _sim(prob, 16, edges, per_particle_counters=False)
    sim.inject()
    got = [[r.facets, r.collisions] for r in sim.run_pipelined()]
    assert got == g["counts"]
    tally = sim.tally_to_host()
    assert abs(float(tally.sum()) - g["tally_sum"]) <= 1e-10 * g["tally_sum"]
    gflux = sim.group_flux_to_host().reshape(8, -1)
    _, groups, total = sim.group_flux_relative_error()
    sim.free()
    print(f"csp full size, 16 batches, 8 groups: R per group "
          f"{np.array2string(groups, precision=3)}, R of the total {total:.3e}")
    assert np.count_nonzero(want) > 0
    assert _groups_close(gflux.sum(axis=0), want)
    assert np.all(np.isfinite(groups)) and np.count_nonzero(groups) >= 4
    assert 0.0 < total < 1e-2


def test_group_relative_error_shrinks_like_one_over_sqrt_n(gpu_lib):
    """10: R of the most populated group's total falls as 1/sqrt(N): 4x the particles halves it.
    With B = 64 the ratio of two independent estimates spreads by about 13 %; [1.3, 3.0] is more
    than five of those spreads on either side of 2."""
    edges = edge_sets(build_problem("csp_small").deck.initial_energy)["log8"]
    rs = []
    for n in (16_000, 64_000):
        sim = _stepped(build_problem("csp_small", nparticles=n), 64, edges,
                       per_particle_counters=False)
        top = int(np.argmax(sim.group_flux_to_host().sum(axis=(1, 2))))
        rs.append(sim.group_flux_relative_error()[1][top])
        sim.free()
    ratio = rs[0] / rs[1]
    print(f"group flux, most populated group: R(16k) = {rs[0]:.3e}, R(64k) = {rs[1]:.3e}, "
          f"ratio {ratio:.2f}")
    assert 1.3 <= ratio <= 3.0, rs
