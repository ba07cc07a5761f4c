"""Flux batches on the GPU (nb200_bank_set_batched_flux_tally): batching the flux moves deposits,
never histories. Counts, per-particle counters and every bank field are bit-identical to the
unbatched run; after a flush the energy tally and the flux equal the unbatched flux run's to
1e-10 per cell; every flux batch equals the flux reference run on its particle range; the
relative errors follow the estimator's formula; every flush path, attachment change and refusal
behaves as the header says."""
import ctypes as C

import numpy as np
import pytest

from conftest import SMALL_DECKS
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.host import NB200_BAD_OPTION, DeviceArray, Simulation, _soa_p
from flux_reference import flux_reference
from test_flux_tally_cpu import stream_expectations
from test_gpu_parity import DEFAULTS, MODES, tally_close
from test_gpu_tally_batches import _rel_close, _relerr_numpy
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


def _run(prob, batches, flux, pipelined=False):
    """Per-timestep counts, bank after every timestep (step by step) or at the end (pipelined),
    per-particle counters, and the flushed energy tally and flux."""
    sim = Simulation(prob, tally_batches=batches, flux_tally=flux)
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
    if flux:
        out["flux"] = sim.flux_to_host().ravel()
    if flux and batches:
        out["flux_batches"] = sim.flux_batches_to_host()
    sim.free()
    return out


def _same_histories(got, want, what):
    assert got["counts"] == want["counts"], what
    for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
        diff = a.bit_equal(b)
        assert sum(diff.values()) == 0, (what, tt, diff)
    assert np.array_equal(got["counters"], want["counters"]), what


@pytest.mark.parametrize("name", SMALL_DECKS + list(VARIANTS))
def test_histories_unchanged(gpu_lib, kernel_mode, name):
    """1: bit-identical histories against the unbatched run without flux; energy tally, flux and
    the sum of the exported flux batches equal to the unbatched flux run's to 1e-10 per cell."""
    prob = _problem(name)
    d = prob.deck
    for pipelined in (False, True):
        base = _run(prob, 0, False, pipelined)
        want = _run(prob, 0, True, pipelined)
        assert np.count_nonzero(want["flux"]) > 0
        for B in BATCHES:
            what = (B, pipelined)
            got = _run(prob, B, True, pipelined)
            _same_histories(got, base, what)
            assert tally_close(got["tally"], want["tally"]), what
            assert tally_close(got["flux"], want["flux"]), what
            assert got["flux_batches"].shape == (B, d.ny, d.nx)
            assert tally_close(got["flux_batches"].sum(axis=0).ravel(), want["flux"]), what


@pytest.mark.parametrize("name", ["csp_small", "split_small", "mixed_small", "absorb_own_grid"])
def test_every_batch_matches_the_reference(gpu_lib, port, name):
    """2: flux batch b after every timestep equals the flux reference run on particles
    [first_b, first_b + n_b) with the whole run's ntotal, to 1e-10 per cell; the energy batches
    equal the same runs' energy tallies to 1e-10 per cell (the flux reference's energy tally is
    the oracle port's bit for bit, tests/test_flux_tally_cpu.py)."""
    prob = _problem(name)
    d = prob.deck
    B = 7
    sim = Simulation(prob, tally_batches=B, flux_tally=True)
    sim.inject()
    ranges = [shard_range(d.nparticles, b, B) for b in range(B)]
    banks = [port.inject(prob, pid0=f, count=n) for f, n in ranges]
    tallies = [np.zeros(d.nx * d.ny) for _ in range(B)]
    fluxes = [np.zeros(d.nx * d.ny) for _ in range(B)]
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        facets = 0
        for b, (f, n) in enumerate(ranges):
            facets += flux_reference().step(prob, banks[b], tt, tallies[b], pid0=f,
                                            ntotal=d.nparticles, flux=fluxes[b])[0]
        assert r.facets == facets, tt
        got_flux = sim.flux_batches_to_host().reshape(B, -1)
        got_tally = sim.tally_batches_to_host().reshape(B, -1)
        for b in range(B):
            assert np.count_nonzero(fluxes[b]) > 0, (tt, b)
            assert tally_close(got_flux[b], fluxes[b]), (tt, b)
            assert tally_close(got_tally[b], tallies[b]), (tt, b)
    sim.free()


def _stepped(prob, B, steps=None, **kw):
    sim = Simulation(prob, tally_batches=B, flux_tally=True, **kw)
    sim.inject()
    for tt in range(1, (steps or prob.deck.iterations) + 1):
        sim.step(tt)
    return sim


@pytest.mark.parametrize("name", ["csp_small", "split_small"])
def test_statistics_match_the_formula(gpu_lib, name):
    """3: device R per cell and of the flux total equals the formula on the exported flux
    batches (1e-12); R is 0 where the mean is 0."""
    prob = build_problem(name)
    d = prob.deck
    B = 16
    sim = _stepped(prob, B)
    S = sim.flux_batches_to_host().reshape(B, -1)
    cell, total = sim.flux_relative_error()
    want = _relerr_numpy(list(S), d.nparticles)
    assert cell.shape == (d.ny, d.nx)
    assert _rel_close(cell.ravel(), want, 1e-12)
    assert np.all(cell.ravel()[S.sum(axis=0) == 0.0] == 0.0)
    assert np.count_nonzero(cell) > 0
    want_total = _relerr_numpy([np.array([S[b].sum()]) for b in range(B)], d.nparticles)[0]
    assert abs(total - want_total) <= 1e-12 * abs(want_total)
    assert 0.0 < total < 1.0
    # the energy statistics are still those of the energy batches
    E = sim.tally_batches_to_host().reshape(B, -1)
    assert _rel_close(sim.tally_relative_error()[0].ravel(), _relerr_numpy(list(E), d.nparticles),
                      1e-12)
    sim.free()


def test_stream_batches_gain_their_share_of_the_distance(gpu_lib, port):
    """4: on stream every flux batch gains n_b v(E0) dt / N per timestep (1e-12), independent of
    the reference; so every batch estimate is the same and R of the flux total is rounding."""
    prob = build_problem("stream_small")
    d = prob.deck
    B = 7
    want_sum, _ = stream_expectations(port, prob)
    sim = Simulation(prob, tally_batches=B, flux_tally=True)
    sim.inject()
    nb = np.array([shard_range(d.nparticles, b, B)[1] for b in range(B)], dtype=np.float64)
    before = np.zeros(B)
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        assert r.collisions == 0 and r.processed == d.nparticles
        now = sim.flux_batches_to_host().reshape(B, -1).sum(axis=1)
        gain = now - before
        want = nb * want_sum / d.nparticles
        assert np.all(np.abs(gain - want) <= 1e-12 * want), (tt, gain, want)
        before = now
    _, total = sim.flux_relative_error()
    print(f"stream_small, {B} batches: relative error of the flux total {total:.3e}")
    assert 0.0 <= total < 1e-12
    sim.free()


def test_every_flush_path(gpu_lib):
    """5: the caller's flux array is untouched until something looks at it; then
    nb200_memcpy_d2h, copy_buffer(RECV), nb200_tally_sync (NULL and the array), nb200_bank_free
    and a detach through either attach function each bring it to the unbatched flux."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    d = prob.deck
    ref = Simulation(prob, flux_tally=True)
    ref.inject()
    ref.run()
    want = ref.flux_to_host().ravel()
    want_tally = ref.tally_to_host()
    ref.free()
    assert np.count_nonzero(want) > 0

    def by_memcpy(sim):
        return sim.flux.download()

    def by_copy_buffer(sim):
        host = np.zeros(d.nx * d.ny)
        src, dst = C.c_void_p(sim.flux.ptr), C.c_void_p(host.ctypes.data)
        lib.copy_buffer(C.c_size_t(host.size), C.byref(src), C.byref(dst), C.c_int(0))
        return host

    def by_tally_sync_null(sim):
        assert lib.nb200_tally_sync(None) == 0
        return _peek(lib, sim.flux)

    def by_tally_sync_flux(sim):
        assert lib.nb200_tally_sync(sim.flux.ptr) == 0
        return _peek(lib, sim.flux)

    def by_tally_sync_other(sim):  # the energy tally's sync leaves the flux alone
        assert lib.nb200_tally_sync(sim.tally.ptr) == 0
        assert not np.any(_peek(lib, sim.flux))
        return by_tally_sync_flux(sim)

    def by_bank_free(sim):
        assert lib.nb200_bank_free(sim.bank) == 0
        sim.bank = None
        return _peek(lib, sim.flux)

    def by_batched_detach(sim):
        assert lib.nb200_bank_set_batched_flux_tally(sim.bank, None, 0) == 0
        return _peek(lib, sim.flux)

    def by_plain_detach(sim):
        assert lib.nb200_bank_set_flux_tally(sim.bank, None, 0) == 0
        return _peek(lib, sim.flux)

    for flush in (by_memcpy, by_copy_buffer, by_tally_sync_null, by_tally_sync_flux,
                  by_tally_sync_other, by_bank_free, by_batched_detach, by_plain_detach):
        sim = _stepped(prob, 7)
        assert not np.any(_peek(lib, sim.flux)), ("deposits reached the flux unflushed", flush)
        assert tally_close(flush(sim), want), flush.__name__
        assert tally_close(sim.tally_to_host(), want_tally), flush.__name__
        sim.free()


def test_memset_flushes_then_zeroes(gpu_lib):
    """5: after nb200_memset_d of the flux array, later flushes add only the later timesteps."""
    prob = build_problem("mixed_small")
    d = prob.deck
    k = 2
    got, want = [], []
    for B in (0, 7):
        sim = Simulation(prob, tally_batches=B, flux_tally=True)
        sim.inject()
        for tt in range(1, d.iterations + 1):
            sim.step(tt)
            if tt == k:
                sim.flux.zero()
                if B:
                    assert not np.any(_peek(gpu_lib, sim.flux))
        (got if B else want).append(sim.flux_to_host().ravel())
        if B:
            got.append(sim.flux_batches_to_host().sum(axis=0).ravel())
        sim.free()
    assert np.count_nonzero(want[0]) > 0
    assert tally_close(got[0], want[0])
    # the batches themselves still hold every timestep: they are what the memset did not zero
    full = _run(prob, 0, True)["flux"]
    assert tally_close(got[1], full)


def _reference_fluxes(prob, port):
    d = prob.deck
    pbank = port.inject(prob)
    ptally = np.zeros(d.nx * d.ny)
    pflux = [np.zeros(d.nx * d.ny) for _ in range(d.iterations)]
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, pbank, tt, ptally, flux=pflux[tt - 1])
    return pflux


def test_detach_and_reattach(gpu_lib, port):
    """6: after a detach the old array stays bitwise frozen; a second array attached later
    receives exactly the later timesteps and its batches start at zero; histories unchanged."""
    lib = gpu_lib
    prob = build_problem("csp_small", iterations=5)
    d = prob.deck
    base = _run(prob, 0, False)
    pflux = _reference_fluxes(prob, port)
    B = 7
    sim = Simulation(prob, tally_batches=B, flux_tally=True)
    sim.inject()
    sim.step(1)
    assert lib.nb200_bank_set_batched_flux_tally(sim.bank, None, 0) == 0
    frozen = _peek(lib, sim.flux)
    assert tally_close(frozen, pflux[0])
    assert lib.nb200_bank_flux_batches(sim.bank, None, 0) == -3
    assert b"not a bank handle with a batched flux" in lib.nb200_last_error()
    second = DeviceArray(d.nx * d.ny)
    for tt in range(2, d.iterations + 1):
        if tt == 4:
            assert lib.nb200_bank_set_batched_flux_tally(sim.bank, second.ptr, second.n) == 0
            assert lib.nb200_bank_flux_relerr(sim.bank, None, None) == -3
            assert b"no timestep" in lib.nb200_last_error()
        sim.step(tt)
        assert np.array_equal(sim.flux_to_host().ravel().view(np.uint64),
                              frozen.view(np.uint64)), tt
        assert sum(sim.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
    out = DeviceArray(B * d.nx * d.ny)
    assert lib.nb200_bank_flux_batches(sim.bank, out.ptr, d.nx * d.ny) == B
    assert tally_close(out.download().reshape(B, -1).sum(axis=0), pflux[3] + pflux[4])
    out.free()
    assert tally_close(second.download(), pflux[3] + pflux[4])
    assert tally_close(sim.tally_to_host(), base["tally"])
    sim.free()
    second.free()


def test_deallocated_array_is_detached(gpu_lib):
    """6: after deallocate_data of the attached array, a fresh array of the same size (often at
    the same address) stays zero through a timestep, and nothing is flushed into it."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    sim = Simulation(prob, tally_batches=7, flux_tally=True)
    sim.inject()
    sim.step(1)
    lib.deallocate_data(sim.flux.ptr)
    sim.flux.ptr = None
    fresh = DeviceArray(sim.flux.n)
    assert lib.nb200_tally_sync(None) == 0
    sim.step(2)
    assert lib.nb200_tally_sync(None) == 0
    assert not np.any(fresh.download())
    assert lib.nb200_bank_flux_batches(sim.bank, None, 0) == -3
    fresh.free()
    sim.flux = None
    sim.free()


@pytest.mark.parametrize("graph", ["pipeline", "pipeline-calls"])
def test_batched_flux_and_plain_banks_alternate(gpu_lib, port, graph):
    """6: a batched-flux bank and a plain bank stepped alternately on one GPU are both right,
    with and without the step graph."""
    _set_mode(gpu_lib, graph)
    try:
        prob = build_problem("csp_small", iterations=5)
        d = prob.deck
        base = _run(prob, 0, False)
        pflux = _reference_fluxes(prob, port)
        a = Simulation(prob, tally_batches=7, flux_tally=True)
        b = Simulation(prob)
        a.inject()
        b.inject()
        for tt in range(1, d.iterations + 1):
            ra, rb = a.step(tt), b.step(tt)
            assert (ra.facets, ra.collisions) == (rb.facets, rb.collisions) == \
                base["counts"][tt - 1][:2]
            for s in (a, b):
                assert sum(s.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
        assert tally_close(a.flux_to_host().ravel(), sum(pflux))
        assert tally_close(a.tally_to_host(), base["tally"])
        assert tally_close(b.tally_to_host(), base["tally"])
        a.free()
        b.free()
    finally:
        _restore(gpu_lib)


def test_refusals(gpu_lib):
    """7: every refusal returns its code and says why."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    n = prob.deck.nx * prob.deck.ny

    def refused(rc, word, code=-3):
        assert rc == code, (rc, word)
        assert word.encode() in lib.nb200_last_error(), lib.nb200_last_error()

    flux = DeviceArray(n)
    junk = (C.c_double * 4)()
    not_a_bank = C.cast(C.addressof(junk), _soa_p)
    refused(lib.nb200_bank_set_batched_flux_tally(not_a_bank, flux.ptr, n), "not a bank handle")
    refused(lib.nb200_bank_flux_batches(not_a_bank, flux.ptr, n), "not a bank handle")
    refused(lib.nb200_bank_flux_relerr(not_a_bank, flux.ptr, None), "not a bank handle")

    plain = Simulation(prob)
    plain.inject()
    refused(lib.nb200_bank_set_batched_flux_tally(plain.bank, flux.ptr, n), "no tally_batches")
    refused(lib.nb200_bank_flux_relerr(plain.bank, None, None), "batched flux")
    plain.free()

    B = 16
    sim = Simulation(prob, tally_batches=B)
    sim.inject()
    sim.step(1, defer=True)
    refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, flux.ptr, n), "enqueued", code=-4)
    sim.step_finish()
    lib.nb200_bank_set_option(sim.bank, b"defer_finish", 0)
    # the plain attach still refuses a batched bank, and names the batched one
    refused(lib.nb200_bank_set_flux_tally(sim.bank, flux.ptr, n), "tally_batches")
    assert b"nb200_bank_set_batched_flux_tally" in lib.nb200_last_error()
    host = np.zeros(n)
    refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, host.ctypes.data, n),
            "not device memory")
    refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, flux.ptr, 0), "cells")
    refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, flux.ptr, (1 << 31) // B), "2^31")
    for name, value in ((b"pipeline", 0), (b"tally_prereduce", 1)):
        prev = lib.nb200_set_option(name, value)  # process-wide: the bank refuses it for itself
        try:
            refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, flux.ptr, n),
                    "pipeline=1 and tally_prereduce=0")
        finally:
            lib.nb200_set_option(name, prev)
    assert lib.nb200_bank_set_batched_flux_tally(sim.bank, flux.ptr, n) == 0
    refused(lib.nb200_bank_flux_batches(sim.bank, None, 0), "no timestep")
    assert lib.nb200_bank_set_option(sim.bank, b"pipeline", 0) == NB200_BAD_OPTION
    assert lib.nb200_bank_set_option(sim.bank, b"tally_prereduce", 1) == NB200_BAD_OPTION
    sim.step(2)
    refused(lib.nb200_bank_flux_batches(sim.bank, flux.ptr, n - 1), "cells")
    assert lib.nb200_bank_flux_relerr(sim.bank, None, None) == 0
    sim.free()

    if lib.nb200_device_count() >= 2:
        import torch
        with torch.cuda.device(1):
            other = torch.zeros(n, dtype=torch.float64, device="cuda:1")
        sim = Simulation(prob, tally_batches=4)
        sim.inject()
        refused(lib.nb200_bank_set_batched_flux_tally(sim.bank, other.data_ptr(), n),
                "not device memory")
        sim.free()
    flux.free()


def test_full_size_csp_with_16_batches(gpu_lib, port):
    """8: csp at full size, B = 16: counts and energy tally total of the reference run, the
    flux per cell against the flux reference (1e-10); R of the flux total is printed."""
    from test_gpu_full_decks import _golden_full
    g = _golden_full()["csp"]
    prob = build_problem("csp")
    d = prob.deck
    sim = Simulation(prob, per_particle_counters=False, tally_batches=16, flux_tally=True)
    sim.inject()
    got = [[r.facets, r.collisions] for r in sim.run_pipelined()]
    assert got == g["counts"]
    tally = sim.tally_to_host()
    assert abs(float(tally.sum()) - g["tally_sum"]) <= 1e-10 * g["tally_sum"]
    flux = sim.flux_to_host().ravel()
    _, total = sim.flux_relative_error()
    sim.free()
    print(f"csp full size, 16 batches: relative error of the flux total {total:.3e}")
    assert 0.0 < total < 1e-2
    bank = port.inject(prob)
    ptally, pflux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, bank, tt, ptally, flux=pflux)
    assert np.count_nonzero(pflux) > 0
    assert tally_close(flux, pflux)


def test_relative_error_shrinks_like_one_over_sqrt_n(gpu_lib):
    """8: R of the flux total falls as 1/sqrt(N): 4x the particles halves it. With B = 64 the
    ratio of two independent estimates spreads by about 13 %; [1.3, 3.0] is more than five of
    those spreads on either side of 2."""
    rs = []
    for n in (16_000, 64_000):
        sim = _stepped(build_problem("csp_small", nparticles=n), 64, per_particle_counters=False)
        rs.append(sim.flux_relative_error()[1])
        sim.free()
    ratio = rs[0] / rs[1]
    print(f"flux: R(16k) = {rs[0]:.3e}, R(64k) = {rs[1]:.3e}, ratio {ratio:.2f}")
    assert 1.3 <= ratio <= 3.0, rs
