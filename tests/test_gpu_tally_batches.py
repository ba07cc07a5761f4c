"""Option tally_batches on the GPU: batching moves deposits, never histories. Per-timestep
counts, per-particle counters and every bank field are bit-identical to the unbatched run; the
caller's tally after a flush equals the unbatched tally to 1e-10 per cell through every flush
path; every batch equals an independent oracle run of its particle range; the relative errors
follow the estimator's formula; and refusals come back as error codes."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import SMALL_DECKS
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.host import NB200_BAD_OPTION, DeviceArray, Simulation
from test_gpu_engine import _capture_stdout
from test_gpu_parity import DEFAULTS, MODES, tally_close
from variants import VARIANTS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BATCHES = (2, 7, 16)


def _problem(name):
    return VARIANTS[name]() if name in VARIANTS else build_problem(name)


@pytest.fixture(params=["pipeline", "pipeline-ieee-div"])
def kernel_mode(request, gpu_lib):
    for k, v in MODES[request.param].items():
        assert gpu_lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION
    yield request.param
    for k, v in DEFAULTS.items():
        gpu_lib.nb200_set_option(k.encode(), v)


def _run(prob, batches, pipelined=False):
    """Per-timestep counts, bank after every timestep (step by step) or at the end
    (pipelined), per-particle counters and the flushed tally."""
    sim = Simulation(prob, tally_batches=batches)
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
    if batches:
        out["batches"] = sim.tally_batches_to_host()
    sim.free()
    return out


@pytest.mark.parametrize("name", SMALL_DECKS + list(VARIANTS))
def test_histories_and_tally_unchanged(gpu_lib, kernel_mode, name):
    """1 and 2: bit-identical histories, tally after a flush (nb200_memcpy_d2h) and the sum of
    the exported batches equal to the unbatched tally to 1e-10 per cell."""
    prob = _problem(name)
    base = _run(prob, 0)
    base_pipe = _run(prob, 0, pipelined=True)
    for B in BATCHES:
        for pipelined in (False, True):
            got = _run(prob, B, pipelined)
            want = base_pipe if pipelined else base
            assert got["counts"] == want["counts"], (B, pipelined)
            for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
                diff = a.bit_equal(b)
                assert sum(diff.values()) == 0, (B, pipelined, tt, diff)
            assert np.array_equal(got["counters"], want["counters"]), (B, pipelined)
            assert tally_close(got["tally"], want["tally"]), (B, pipelined)
            assert got["batches"].shape == (B, prob.deck.ny, prob.deck.nx)
            assert tally_close(got["batches"].sum(axis=0).ravel(), want["tally"]), (B, pipelined)


def _stepped(prob, B, steps=None):
    sim = Simulation(prob, tally_batches=B)
    sim.inject()
    for tt in range(1, (steps or prob.deck.iterations) + 1):
        sim.step(tt)
    return sim


def _peek(lib, tally):
    """The device tally WITHOUT flushing: accumulated into a scratch buffer on the device."""
    scratch = DeviceArray(tally.n)
    assert lib.nb200_accumulate(scratch.ptr, tally.ptr, tally.n) == 0
    out = scratch.download()
    scratch.free()
    return out


def test_every_flush_path(gpu_lib, monkeypatch):
    """2: the caller's tally stays as it was until something looks at it; then validate
    (same printed lines), nb200_memcpy_d2h, copy_buffer(RECV), nb200_tally_sync and
    nb200_bank_free each bring it to the unbatched tally."""
    prob = build_problem("csp_small")
    d = prob.deck
    ref = Simulation(prob)
    ref.inject()
    ref.run()
    want = ref.tally_to_host()
    monkeypatch.chdir(ROOT)  # validate reads problems/neutral.tests from the run directory
    want_lines = _capture_stdout(lambda: ref.validate("problems/csp.params"))
    ref.free()
    assert "Final global_energy_tally" in want_lines and "Expected" in want_lines

    def check(flush):
        sim = _stepped(prob, 7)
        assert not np.any(_peek(gpu_lib, sim.tally)), "deposits reached the tally unflushed"
        got = flush(sim)
        assert tally_close(got, want), flush
        sim.free()

    def by_validate(sim):
        assert _capture_stdout(lambda: sim.validate("problems/csp.params")) == want_lines
        return _peek(gpu_lib, sim.tally)

    def by_copy_buffer(sim):
        host = np.zeros(d.nx * d.ny)
        src, dst = C.c_void_p(sim.tally.ptr), C.c_void_p(host.ctypes.data)
        gpu_lib.copy_buffer(C.c_size_t(host.size), C.byref(src), C.byref(dst), C.c_int(0))
        return host

    def by_tally_sync(sim):
        sim.tally_sync()
        return _peek(gpu_lib, sim.tally)

    def by_bank_free(sim):
        assert gpu_lib.nb200_bank_free(sim.bank) == 0
        sim.bank = None
        return _peek(gpu_lib, sim.tally)

    for flush in (by_validate, lambda sim: sim.tally.download(), by_copy_buffer, by_tally_sync,
                  by_bank_free):
        check(flush)


def test_batches_follow_the_tally_pointer(gpu_lib):
    """A timestep into another tally flushes into the old one and starts over."""
    prob = build_problem("mixed_small")
    ref = Simulation(prob)
    ref.inject()
    r1 = ref.step(1)
    t1 = ref.tally_to_host()
    other = DeviceArray(t1.size)
    ref.step(2, tally_ptr=other.ptr)
    t2 = other.download()
    ref.free()
    other.free()
    sim = Simulation(prob, tally_batches=4)
    sim.inject()
    assert sim.step(1).facets == r1.facets
    other = DeviceArray(t1.size)
    sim.step(2, tally_ptr=other.ptr)
    assert tally_close(_peek(gpu_lib, sim.tally), t1)  # flushed when the target changed
    assert tally_close(sim.tally_batches_to_host().sum(axis=0).ravel(), t2)
    assert tally_close(other.download(), t2)
    sim.free()
    other.free()


@pytest.mark.parametrize("name", ["csp_small", "split_small", "mixed_small", "absorb_own_grid"])
def test_every_batch_matches_the_oracle(gpu_lib, port, name):
    """3: batch b after every timestep equals the oracle port run on particles
    [first_b, first_b + n_b) with the whole run's ntotal, to 1e-10 per cell."""
    prob = _problem(name)
    d = prob.deck
    B = 7
    sim = Simulation(prob, tally_batches=B)
    sim.inject()
    ranges = [shard_range(d.nparticles, b, B) for b in range(B)]
    banks = [port.inject(prob, pid0=f, count=n) for f, n in ranges]
    tallies = [np.zeros(d.nx * d.ny) for _ in range(B)]
    for tt in range(1, d.iterations + 1):
        r = sim.step(tt)
        facets = 0
        for b, (f, n) in enumerate(ranges):
            facets += port.step(prob, banks[b], tt, tallies[b], pid0=f, ntotal=d.nparticles)[0]
        assert r.facets == facets, tt
        got = sim.tally_batches_to_host().reshape(B, -1)
        for b in range(B):
            assert tally_close(got[b], tallies[b]), (tt, b)
    sim.free()


def _relerr_numpy(batches, n):
    """The estimator in batch order: x_b = S_b N / n_b, m, s^2, R = sqrt(s^2 / B) / |m|."""
    B = len(batches)
    nb = [shard_range(n, b, B)[1] for b in range(B)]
    x = [batches[b] * n / nb[b] for b in range(B)]
    s = np.zeros_like(x[0])
    for b in range(B):
        s = s + x[b]
    m = s / B
    ss = np.zeros_like(m)
    for b in range(B):
        ss = ss + (x[b] - m) * (x[b] - m)
    var = ss / (B - 1)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(m == 0.0, 0.0, np.sqrt(var / B) / np.abs(m))
    return r


def _rel_close(a, b, rtol):
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b))))


@pytest.mark.parametrize("name", ["csp_small", "split_small"])
def test_statistics_match_the_formula(gpu_lib, name):
    """4: device R per cell and of the total equals the formula on the exported batches."""
    prob = build_problem(name)
    d = prob.deck
    B = 16
    sim = _stepped(prob, B)
    S = sim.tally_batches_to_host().reshape(B, -1)
    cell, total = sim.tally_relative_error()
    want = _relerr_numpy(list(S), d.nparticles)
    assert cell.shape == (d.ny, d.nx)
    assert _rel_close(cell.ravel(), want, 1e-12)
    assert np.all(cell.ravel()[S.sum(axis=0) == 0.0] == 0.0)
    assert np.count_nonzero(cell) > 0
    want_total = _relerr_numpy([np.array([S[b].sum()]) for b in range(B)], d.nparticles)[0]
    assert abs(total - want_total) <= 1e-12 * abs(want_total)
    assert 0.0 < total < 1.0
    sim.free()


def test_full_size_csp_with_16_batches(gpu_lib):
    """5: csp at full size, B = 16: the reference run's per-timestep counts, tally total, 64 x 64
    block sums and per-cell samples; R of the total is printed."""
    from recorded import tally_matches_sample
    from test_gpu_full_decks import _golden_full
    g = _golden_full()["csp"]
    prob = build_problem("csp")
    d = prob.deck
    sim = Simulation(prob, per_particle_counters=False, tally_batches=16)
    sim.inject()
    got = [[r.facets, r.collisions] for r in sim.run_pipelined()]
    assert got == g["counts"]
    tally = sim.tally_to_host()
    assert abs(float(tally.sum()) - g["tally_sum"]) <= 1e-10 * g["tally_sum"]
    blocks = 64
    by, bx = d.ny // blocks, d.nx // blocks
    img = tally.reshape(d.ny, d.nx)[:by * blocks, :bx * blocks] \
        .reshape(blocks, by, blocks, bx).sum(axis=(1, 3)).ravel()
    want = np.array(g["tally_block_sums"])
    assert np.all(np.abs(img - want) <= 1e-10 * np.maximum(np.abs(img), np.abs(want)))
    assert tally_matches_sample(tally, "csp", 1e-10)
    _, total = sim.tally_relative_error()
    print(f"csp full size, 16 batches: relative error of the tally total {total:.3e}")
    assert 0.0 < total < 1e-2
    sim.free()


def test_relative_error_shrinks_like_one_over_sqrt_n(gpu_lib):
    """6: R of the total falls as 1/sqrt(N), so 4x the particles halves it. R from B batches is
    itself an estimate: s^2 has B - 1 = 63 degrees of freedom, so s (and R) has a relative
    spread of about 1/sqrt(2 (B - 1)) = 9 %, and the ratio of two independent estimates about
    13 %. [1.3, 3.0] around the expected 2 is more than five of those spreads on either side."""
    rs = []
    for n in (16_000, 64_000):
        sim = _stepped(build_problem("csp_small", nparticles=n), 64)
        rs.append(sim.tally_relative_error()[1])
        sim.free()
    ratio = rs[0] / rs[1]
    print(f"R(16k) = {rs[0]:.3e}, R(64k) = {rs[1]:.3e}, ratio {ratio:.2f}")
    assert 1.3 <= ratio <= 3.0, rs


def _host_bank(n):
    prob = build_problem("csp_small")
    from oracle.oracle import OraclePort
    return prob, OraclePort().inject(prob, 0, n)


def test_refusals(gpu_lib):
    """7: each case returns an error code and says why; nothing terminates the process."""
    lib = gpu_lib
    _, host = _host_bank(50)
    st = host.as_struct()
    out = C.POINTER(type(st))()

    def create(pid_first=0, count=50):
        return lib.nb200_bank_create(C.byref(st), count, pid_first, C.byref(out))

    def refused(rc, word):
        assert rc != 0, word
        assert word.encode() in lib.nb200_last_error(), lib.nb200_last_error()

    assert lib.nb200_set_option(b"tally_batches", 4) != NB200_BAD_OPTION
    try:
        prev = lib.nb200_set_option(b"ngpus", 2)
        refused(create(), "several GPUs")
        lib.nb200_set_option(b"ngpus", prev)
        blob = (C.c_char * 256)()
        assert lib.nb200_mp_init(2, 0, 1024, blob) == 0
        refused(create(), "multi-process group")
        lib.nb200_mp_finalize()
        refused(create(pid_first=5, count=45), "starts at particle 5")
        refused(create(count=3), "exceeds the bank's 3 particles")
        for name, value in ((b"pipeline", 0), (b"tally_prereduce", 1)):
            prev = lib.nb200_set_option(name, value)
            refused(create(), name.decode())
            lib.nb200_set_option(name, prev)
        assert create() == 0
        bank = out
        assert lib.nb200_bank_set_option(bank, b"pipeline", 0) == NB200_BAD_OPTION
        assert b"tally_batches" in lib.nb200_last_error()
        assert lib.nb200_bank_set_option(bank, b"tally_prereduce", 1) == NB200_BAD_OPTION
        assert lib.nb200_bank_set_option(bank, b"tally_batches", 2) == NB200_BAD_OPTION
        assert lib.nb200_bank_set_option(bank, b"fast_div", 0) != NB200_BAD_OPTION
        _, more = _host_bank(2)
        refused(lib.nb200_bank_append(bank, C.byref(more.as_struct()), 2), "cannot grow")
        refused(lib.nb200_bank_tally_batches(bank, None, 0), "no timestep")
        lib.nb200_bank_free(bank)
    finally:
        lib.nb200_set_option(b"tally_batches", 0)
    assert create() == 0
    refused(lib.nb200_bank_tally_relerr(out, None, None), "not a bank handle created with")
    lib.nb200_bank_free(out)


TODAY_KEYS = {"deck", "nx", "ny", "device", "tally_total", "expected", "relative_error",
              "tolerance", "verdict", "steps"}
NEW_KEYS = {"tally_batches", "tally_total_relative_error"}


def test_results_json(gpu_lib, tmp_path, monkeypatch):
    """8: validate's JSON has the two new keys for a batched bank, exactly today's otherwise."""
    path = tmp_path / "results.json"
    monkeypatch.setenv("NB200_RESULTS_JSON", str(path))
    monkeypatch.chdir(ROOT)
    prob = build_problem("csp_small")
    for B in (0, 8):
        sim = _stepped(prob, B)
        sim.validate("problems/csp.params")  # an entry of problems/neutral.tests
        doc = json.loads(path.read_text())
        if B:
            assert set(doc) == TODAY_KEYS | NEW_KEYS
            assert doc["tally_batches"] == B
            assert doc["tally_total_relative_error"] == pytest.approx(
                sim.tally_relative_error()[1], rel=1e-12)
        else:
            assert set(doc) == TODAY_KEYS
        sim.free()
        path.unlink()
