"""The tally collective of sharded runs on the GPU (csrc/group.cu, capi.cu: group_layout,
group_reduce, group_flush, enqueue_step's group branch, nb200_mp_init / nb200_mp_connect).

* Multi-process groups: N rank processes (torch.multiprocessing, spawn), blobs exchanged with a
  gloo all_gather over 127.0.0.1, every rank on the same GPU (CUDA IPC maps memory between
  processes on one device, so the whole peer-memory protocol runs on one B200) or rank r on
  device r. Several cases per spawn, a new group per case.
* In-process sharding (option ngpus) over 2, 3, 5 and 8 GPUs, both collective flavours.
* nb200_update_replicas, and nb200_accumulate[_clear] against numpy.

Every case is held to three references: the oracle port on the whole bank (counts, shards bit
for bit, per-particle counters, the tally at every look to 1e-10 per cell); every rank's copy of
the tally equal to every other rank's, bit for bit; and, on the deterministic banks of
collective_cases.exact_bank, the rank-order sum that group.cu documents, bit for bit for the
peer-memory flavour and within the summation bound for NCCL.

Ranks never assert inside the protocol (a rank that stops early leaves its peers in the bounded
wait): they report data, the parent asserts. Every look at a tally is a download, which flushes,
so every rank makes the same looks in the same order."""
import ctypes as C
import os
import queue
import socket
import time
import traceback
from dataclasses import replace
from datetime import timedelta

import numpy as np
import pytest

from collective_cases import (Case, SCHEDULES, exact_bank, group_events, layout,
                              rank_order_looks, summation_bound_violations, timesteps, windows)
from neutral_b200.decks import build_problem, shard_range
from neutral_b200.host import NB200_MP_BLOB_BYTES, DeviceArray, Simulation, _check
from test_gpu_parity import tally_close

pytestmark = pytest.mark.gpu

GUARD = 2


class Tallies:
    """The caller's tallies "A" and "B", each `offset` doubles into an allocation of its own
    (allocate_data: 256-byte aligned), followed by GUARD doubles."""

    def __init__(self, lib, ncells: int, offset: int):
        self.lib, self.ncells, self.offset = lib, ncells, offset
        self.base = {k: DeviceArray(ncells + offset + GUARD) for k in "AB"}

    def ptr(self, k: str) -> int:
        return self.base[k].ptr + 8 * self.offset

    def look(self, k: str) -> np.ndarray:
        """A download of the tally: flushes the group when it is the group's tally."""
        out = np.empty(self.ncells)
        _check(self.lib.nb200_memcpy_d2h(out.ctypes.data, self.ptr(k), self.ncells * 8),
               "memcpy_d2h")
        return out

    def outside(self) -> np.ndarray:
        """The doubles of both allocations that are not the tallies (must stay 0)."""
        parts = []
        for a in self.base.values():
            whole = a.download()
            parts += [whole[:self.offset], whole[self.offset + self.ncells:]]
        return np.concatenate(parts)

    def free(self) -> None:
        for a in self.base.values():
            a.free()


def _key(r):
    return (r.facets, r.collisions, r.processed)


def run_schedule(sim: Simulation, schedule: str, tallies: Tallies) -> dict:
    """The schedule's timesteps and looks on one rank (or one sharded bank)."""
    counts, looks = {}, []
    for op in SCHEDULES[schedule]:
        if op[0] == "step":
            counts[op[1]] = _key(sim.step(op[1], tally_ptr=tallies.ptr(op[2])))
        elif op[0] == "look":
            looks.append(tallies.look(op[1]))
        else:  # Simulation.run_pipelined into tally A: `depth` timesteps in flight
            _, first, n, depth = op
            inflight = []
            for tt in range(first, first + n):
                sim.step(tt, tally_ptr=tallies.ptr("A"), defer=True)
                inflight.append(tt)
                if len(inflight) >= depth:
                    counts[inflight.pop(0)] = _key(sim.step_finish())
            while inflight:
                counts[inflight.pop(0)] = _key(sim.step_finish())
    return dict(counts=counts, looks=looks, outside=tallies.outside(),
                bank=sim.bank_to_host().arrays,
                counters=sim.counters_to_host() if sim.counters else None)


def _load(sim: Simulation, case: Case, prob, nranks: int) -> None:
    if case.bank == "exact":
        sim.load_bank(exact_bank(prob, nranks).slice(sim.pid0, sim.count))
    else:
        sim.inject()


# ---------------------------------------------------------------------------- references --


def port_schedule(port, prob, bank, schedule: str):
    """The oracle port on the whole bank: counts per timestep, the tally at every look, the final
    bank and per-particle counters."""
    d = prob.deck
    bank = bank.copy()
    tallies = {"A": np.zeros(d.nx * d.ny), "B": np.zeros(d.nx * d.ny)}
    ctr = np.zeros((3, len(bank)), dtype=np.uint64)
    counts, looks = {}, []
    for op in SCHEDULES[schedule]:
        if op[0] == "look":
            looks.append(tallies[op[1]].copy())
        else:
            for tt, t in timesteps([op]):
                counts[tt] = port.step(prob, bank, tt, tallies[t], counters=ctr)
    return counts, looks, bank, ctr


def rank_deltas(prob, bank, nranks: int, wins):
    """deltas[r][window]: shard r of `bank` stepped on one GPU, outside any group, into a freshly
    zeroed array for every reduction window."""
    d = prob.deck
    out = []
    for r in range(nranks):
        sim = Simulation(prob, rank=r, nranks=nranks, per_particle_counters=False)
        sim.load_bank(bank.slice(sim.pid0, sim.count))
        buf = DeviceArray(d.nx * d.ny)
        per = {}
        for w in wins:
            buf.zero()
            for tt in w:
                sim.step(tt, tally_ptr=buf.ptr)
            per[w] = buf.download()
        out.append(per)
        buf.free()
        sim.free()
    return out


def check_case(port, case: Case, nranks: int, results, flavour: str) -> None:
    """results: [(first particle, count, run_schedule result)] of every rank (one entry for an
    ngpus bank); flavour: "peer" or "nccl", the collective that combined them."""
    prob = case.problem(nranks)
    d = prob.deck
    ncells = d.nx * d.ny
    bank = case.host_bank(prob, nranks, port)
    want_counts, want_looks, want_bank, want_ctr = port_schedule(port, prob, bank, case.schedule)
    # 1. the oracle port
    got_counts = {tt: tuple(sum(res["counts"][tt][i] for _, _, res in results) for i in range(3))
                  for tt in want_counts}
    assert got_counts == want_counts
    for first, count, res in results:
        for k, v in want_bank.arrays.items():
            assert res["bank"][k].tobytes() == v[first:first + count].tobytes(), (first, k)
        if res["counters"] is not None:
            assert np.array_equal(res["counters"], want_ctr[:, first:first + count]), first
        assert not np.any(res["outside"]), "a write outside the tally"
        assert len(res["looks"]) == len(want_looks)
        for i, (got, want) in enumerate(zip(res["looks"], want_looks)):
            assert tally_close(got, want), (first, "look", i)
    # 2. every rank holds the same tally
    for _, _, res in results[1:]:
        for a, b in zip(res["looks"], results[0][2]["looks"]):
            assert a.tobytes() == b.tobytes(), "ranks disagree on the tally"
    if case.bank != "exact":
        return
    # 3. the rank-order sum
    events = group_events(SCHEDULES[case.schedule], case.reduce_every)
    deltas = rank_deltas(prob, bank, nranks, windows(events))
    got = results[0][2]["looks"]
    if flavour == "peer":
        want = rank_order_looks(events, deltas, ncells)
        for i, (g, w) in enumerate(zip(got, want)):
            bad = np.flatnonzero(g.view(np.uint64) != w.view(np.uint64))
            assert bad.size == 0, (f"look {i}: {bad.size} cells differ from the rank-order sum, "
                                   f"first {bad[:5]} of slices {layout(ncells, nranks)}")
        if nranks >= 3 and ncells >= 1000:  # the check tells the rank order from the reverse
            rev = rank_order_looks(events, deltas[::-1], ncells)
            assert any(not np.array_equal(a, b) for a, b in zip(rev, want))
    else:
        assert summation_bound_violations(events, deltas, got, ncells) == []


# ------------------------------------------------------------------- multi-process groups --

#: cases per group size, every rank on one GPU (and again one rank per GPU where there are enough)
SAME_GPU = {
    2: [Case("m9999", "exact", 0, 592, "looks"),
        Case("m9999", "exact", 1, 1, "looks"),
        Case("m9999", "exact", 2, 3, "second_tally"),
        Case("m305909", "inject", 1, 592, "looks", nparticles=3000),
        Case("m305909", "exact", 2, 3, "second_tally", offset=1),
        Case("csp_small", "inject", 1, 592, "pipe4"),
        Case("mixed_small", "inject", 0, 3, "second_tally", offset=1)],
    3: [Case("m9999", "exact", 0, 592, "looks"),
        Case("m9999", "exact", 1, 3, "pipe3"),
        Case("m9999", "exact", 2, 1, "second_tally"),
        Case("m9999", "exact", 1, 592, "pipe4", offset=1),
        Case("csp_small", "inject", 2, 592, "looks")],
    4: [Case("m9", "exact", 0, 1, "looks"),
        Case("m9", "exact", 1, 3, "pipe4"),
        Case("m9", "exact", 2, 592, "second_tally"),
        Case("m9", "inject", 1, 592, "looks", nparticles=400),
        Case("mixed_small", "inject", 1, 1, "pipe3")],
}
#: NCCL, and the fallback to it when peer mapping is refused: one rank per GPU only
SPREAD_ONLY = {
    2: [(replace(SAME_GPU[2][1], collective=0), False),
        (replace(SAME_GPU[2][3], collective=0), False),
        (SAME_GPU[2][0], True)],
    3: [(replace(SAME_GPU[3][1], collective=0), False),
        (replace(SAME_GPU[3][2], collective=0), False),
        (SAME_GPU[3][3], True)],
    4: [(replace(SAME_GPU[4][2], collective=0), False)],
}


def _plan(placement: str, nranks: int):
    plan = [(c, False) for c in SAME_GPU[nranks]]
    return plan + SPREAD_ONLY[nranks] if placement == "spread" else plan


def _case_id(case: Case, ipc_fail: bool) -> str:
    return case.id + ("-ipcfail" if ipc_fail else "")


MP_PARAMS = [(p, n, c, f) for p in ("same", "spread") for n in SAME_GPU for c, f in _plan(p, n)]


def _connect(lib, dist, torch, world: int, rank: int, ncells: int) -> str:
    """nb200_mp_init, the exchange of the blobs, nb200_mp_connect on every rank; when a peer
    cannot be mapped (-7), every rank finalizes and forms the group again with the NCCL flavour,
    as bench.py's connect_group does. Returns the flavour and, after a fallback, why."""

    def attempt():
        blob = (C.c_char * NB200_MP_BLOB_BYTES)()
        rc = lib.nb200_mp_init(world, rank, ncells, blob)
        mine = torch.frombuffer(bytearray(blob.raw), dtype=torch.uint8)
        everyone = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(everyone, mine)
        if rc == 0:
            rc = lib.nb200_mp_connect(b"".join(t.numpy().tobytes() for t in everyone))
        ok = torch.tensor([1 if rc == 0 else 0])
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item()), rc

    ok, rc = attempt()
    if ok:
        return "peer" if lib.nb200_get_option(b"collective") else "nccl"
    why = f"{rc}: {lib.nb200_last_error().decode()}"
    lib.nb200_mp_finalize()
    lib.nb200_set_option(b"collective", 0)
    ok, rc = attempt()
    if not ok:
        raise RuntimeError(f"cannot form the group: {why}; {rc}: "
                           f"{lib.nb200_last_error().decode()}")
    return f"nccl after {why}"


def _case_in_group(lib, dist, torch, rank: int, nranks: int, case: Case, ipc_fail: bool):
    prob = case.problem(nranks)
    d = prob.deck
    for name, value in ((b"collective", case.collective), (b"reduce_ctas", case.reduce_ctas),
                        (b"tally_reduce_every", case.reduce_every)):
        lib.nb200_set_option(name, value)
    if ipc_fail:
        os.environ["NB200_TEST_IPC_FAIL"] = "1"
    try:
        how = _connect(lib, dist, torch, nranks, rank, d.nx * d.ny)
    finally:
        os.environ.pop("NB200_TEST_IPC_FAIL", None)
    sim = Simulation(prob, rank=rank, nranks=nranks)
    _load(sim, case, prob, nranks)
    tallies = Tallies(lib, d.nx * d.ny, case.offset)
    out = run_schedule(sim, case.schedule, tallies)
    out["how"] = how
    sim.free()
    tallies.free()
    dist.barrier()  # nobody's slab is unmapped while a peer could still read it
    lib.nb200_mp_finalize()
    return out


def _rank_main(rank, nranks, placement, plan, port_no, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port_no), OMP_NUM_THREADS="1")
    import torch
    import torch.distributed as dist
    try:
        dist.init_process_group("gloo", rank=rank, world_size=nranks,
                                timeout=timedelta(seconds=120))
    except BaseException:
        q.put((rank, "error", traceback.format_exc()))
        return
    try:
        err = ""
        try:  # every device stays visible; the rank selects its own, as bench.py does
            torch.cuda.set_device(rank if placement == "spread" else 0)
            torch.zeros(1, device="cuda")
            from neutral_b200.host import load_library
            lib = load_library()
            if lib.nb200_device_count() <= 0:
                err = "the library sees no device"
        except Exception as exc:
            err = f"{type(exc).__name__}: {exc}"
        errs = [None] * nranks
        dist.all_gather_object(errs, err)
        if any(errs):
            q.put((rank, "nocontext", "; ".join(f"rank {r}: {e}" for r, e in enumerate(errs) if e)))
            return
        lib.nb200_set_option(b"print", 0)
        results = {}
        for case, ipc_fail in plan:
            results[_case_id(case, ipc_fail)] = _case_in_group(lib, dist, torch, rank, nranks,
                                                               case, ipc_fail)
        q.put((rank, "ok", results))
    except BaseException:
        q.put((rank, "error", traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _spawn(placement: str, nranks: int, timeout: float = 600.0):
    """Runs every case of the plan in one group of `nranks` processes; returns
    {rank: (status, payload)}. Children are joined with timeouts, then killed and reaped."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port_no = _free_port()
    procs = [ctx.Process(target=_rank_main,
                         args=(r, nranks, placement, _plan(placement, nranks), port_no, q))
             for r in range(nranks)]
    got = {}
    try:
        for p in procs:
            p.start()
        deadline = time.monotonic() + timeout
        while len(got) < nranks:
            try:
                rank, status, payload = q.get(timeout=2.0)
                got[rank] = (status, payload)
                continue
            except queue.Empty:
                pass
            gone = [r for r, p in enumerate(procs) if p.exitcode is not None and r not in got]
            if gone:
                time.sleep(1.0)  # a result still in the pipe
                while not q.empty():
                    rank, status, payload = q.get()
                    got[rank] = (status, payload)
                gone = [r for r in gone if r not in got]
                if gone:
                    return {r: ("error", f"exited with {procs[r].exitcode} before reporting")
                            for r in gone}
            if time.monotonic() > deadline:
                return {0: ("error", f"no result after {timeout} s")}
        for p in procs:
            p.join(timeout=60)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
            p.join(timeout=10)
    return got


_MP_RUNS = {}


def _mp_results(placement: str, nranks: int):
    key = (placement, nranks)
    if key not in _MP_RUNS:
        _MP_RUNS[key] = _spawn(placement, nranks)
    return _MP_RUNS[key]


@pytest.mark.parametrize("placement,nranks,case,ipc_fail", MP_PARAMS,
                         ids=[f"{p}-n{n}-{_case_id(c, f)}" for p, n, c, f in MP_PARAMS])
def test_multi_process_group(gpu_lib, port, placement, nranks, case, ipc_fail):
    """N processes form a group (nb200_mp_init / nb200_mp_connect) and step their shards; every
    rank's tally at every look against the port, the other ranks and the rank-order sum."""
    if placement == "spread" and gpu_lib.nb200_device_count() < nranks:
        pytest.skip(f"one rank per GPU needs {nranks} GPUs, "
                    f"{gpu_lib.nb200_device_count()} visible")
    prob = case.problem(nranks)
    ncells = prob.deck.nx * prob.deck.ny
    assert sum(c for _, c in layout(ncells, nranks)) == ncells
    runs = _mp_results(placement, nranks)
    statuses = {s for s, _ in runs.values()}
    if statuses == {"nocontext"}:
        pytest.skip(f"a rank cannot create a CUDA context: {runs[0][1]}")
    errors = {r: p for r, (s, p) in runs.items() if s != "ok"}
    assert not errors, errors
    results = []
    for r in range(nranks):
        res = runs[r][1][_case_id(case, ipc_fail)]
        first, count = shard_range(prob.deck.nparticles, r, nranks)
        results.append((first, count, res))
    hows = {res["how"] for _, _, res in results}
    assert len(hows) == 1
    how = hows.pop()
    if ipc_fail:
        assert how.startswith("nccl after -7"), how
    else:
        assert how == ("peer" if case.collective else "nccl"), how
    check_case(port, case, nranks, results, "peer" if how == "peer" else "nccl")


# --------------------------------------------------------------- in-process sharding (ngpus) --

NGPUS_CASES = [Case("m9999", "exact", 0, 592, "looks"),
               Case("m9999", "exact", 1, 3, "pipe4"),
               Case("m9", "exact", 2, 1, "second_tally"),
               Case("m305909", "inject", 2, 592, "looks", nparticles=3000, offset=1),
               Case("m305909", "exact", 1, 3, "pipe3"),
               Case("csp_small", "inject", 1, 592, "second_tally"),
               Case("mixed_small", "inject", 0, 1, "looks", offset=1)]
NGPUS_PARAMS = [(n, replace(c, collective=f)) for n in (2, 3, 5, 8) for c in NGPUS_CASES
                for f in (1, 0)]


@pytest.mark.parametrize("nranks,case", NGPUS_PARAMS,
                         ids=[f"n{n}-{c.id}" for n, c in NGPUS_PARAMS])
def test_bank_sharded_inside_the_library(gpu_lib, port, nranks, case):
    """One process, `nranks` GPUs (option ngpus), on the same meshes, schedules and references
    as the multi-process groups."""
    if gpu_lib.nb200_device_count() < nranks:
        pytest.skip(f"needs {nranks} GPUs, {gpu_lib.nb200_device_count()} visible")
    prob = case.problem(nranks)
    d = prob.deck
    prev = {name: gpu_lib.nb200_set_option(name, value) for name, value in
            ((b"collective", case.collective), (b"reduce_ctas", case.reduce_ctas),
             (b"tally_reduce_every", case.reduce_every))}
    try:
        # NCCL flavour: no peer access, so the secondary shards cannot reach the counters
        sim = Simulation(prob, ngpus=nranks, per_particle_counters=bool(case.collective))
        _load(sim, case, prob, nranks)
        assert gpu_lib.nb200_bank_gpus(sim.bank) == nranks
        tallies = Tallies(gpu_lib, d.nx * d.ny, case.offset)
        res = run_schedule(sim, case.schedule, tallies)
        sim.free()
        tallies.free()
    finally:
        for name, value in prev.items():
            gpu_lib.nb200_set_option(name, value)
    check_case(port, case, nranks, [(0, d.nparticles, res)],
               "peer" if case.collective else "nccl")


def test_update_replicas_after_an_in_place_density_edit(gpu_lib, port):
    """The secondary GPUs of a sharded bank work on replicas of the density: after the caller
    edits it in place and calls nb200_update_replicas, every shard transports against the new
    values."""
    if gpu_lib.nb200_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    prob = build_problem("mixed_small", iterations=4)
    d = prob.deck
    sim = Simulation(prob, ngpus=min(gpu_lib.nb200_device_count(), 3))
    sim.inject()
    bank = port.inject(prob)
    tally = np.zeros(d.nx * d.ny)
    ctr = np.zeros((3, len(bank)), dtype=np.uint64)
    for tt in range(1, d.iterations + 1):
        if tt == 3:  # a band of cells through the source and the dense boxes
            prob.density[30:45, :] = 3.0
            sim.density.upload(prob.density.ravel())
            assert gpu_lib.nb200_update_replicas() == 0
        want = port.step(prob, bank, tt, tally, counters=ctr)
        assert _key(sim.step(tt)) == want, tt
        assert sum(sim.bank_to_host().bit_equal(bank).values()) == 0, tt
    assert np.array_equal(sim.counters_to_host(), ctr)
    assert tally_close(sim.tally_to_host(), tally)
    sim.free()


# ------------------------------------------------------------- nb200_accumulate[_clear] --

ACC_N = [1, 2, 3, 606207, 606208, 606209, 1212417, 5000001]  # one grid pass: 606 208


def _values(rng, n):
    special = np.array([0.0, -0.0, 5e-324, -5e-324, 1e-310, -2.5e-315, 2.2250738585072014e-308,
                        1e300, -1e300, 1e-300, -1e-300, 1.7e308, -1.7e308, 1.0, -1.0, 3.0])
    v = np.where(rng.random(n) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-320.0, 305.0, n)
    pick = rng.random(n) < 0.3
    v[pick] = special[rng.integers(len(special), size=int(pick.sum()))]
    return v


@pytest.mark.parametrize("clear", [False, True])
@pytest.mark.parametrize("dst_off,src_off", [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("n", ACC_N)
def test_accumulate_against_numpy(gpu_lib, n, dst_off, src_off, clear):
    """dst = dst + src, one IEEE addition per element, bit for bit as numpy; src all +0.0 after
    the clear; the doubles around both ranges untouched. Pointers at +1 element are only 8-byte
    aligned."""
    rng = np.random.default_rng(n + 10 * dst_off + 20 * src_off)
    dst, src = _values(rng, n), _values(rng, n)
    host_d = np.full(dst_off + n + GUARD, 7.0)
    host_s = np.full(src_off + n + GUARD, 3.0)
    host_d[dst_off:dst_off + n], host_s[src_off:src_off + n] = dst, src
    dd, ds = DeviceArray.from_host(host_d), DeviceArray.from_host(host_s)
    try:
        pd, ps = dd.ptr + 8 * dst_off, ds.ptr + 8 * src_off
        rc = gpu_lib.nb200_accumulate_clear(pd, ps, n) if clear else \
            gpu_lib.nb200_accumulate(pd, ps, n)
        assert rc == 0
        got_d, got_s = dd.download(), ds.download()
    finally:
        dd.free()
        ds.free()
    with np.errstate(over="ignore"):
        want = dst + src
    assert got_d[dst_off:dst_off + n].view(np.uint64).tobytes() == want.view(np.uint64).tobytes()
    if clear:
        assert not np.any(got_s[src_off:src_off + n].view(np.uint64))
    else:
        assert got_s[src_off:src_off + n].tobytes() == src.tobytes()
    assert np.all(got_d[:dst_off] == 7.0) and np.all(got_d[dst_off + n:] == 7.0)
    assert np.all(got_s[:src_off] == 3.0) and np.all(got_s[src_off + n:] == 3.0)
