#!/usr/bin/env python3
"""bench.py - particle events/s of neutral's particle-history hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--deck csp] [--particles P] [--scaling weak|strong] [--dump-outputs DIR]

One "step" = one complete run of the deck named in ``config.workload`` (default csp: 4000 x
4000 mesh, 1e6 particles per GPU, 10 timesteps of solve_transport_2d) from the freshly
injected bank, ending with the caller-visible tally complete. Prints ONE JSON line (rank 0):

* ``value``     whole-job events/s ( facets + collisions + census over all ranks and the K
                timed steps / device time, max over ranks ), inputs resident in HBM;
* ``e2e``       the same metric with HOST buffers: every step uploads the deck (mesh,
                cross sections, bank) from pinned host memory, runs the timesteps through
                solve_transport_2d, and reads tally and bank back (double-buffered: the
                copies of neighbouring steps overlap a step's transport);
* ``roofline``  the history kernel against the ceiling that binds it - the rate at which the
                L2 retires FP64 reductions, MEASURED IN THIS RUN by the library's microbenchmark
                (one reduction per facet / census / death, omp3/neutral.c:408-420) - with the
                SURVEY.md 8d HBM model (facet 200 B, collision 176 B, census 192 B, fatal
                collision +16 B against the measured HBM peak) kept beside it as ``hbm``;
* ``parity``    the timed runs' own results against tests/golden/full_decks.json (generated
                from the unmodified reference omp3 library): per-timestep event counts summed
                over the ranks, sha256 of every field of the final bank, tally total and
                64 x 64 block sums;
* ``decks``     (N = 1) resident events/s of the other BASELINE.json decks;
* ``cpu_baseline`` the unmodified reference omp3 build (oracle/_ref) on this box's host
                cores on the full deck (N = 1 only).

``--impl reference`` times the reference's own CPU implementation instead (rank 0 only).
N > 1 (torchrun, one process per GPU): every rank transports a contiguous particle range
(global RNG keys) against replicated mesh and tables; ``--scaling weak`` (default) grows the
global bank with N (``deck.nparticles`` per GPU), ``--scaling strong`` splits the deck's own
bank. The tally is combined inside the library: a peer-memory reduce-scatter kernel per
timestep over CUDA IPC (csrc/nb_group.cuh), or NCCL with ``--opts collective=0``.
torch.distributed is used to exchange the IPC handles and to reduce the timings, nothing else.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree

METRIC = "particle_events_per_sec"
UNIT = "events/s"
# SURVEY.md 8d: algorithmic bytes per event of the event-based model
B_FACET, B_COLLISION, B_CENSUS, B_DEATH_EXTRA = 200.0, 176.0, 192.0, 16.0
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
# warp instructions one collision round of a warp issues (profiles/r01/ncu_final2_scatter_lines.txt)
COLLISION_WARP_INSTRUCTIONS = 800.0
GOLDEN_FULL = os.path.join(ROOT, "tests", "golden", "full_decks.json")
OTHER_DECKS = ("stream", "split", "scatter")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--deck", default="csp")
    ap.add_argument("--particles", type=int, default=0,
                    help="override particles (per GPU when weak scaling, global when strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-decks", action="store_true")
    ap.add_argument("--opts", default="", help="library options, e.g. pipeline=0,fast_div=0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def workload_config(deck, nglobal: int, world: int, scaling: str):
    """The `config` object: identical in both arms for the same command line."""
    per_gpu = nglobal // world
    return {"workload": f"{deck.name}.params: {deck.nx}x{deck.ny} mesh, {per_gpu} particles per "
                        f"GPU ({nglobal} global), {deck.iterations} timesteps per step, fresh "
                        "bank each step",
            "deck": deck.name, "mesh": [deck.nx, deck.ny], "particles_global": nglobal,
            "timesteps_per_step": deck.iterations, "scaling": scaling,
            "l2_policy": "inputs larger than L2 (density + tally = "
                         f"{2 * deck.nx * deck.ny * 8 / 2**20:.0f} MiB, random access)"}


def global_particles(deck, args, world: int) -> int:
    if args.scaling == "strong":
        return args.particles or deck.nparticles
    return (args.particles or deck.nparticles) * world


# ------------------------------------------------------------------------------ clocks --

class ClockSampler:
    """Samples nvidia-smi every 100 ms (B200_PROFILING.md clocks line). It is started before
    the warm-up so that it is already reporting when the timed regions begin; only samples
    that arrived inside a timed region (`window(t0, t1)`) count."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []  # (arrival time, csv line)
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window(self, t0: float, t1: float):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # a sample describes the 100 ms before it arrived
        inside = [ln for t, ln in self.lines
                  if any(t0 <= t <= t1 + 0.1 for t0, t1 in self.windows)]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------- reference (CPU) arm --

def reference_rate(deck_name: str, nglobal: int, budget_seconds: float, steps: int = 1,
                   warmup: int = 0):
    """Times the unmodified reference omp3 build (oracle/_ref, else the oracle port) on this
    host, all cores. Each step is the FULL deck (`nglobal` particles) when `steps + warmup` of
    them fit `budget_seconds`, else the largest particle sample that does (the rate is
    scale-free: histories are independent). Returns a dict for the JSON line."""
    from neutral_b200.decks import build_problem, load_deck
    from oracle.oracle import OraclePort, ReferenceOmp3

    cores = len(os.sched_getaffinity(0))
    # All the host threads the box has, whatever the launcher exported: torchrun sets
    # OMP_NUM_THREADS=1 for its workers, which would time the reference on one core while
    # reporting sixteen. NB200_REF_THREADS overrides.
    cores = int(os.environ.get("NB200_REF_THREADS", cores))
    os.environ["OMP_NUM_THREADS"] = str(cores)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    kind = "reference" if ReferenceOmp3.available() else "port"
    eng = ReferenceOmp3() if kind == "reference" else OraclePort()
    try:  # the OpenMP runtime may have read the environment before this point (torch loads one)
        C.CDLL("libgomp.so.1").omp_set_num_threads(cores)
    except OSError:
        pass
    deck = load_deck(deck_name)

    def run_once(nparticles):
        prob = build_problem(deck, nparticles=nparticles)
        d = prob.deck
        tally = np.zeros(d.nx * d.ny)
        bank = eng.inject(prob)
        dead = (lambda: bank["dead"]) if kind == "reference" else (lambda: bank.dead)
        events, seconds = 0, 0.0
        for tt in range(1, d.iterations + 1):
            t0 = time.perf_counter()
            counts = eng.step(prob, bank, tt, tally)  # (facets, collisions[, processed])
            seconds += time.perf_counter() - t0
            # census events = particles still alive after the step (SURVEY.md 8d)
            events += counts[0] + counts[1] + int(np.count_nonzero(dead() == 0))
        return events, seconds

    # calibrate on a small sample, then decide between the full deck and a bounded sample
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)  # the reference prints "Particles N" every timestep
    try:
        n0 = min(nglobal, max(2000 * cores, 100_000))
        ev0, s0 = run_once(n0)
        per_particle_s = s0 / n0
        runs = max(steps + warmup, 1)
        n = nglobal
        # a small sample over-estimates the cost per particle (thread imbalance, cold caches):
        # the full deck runs unless the estimate misses the budget by more than a fifth
        if per_particle_s * nglobal * runs > 1.2 * budget_seconds:
            n = int(max(n0, min(nglobal, budget_seconds / runs / per_particle_s)))
        times, events = [], 0
        for i in range(warmup + steps):
            ev, s = run_once(n)
            if i >= warmup:
                times.append(s)
                events += ev
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    total = sum(times)
    what = "the full deck" if n == nglobal else "a bounded sample"
    return {"value": events / total, "unit": UNIT, "cores": cores, "kind": kind,
            "full_deck": n == nglobal,
            "sample": f"{deck.name}: {n} of {nglobal} particles ({what}), {deck.iterations} "
                      f"timesteps, {deck.nx}x{deck.ny} mesh, {steps} run(s) of "
                      f"{total / max(steps, 1):.1f} s, OMP threads={cores}",
            "ms_per_step": 1e3 * total / max(steps, 1), "events_per_step": events / max(steps, 1)}


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    from neutral_b200.decks import load_deck
    deck = load_deck(args.deck)
    nglobal = global_particles(deck, args, max(world, args.gpus, 1))
    budget = float(os.environ.get("NB200_REF_BUDGET_S", "480"))
    res = reference_rate(args.deck, nglobal, budget, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(deck, nglobal, max(world, args.gpus, 1), args.scaling),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample",
                                             "full_deck")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------- b200 (GPU) arm --

def algorithmic_bytes(results):
    return sum(r.facets * B_FACET + r.collisions * B_COLLISION + r.census * B_CENSUS +
               r.deaths * B_DEATH_EXTRA for r in results)


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch(deck_name):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            entry = json.load(f).get(deck_name, {})
            return entry.get("dram_bytes_per_launch"), entry.get("source")
    except (OSError, ValueError):
        return None, None


def fused_history_bytes(results):
    """Lower bound on the bytes a fused-history kernel must move (SURVEY.md 8d, B_hist): the
    80-byte record in and out once per particle-timestep, the entered cell's density and the
    tally read-modify-write per facet, the tally RMW per census or death."""
    return sum(r.processed * 160.0 + r.facets * 24.0 + (r.census + r.deaths) * 16.0
               for r in results)


def measure_red_peaks(lib):
    """The L2 FP64-reduction ceiling of THIS GPU, measured now (csrc/microbench.cu): ~60 ms."""
    out = {}
    rate = C.c_double(0.0)
    for name, pattern, mib in (("peak_l2_resident_strided", 3, 16), ("mesh_walk_128MiB", 1, 128),
                               ("random_128MiB", 0, 128)):
        if lib.nb200_microbench_red(pattern, mib << 20, 400, C.byref(rate)) == 0:
            out[name] = rate.value
    return out


def block_sums(tally, nx, ny, blocks=64):
    t = tally.reshape(ny, nx)
    by, bx = ny // blocks, nx // blocks
    return t[:by * blocks, :bx * blocks].reshape(blocks, by, blocks, bx).sum(axis=(1, 3)).ravel()


def golden_for(deck, nglobal):
    try:
        with open(GOLDEN_FULL) as f:
            g = json.load(f)
    except (OSError, ValueError):
        return None, None
    from neutral_b200.decks import load_deck
    base = deck.name[:-len("_scaled")] if deck.name.endswith("_scaled") else deck.name
    key = base if nglobal == load_deck(base).nparticles else f"{base}@{nglobal}"
    return g.get(key), key


def parity_report(deck, nglobal, counts_global, tally, bank_hashes, live):
    """Compares what the timed runs produced with the reference-generated fixture."""
    g, key = golden_for(deck, nglobal)
    if g is None:
        return {"fixture": key, "checked": False,
                "why": "no fixture for this deck and particle count in tests/golden/full_decks.json"}
    rep = {"fixture": f"tests/golden/full_decks.json[{key}] (unmodified reference omp3 library)",
           "checked": True}
    rep["counts_match"] = [list(c) for c in counts_global] == g["counts"]
    rep["timesteps"] = len(counts_global)
    rep["facets"] = int(sum(c[0] for c in counts_global))
    rep["collisions"] = int(sum(c[1] for c in counts_global))
    if live is not None:
        rep["live_particles_match"] = int(live) == g["live"]
    if bank_hashes is not None:
        rep["bank_bit_identical"] = bank_hashes == g["final_hashes"]
    if tally is not None:
        total = float(tally.sum())
        rep["tally_sum"] = total
        rep["tally_sum_rel_err"] = abs(total - g["tally_sum"]) / abs(g["tally_sum"])
        img, want = block_sums(tally, deck.nx, deck.ny), np.array(g["tally_block_sums"])
        scale = np.maximum(np.maximum(np.abs(img), np.abs(want)), 1e-300)
        rep["tally_block_max_rel_err"] = float(np.max(np.abs(img - want) / scale))
        rep["tally_tolerance"] = 1e-10  # north_star's per-cell bound, applied to the block sums
        rep["tally_match"] = bool(rep["tally_sum_rel_err"] <= 1e-10 and
                                  rep["tally_block_max_rel_err"] <= 1e-10)
    rep["ok"] = all(v for k, v in rep.items() if k.endswith("_match") or k == "bank_bit_identical")
    return rep


DUMP_SAMPLE = 1 << 18  # particles and tally cells sampled per dump (fixed seed): ~20 MB in all


def dump_outputs(out_dir, deck, last_run, bank, tally):
    """Writes what the last timed step returned to its caller as DIR/<name>.npy (float64): the
    per-timestep counts, the tally and every bank field - the larger arrays as a fixed, seeded
    sample of indices (written beside them) plus the tally's 64 x 64 block sums, so that two
    builds can be compared output for output on the same inputs."""
    os.makedirs(out_dir, exist_ok=True)

    def sample(n):
        if n <= DUMP_SAMPLE:
            return np.arange(n)
        return np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))

    out = {"counts": np.array([[r.facets, r.collisions, r.processed, r.census, r.deaths]
                               for r in last_run], dtype=np.float64),
           "tally_block_sums": block_sums(tally, deck.nx, deck.ny)}
    cells = sample(tally.size)
    out["tally_sample_index"], out["tally_sample"] = cells.astype(np.float64), tally[cells]
    pids = sample(len(bank))
    out["bank_sample_index"] = pids.astype(np.float64)
    for k, a in bank.arrays.items():
        out[f"bank_{k}"] = a[pids].astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def connect_group(lib, dist, torch, world, rank, ncells):
    """One library-side tally group over the ranks of this job: every rank allocates its slab,
    the CUDA-IPC handles travel through torch.distributed, every rank maps its peers."""
    from neutral_b200.host import NB200_MP_BLOB_BYTES

    def attempt():
        blob = (C.c_char * NB200_MP_BLOB_BYTES)()
        rc = lib.nb200_mp_init(world, rank, ncells, blob)
        mine = torch.frombuffer(bytearray(blob.raw), dtype=torch.uint8).cuda()
        everyone = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(everyone, mine)
        if rc == 0:
            blobs = b"".join(t.cpu().numpy().tobytes() for t in everyone)
            rc = lib.nb200_mp_connect(blobs)
        ok = torch.tensor([1 if rc == 0 else 0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item())

    if attempt():
        return "peer-memory reduce-scatter kernel over CUDA IPC" \
            if lib.nb200_get_option(b"collective") else "NCCL reduce-scatter (in-library)"
    why = lib.nb200_last_error().decode()
    lib.nb200_mp_finalize()
    lib.nb200_set_option(b"collective", 0)  # no peer path between these GPUs: NCCL flavour
    if not attempt():
        raise RuntimeError(f"cannot form the tally group: {why}; "
                           f"{lib.nb200_last_error().decode()}")
    return f"NCCL reduce-scatter (in-library; peer mapping failed: {why})"


def time_other_decks(lib, torch, names):
    """Resident events/s of the other BASELINE.json decks on one GPU (1 warm-up + 2 runs)."""
    from neutral_b200.decks import build_problem
    from neutral_b200.host import Simulation, _check, _soa_p
    out = {}
    for name in names:
        try:
            prob = build_problem(name)
            sim = Simulation(prob, per_particle_counters=False)
            sim.inject()
            snap = _soa_p()
            injected = sim.bank_to_host()  # must outlive as_struct(): the struct aliases it
            st = injected.as_struct()
            _check(lib.nb200_bank_create(C.byref(st), sim.count, sim.pid0, C.byref(snap)), "snap")
            del injected
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            res = []
            for i in range(3):
                _check(lib.nb200_bank_copy(sim.bank, snap), "bank_copy")
                sim.tally.zero()
                if i == 1:
                    torch.cuda.synchronize()
                    ev0.record()
                r = sim.run_pipelined()
                if i >= 1:
                    res += r
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / 2
            g, key = golden_for(prob.deck, prob.deck.nparticles)
            counts = [[r.facets, r.collisions] for r in res[:prob.deck.iterations]]
            out[name] = {"value": sum(r.events for r in res) / 2 / (ms / 1e3), "unit": UNIT,
                         "ms_per_step": ms, "particles": prob.deck.nparticles,
                         "timesteps_per_step": prob.deck.iterations,
                         "history_kernel_ms_per_step": sum(r.kernel_ns for r in res) / 2e6,
                         "counts_match_reference": (counts == g["counts"]) if g else None}
            lib.nb200_bank_free(snap)
            sim.free()
        except Exception as exc:  # a reported extra, never a gate
            out[name] = {"value": None, "error": str(exc)}
    return out


def run_b200_arm(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist

    from neutral_b200.bank import ALL_FIELDS, ParticleSoA
    from neutral_b200.decks import build_problem, load_deck
    from neutral_b200.host import NB200_BAD_OPTION, Simulation, _check, _soa_p, load_library

    torch.cuda.set_device(local_rank)
    if world > 1:
        # one process per GPU on one box: give every rank its own block of host cores, so that
        # eight hosts enqueueing kernels and copies do not migrate over each other
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = len(cores) // world
            if per >= 1:
                os.sched_setaffinity(0, cores[local_rank * per:(local_rank + 1) * per])
        except OSError:
            pass
        # stdout carries the one JSON line: keep NCCL's version banner off it
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = load_library(build=False)
    lib.initialise_devices.restype = None
    lib.nb200_set_option(b"print", 0)
    opts = dict(kv.split("=") for kv in args.opts.split(",") if kv)
    for k, v in opts.items():
        if lib.nb200_set_option(k.encode(), int(v)) == NB200_BAD_OPTION:
            sys.exit(f"bad library option {k}={v}: {lib.nb200_last_error().decode()}")
    pipeline = int(opts.get("pipeline", 1))
    reduce_every = lib.nb200_get_option(b"tally_reduce_every")

    deck = load_deck(args.deck)
    nglobal = global_particles(deck, args, world)
    prob = build_problem(deck, nparticles=nglobal)
    d = prob.deck
    ncells = d.nx * d.ny

    collective = None
    if world > 1:
        collective = connect_group(lib, dist, torch, world, rank, ncells)

    stage("problem built, injecting")
    sim = Simulation(prob, rank=rank, nranks=world, per_particle_counters=False)
    sim.inject()
    start_bank = sim.bank_to_host()  # host copy of the freshly injected shard
    # resident snapshot the timed steps restart from
    snap = _soa_p()
    st = start_bank.as_struct()
    _check(lib.nb200_bank_create(C.byref(st), sim.count, sim.pid0, C.byref(snap)), "snapshot")

    def one_step():
        """One deck run from the injected state to the complete tally; returns the StepResults.
        The timesteps are enqueued without a host round trip between them (defer_finish); in a
        sharded run every timestep's tally delta is reduce-scattered inside the library beside
        the next timestep, and the run ends with the all-gather into the caller's tally."""
        _check(lib.nb200_bank_copy(sim.bank, snap), "bank_copy")
        sim.tally.zero()
        out = sim.run_pipelined()
        if world > 1:
            sim.tally_sync()
        return out

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stage("warm-up")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        one_step()

    stage("timed region")
    launches0 = lib.nb200_kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    wall0 = time.time()
    ev0.record()
    timed = []
    for _ in range(args.steps):
        timed += one_step()
    ev1.record()
    fence()
    sampler.window(wall0, time.time())
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = lib.nb200_kernel_launches() - launches0

    events = sum(r.events for r in timed)
    kernel_ns = sum(r.kernel_ns for r in timed)
    sort_ns = sum(r.sort_ns for r in timed)
    hist_launches = len(timed)
    alg_bytes = algorithmic_bytes(timed)
    reductions = sum(r.facets + r.census + r.deaths for r in timed)
    collisions = sum(r.collisions for r in timed)
    if args.dump_outputs and rank == 0:  # a sharded run dumps rank 0's part of the bank
        dump_outputs(args.dump_outputs, d, timed[-d.iterations:], sim.bank_to_host(),
                     sim.tally_to_host())

    stage("parity")
    # ---- parity of the timed runs themselves (outside the timed region) ----------------
    last_run = timed[-d.iterations:]
    counts_local = torch.tensor([[r.facets, r.collisions] for r in last_run], dtype=torch.int64,
                                device="cuda")
    if world > 1:
        dist.all_reduce(counts_local)
    counts_global = counts_local.tolist()
    parity = None
    if not args.no_parity:
        final_bank = sim.bank_to_host()
        live = torch.tensor([int(np.count_nonzero(final_bank.dead == 0))], device="cuda")
        hashes = None
        if world > 1:
            dist.all_reduce(live)
        if nglobal <= 32_000_000:  # gather the shards' fields on rank 0 (injection order)
            hashes = {}
            for k in ALL_FIELDS:
                mine = torch.from_numpy(np.ascontiguousarray(final_bank.arrays[k])).cuda()
                if world > 1:
                    sizes = [0] * world
                    dist.all_gather_object(sizes, int(mine.numel()))
                    parts = [torch.empty(s, dtype=mine.dtype, device="cuda") for s in sizes] \
                        if rank == 0 else None
                    dist.gather(mine, parts, dst=0) if len(set(sizes)) == 1 else \
                        _gather_ragged(dist, torch, mine, parts, sizes, rank)
                    whole = torch.cat(parts).cpu().numpy() if rank == 0 else None
                else:
                    whole = final_bank.arrays[k]
                if rank == 0:
                    hashes[k] = hashlib.sha256(np.ascontiguousarray(whole).tobytes()).hexdigest()
        tally_host = sim.tally_to_host() if rank == 0 else None
        if rank == 0:
            parity = parity_report(d, nglobal, counts_global, tally_host, hashes, int(live.item()))
    tally_sum = float(sim.tally_to_host().sum()) if rank == 0 else 0.0

    # ---- e2e: host buffers in, host buffers out, every step ---------------------------
    # Every step uploads ALL of its inputs (mesh, edges, cross-section tables, bank) from
    # pinned host memory and downloads its results (tally, bank) to pinned host memory. The
    # steps are independent, so the transfers are double-buffered the way a production host
    # would: two device-side working sets; while step i transports on set i%2, the upload of
    # step i+1 and the download of step i-1 run on their own copy streams. Nothing is skipped:
    # the timed region holds K full uploads, K full runs and K full downloads.
    stage("e2e")
    e2e = None
    if not args.no_e2e:
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        h_density, h_ex, h_ey = pin(prob.density.ravel()), pin(prob.edgex), pin(prob.edgey)
        h_cs = [pin(a) for pair in (prob.cs_scatter, prob.cs_absorb) for a in pair]
        h_bank = {k: pin(v) for k, v in start_bank.arrays.items()}
        nbytes = lambda t: t.numel() * t.element_size()

        class WorkingSet:
            def __init__(self, s):
                self.sim = s
                self.view = ParticleSoA()
                _check(lib.nb200_bank_view(s.bank, C.byref(self.view)), "bank_view")
                self.inputs = [(s.density, h_density), (s.edgex, h_ex), (s.edgey, h_ey)] + \
                    list(zip(s._cs_arrays, h_cs))
                self.out_tally = torch.empty(ncells, dtype=torch.float64).pin_memory()
                self.out_bank = {k: torch.empty_like(v).pin_memory() for k, v in h_bank.items()}
                self.uploaded = torch.cuda.Event()
                self.downloaded = torch.cuda.Event()

            def field_ptr(self, k):
                return C.cast(getattr(self.view, k), C.c_void_p).value

        sim_b = Simulation(prob, rank=rank, nranks=world, per_particle_counters=False)
        sim_b.load_bank(start_bank)
        sets = [WorkingSet(sim), WorkingSet(sim_b)]
        up, down = torch.cuda.Stream(), torch.cuda.Stream()
        h2d = sum(nbytes(t) for _, t in sets[0].inputs) + sum(nbytes(t) for t in h_bank.values())
        d2h = ncells * 8 + sum(nbytes(t) for t in h_bank.values())

        def enqueue_upload(ws):
            up.wait_event(ws.downloaded)  # the set's previous results must have left it
            for dev, host in ws.inputs:
                _check(lib.nb200_memcpy_h2d_async(dev.ptr, host.data_ptr(), nbytes(host),
                                                  up.cuda_stream), "h2d")
            for k in ALL_FIELDS:
                _check(lib.nb200_memcpy_h2d_async(ws.field_ptr(k), h_bank[k].data_ptr(),
                                                  nbytes(h_bank[k]), up.cuda_stream), "h2d bank")
            ws.uploaded.record(up)

        trace = {} if os.environ.get("NB200_E2E_TRACE") else None

        def lap(name, t0):
            if trace is not None:
                trace[name] = trace.get(name, 0.0) + time.perf_counter() - t0
            return time.perf_counter()

        def transport(ws, once_fed=None):
            t = time.perf_counter()
            torch.cuda.current_stream().wait_event(ws.uploaded)
            if trace is not None:
                ws.uploaded.synchronize()
                t = lap("wait_upload", t)
            _check(lib.nb200_bank_import(ws.sim.bank), "bank_import")
            ws.sim.tally.zero()
            t = lap("import+zero (enqueue)", t)
            out = ws.sim.run_pipelined(once_fed=once_fed)
            t = lap("timesteps", t)
            if world > 1:
                ws.sim.tally_sync()
                t = lap("tally sync", t)
            _check(lib.nb200_bank_export(ws.sim.bank), "bank_export")  # synchronises
            lap("export", t)
            return out

        def enqueue_download(ws):
            _check(lib.nb200_memcpy_d2h_async(ws.out_tally.data_ptr(), ws.sim.tally.ptr,
                                              ncells * 8, down.cuda_stream), "d2h")
            for k in ALL_FIELDS:
                _check(lib.nb200_memcpy_d2h_async(ws.out_bank[k].data_ptr(), ws.field_ptr(k),
                                                  nbytes(h_bank[k]), down.cuda_stream), "d2h bank")
            ws.downloaded.record(down)

        def e2e_run(nsteps):
            # The ~30 copy calls of a step (download of the previous run's results, upload of
            # the next run's inputs) are issued once the GPU has this run's first timesteps
            # queued, not in the gap between two runs where it would sit idle behind them.
            out = []
            enqueue_upload(sets[0])
            for i in range(nsteps):
                def copies_of_the_neighbours(i=i):
                    if i > 0:
                        enqueue_download(sets[(i - 1) & 1])
                    if i + 1 < nsteps:
                        enqueue_upload(sets[(i + 1) & 1])
                out += transport(sets[i & 1], copies_of_the_neighbours)
            if nsteps > 0:
                enqueue_download(sets[(nsteps - 1) & 1])
            up.synchronize()
            down.synchronize()
            return out

        e2e_run(min(args.warmup, 2))
        fence()
        t0 = time.perf_counter()
        e2e_res = e2e_run(args.steps)
        fence()
        e2e_s = time.perf_counter() - t0
        if trace is not None:
            print("e2e host trace (ms per step):",
                  {k: round(1e3 * v / (args.steps + min(args.warmup, 2)), 3)
                   for k, v in trace.items()}, file=sys.stderr)
        sampler.window(time.time() - e2e_s, time.time())
        last = sets[(args.steps - 1) & 1]
        e2e = {"events": sum(r.events for r in e2e_res), "seconds": e2e_s, "h2d": h2d,
               "hist_ms": sum(r.kernel_ns for r in e2e_res) / 1e6 / args.steps,
               "sort_ms": sum(r.sort_ns for r in e2e_res) / 1e6 / args.steps,
               "d2h": d2h, "tally_sum": float(last.out_tally.sum()),
               "live_out": int((last.out_bank["dead"] == 0).sum())}

    stage("reduce over ranks")
    clocks = sampler.stop() if rank == 0 else None  # samples of both timed regions

    # ---- reduce over ranks -------------------------------------------------------------
    if world > 1:
        t = torch.tensor([elapsed_ms, e2e["seconds"] if e2e else 0.0,
                          kernel_ns / max(hist_launches, 1)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = torch.tensor([events, e2e["events"] if e2e else 0, launches, reductions, collisions,
                          e2e["live_out"] if e2e else 0],
                         device="cuda", dtype=torch.float64)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        elapsed_ms, e2e_seconds, slowest_launch_ns = float(t[0]), float(t[1]), float(t[2])
        events_all, e2e_events_all, launches_all = float(c[0]), float(c[1]), int(c[2])
        e2e_live_all = int(c[5])
    else:
        e2e_seconds = e2e["seconds"] if e2e else 0.0
        events_all, e2e_events_all, launches_all = float(events), \
            float(e2e["events"]) if e2e else 0.0, int(launches)
        slowest_launch_ns = kernel_ns / max(hist_launches, 1)
        e2e_live_all = e2e["live_out"] if e2e else 0

    if rank != 0:
        if world > 1:
            lib.nb200_mp_finalize()
            dist.destroy_process_group()
        return

    # ---- roofline: per-launch figures of THIS rank's history kernel (rank 0) -------------
    stage("roofline microbenchmark")
    red = measure_red_peaks(lib)
    red_peak = red.get("peak_l2_resident_strided")
    ach_red = reductions / max(kernel_ns, 1) * 1e9
    hbm_peak, hbm_src = measured_hbm_peak()
    ach_gbs = alg_bytes / max(kernel_ns, 1)  # bytes per ns == GB/s
    traffic, traffic_src = ncu_traffic_per_launch(deck.name)
    sm_hz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_hz * 1e6 * 32.0 / COLLISION_WARP_INSTRUCTIONS
    roofline = {
        "bound": "l2_fp64_atomics", "kernel": "k_history" if pipeline else "k_history_direct",
        "achieved": ach_red, "peak": red_peak, "unit": "fp64 reductions/s",
        "frac": ach_red / red_peak if red_peak else None,
        "peak_source": "measured in this run: nb200_microbench_red (csrc/microbench.cu), "
                       "red.global.add.f64 into an L2-resident 16 MiB footprint, 2 integer "
                       "instructions per reduction",
        "peak_other_patterns": {k: v for k, v in red.items() if k != "peak_l2_resident_strided"},
        "reductions_per_launch": reductions / max(hist_launches, 1),
        "avg_launch_ms": kernel_ns / max(hist_launches, 1) / 1e6,
        "slowest_rank_avg_launch_ms": slowest_launch_ns / 1e6,
        "launches_timed": hist_launches,
        "kernel_share_of_step": (kernel_ns / 1e6) / max(elapsed_ms, 1e-9),
        "sort_phase_share_of_step": (sort_ns / 1e6) / max(elapsed_ms, 1e-9),
        "traffic": traffic,
        # collision-dominated decks are bound by issue slots, not by the reductions: what the
        # SMs could retire if every slot issued one of the ~800 warp instructions a collision
        # round of 32 lanes costs (profiles/r01/ncu_final2_scatter_lines.txt)
        "issue_bound": {"achieved": collisions / max(kernel_ns, 1) * 1e9, "peak": issue_peak,
                        "unit": "collisions/s",
                        "frac": collisions / max(kernel_ns, 1) * 1e9 / issue_peak,
                        "peak_source": "148 SMs x 4 schedulers x SM clock x 32 lanes / "
                                       f"{COLLISION_WARP_INSTRUCTIONS:.0f} warp instructions per "
                                       "collision round (ncu source counters)"},
        # SURVEY.md 8d's contract figure: the bytes an EVENT-STEPPED implementation would move
        # (record in and out per event). This design keeps a history in registers for a whole
        # timestep, so those bytes are not moved and `frac` reads above 1: model_bytes is a
        # model, `traffic` is what ncu measured the kernel to move per launch.
        "hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach_gbs / hbm_peak, "peak_source": hbm_src,
                "model_bytes_per_launch": alg_bytes / max(hist_launches, 1),
                "fused_bound_bytes_per_launch": fused_history_bytes(timed) / max(hist_launches, 1),
                "traffic": traffic, "traffic_source": traffic_src,
                "traffic_command": "ncu --set full --clock-control none -k regex:k_history "
                                   "python bench.py --steps 1 --warmup 1 --no-cpu-baseline "
                                   "--no-e2e --no-decks (dram__bytes_read.sum + "
                                   "dram__bytes_write.sum)"},
        "note": "k_history is bound by L2 FP64 atomics (facets) and FP64/INT issue (collisions), "
                "not by HBM (DESIGN.md 5); roofline.hbm carries BASELINE.md 5's HBM figure with "
                "the same keys (bound, achieved, peak, unit, frac, traffic)",
    }
    line = {
        "metric": METRIC, "value": events_all / (elapsed_ms / 1e3), "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(deck, nglobal, world, args.scaling),
        "run": {"parallelism": (f"particle-sharded x{world}: private tally buffers combined by the "
                                f"library's {collective} "
                                + ("once per deck run, when the tally is read"
                                   if reduce_every == 0 else
                                   f"every {reduce_every} timestep(s) beside the next timestep's "
                                   "transport")
                                + ", all-gather into the caller's tally once per deck run")
                if world > 1 else "single GPU",
                "options": args.opts or "defaults (pipeline=1,fast_div=1,tile_shift=8,"
                                        "length_bins=512,step_graph=1)",
                "timesteps_in_flight": 3,
                "events_per_step": events_all / args.steps,
                "tally_sum": tally_sum},
        "roofline": roofline,
        "clocks": clocks,
        "gpu_launches": launches_all,
    }
    if parity is not None:
        line["parity"] = parity
    if e2e:
        line["e2e"] = {"value": e2e_events_all / e2e_seconds, "unit": UNIT,
                       "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                       "ms_per_step": 1e3 * e2e_seconds / args.steps,
                       "history_kernel_ms_per_step": e2e["hist_ms"],
                       "sort_phase_ms_per_step": e2e["sort_ms"],
                       "tally_sum": e2e["tally_sum"], "live_particles_out": e2e_live_all,
                       "pipeline": "double-buffered: upload of step i+1 and download of step "
                                   "i-1 overlap the transport of step i"}
    if e2e:
        try:  # what the e2e loop downloaded last against the resident run of the same deck
            line["e2e"]["tally_matches_resident"] = bool(
                abs(e2e["tally_sum"] - tally_sum) <= 1e-10 * abs(tally_sum))
            line["e2e"]["live_matches_resident"] = bool(e2e_live_all == int(live.item()))
        except Exception:  # (no parity pass, no live count): a reported extra, never a gate
            pass
    stage("other decks")
    if world == 1 and not args.no_decks:
        line["decks"] = time_other_decks(lib, torch, [n for n in OTHER_DECKS if n != deck.name])
    stage("cpu baseline")
    if world == 1 and not args.no_cpu_baseline:
        try:
            res = reference_rate(args.deck, nglobal, budget_seconds=40.0)
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample",
                                                        "full_deck")}
        except Exception as exc:  # the baseline is a reported number, never a gate
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                    "sample": f"unavailable: {exc}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        lib.nb200_mp_finalize()
        dist.destroy_process_group()


def _gather_ragged(dist, torch, mine, parts, sizes, rank):
    """dist.gather needs equal sizes: pad to the largest shard, trim on rank 0."""
    biggest = max(sizes)
    padded = torch.zeros(biggest, dtype=mine.dtype, device="cuda")
    padded[:mine.numel()] = mine
    bufs = [torch.empty(biggest, dtype=mine.dtype, device="cuda") for _ in sizes] \
        if rank == 0 else None
    dist.gather(padded, bufs, dst=0)
    if rank == 0:
        for i, s in enumerate(sizes):
            parts[i] = bufs[i][:s]


def stage(msg: str) -> None:
    """Progress marker on stderr (NB200_BENCH_VERBOSE=1): where a slow run spends its time."""
    if os.environ.get("NB200_BENCH_VERBOSE"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def main():
    args = parse_args()
    if os.environ.get("NB200_BENCH_WATCHDOG"):
        # a run that is still going after that many seconds dumps every thread's stack and exits
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["NB200_BENCH_WATCHDOG"]), exit=True)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        sys.exit("bench.py --gpus N>1 must be launched with torch.distributed.run "
                 "(one process per GPU)")
    run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
