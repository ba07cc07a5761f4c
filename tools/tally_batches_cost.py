"""What option tally_batches costs: csp, split and stream at full size, resident on one GPU and
run with Simulation.run_pipelined, for B in {0, 4, 8, 16, 32} and both layouts of the batch slab
(batch-major, the product; cell-major, built with -DNB_TALLY_BATCH_CELL_MAJOR=1 into a library
of its own). Each (deck, B) restarts from the injected bank, warms up, then times --runs deck
runs with CUDA events: median ms per deck run and events/s. Behind each timed run the flush into
the caller's tally (nb200_tally_sync) and the statistics (nb200_bank_tally_relerr, per cell and
of the total) are timed on the host clock; both calls end in a stream synchronisation.

    python tools/tally_batches_cost.py --out profiles/r03/tally_batches_cost.json

The GPU's name and power limit are written into the same output. Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = {"batch-major": ("", "libneutral_b200.so"),
           "cell-major": ("-DNB_TALLY_BATCH_CELL_MAJOR=1", "libneutral_b200.cellmajor.so")}


def gpu_identity() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (q.stdout.splitlines()[0].split(", ") + ["?"] * 3)[:3]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def worker(args) -> dict:
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch

    from neutral_b200.build import build_library
    from neutral_b200.decks import build_problem
    from neutral_b200.host import DeviceArray, Simulation, _check, _soa_p, load_library

    if args.layout != "batch-major":
        build_library(force=True)  # the variant named by NB200_LIB / NB200_DEFINES
    lib = load_library(build=True)
    if lib.nb200_device_count() <= 0:
        raise SystemExit("tally_batches_cost.py needs a CUDA device")
    out = {}
    for deck in args.decks:
        prob = build_problem(deck)
        ref_sim = Simulation(prob, per_particle_counters=False)
        ref_sim.inject()
        injected = ref_sim.bank_to_host()
        ref_sim.free()
        st = injected.as_struct()
        snap = _soa_p()
        _check(lib.nb200_bank_create(C.byref(st), len(injected), 0, C.byref(snap)), "snapshot")
        for B in args.batches:
            sim = Simulation(prob, per_particle_counters=False, tally_batches=B)
            sim.inject()
            relerr = DeviceArray(prob.deck.nx * prob.deck.ny)
            total = C.c_double()
            ms, flush_ms, stats_ms, events = [], [], [], []
            for i in range(args.warmup + args.runs):
                _check(lib.nb200_bank_copy(sim.bank, snap), "bank_copy")
                sim.tally.zero()
                torch.cuda.synchronize()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                res = sim.run_pipelined()
                ev1.record()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sim.tally_sync()
                t1 = time.perf_counter()
                if B:
                    _check(lib.nb200_bank_tally_relerr(sim.bank, C.c_void_p(relerr.ptr),
                                                       C.byref(total)), "relerr")
                t2 = time.perf_counter()
                if i >= args.warmup:
                    ms.append(ev0.elapsed_time(ev1))
                    events.append(sum(r.events for r in res))
                    flush_ms.append((t1 - t0) * 1e3)
                    stats_ms.append((t2 - t1) * 1e3)
            med = statistics.median(ms)
            row = {"ms_per_deck_run": med, "ms_min": min(ms), "ms_max": max(ms),
                   "events_per_s": statistics.median(events) / (med / 1e3), "runs": len(ms),
                   "tally_total": float(np.sum(sim.tally_to_host()))}
            if B:
                row.update(flush_ms=statistics.median(flush_ms),
                           statistics_ms=statistics.median(stats_ms),
                           total_relative_error=total.value)
            out[f"{deck}/B={B}"] = row
            print(args.layout, deck, B, json.dumps(row), flush=True)
            relerr.free()
            sim.free()
        lib.nb200_bank_free(snap)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--decks", nargs="+", default=["csp", "split", "stream"])
    ap.add_argument("--batches", nargs="+", type=int, default=[0, 4, 8, 16, 32])
    ap.add_argument("--layouts", nargs="+", default=list(LAYOUTS), choices=list(LAYOUTS))
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="JSON file for the results")
    ap.add_argument("--layout", default=None, help=argparse.SUPPRESS)  # worker process
    ap.add_argument("--worker-out", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.layout:
        with open(args.worker_out, "w") as f:
            json.dump(worker(args), f)
        return
    result = {"what": "ms per resident deck run (run_pipelined, CUDA events, median), events/s, "
                      "flush and statistics ms (host clock, median)",
              **gpu_identity(), "runs": args.runs, "warmup": args.warmup, "layouts": {}}
    for layout in args.layouts:
        defines, lib = LAYOUTS[layout]
        env = dict(os.environ, NB200_DEFINES=defines, NB200_LIB=lib)
        fd, tmp = tempfile.mkstemp(suffix=".json")
        os.close(fd)
        cmd = [sys.executable, os.path.abspath(__file__), "--layout", layout, "--worker-out", tmp,
               "--runs", str(args.runs), "--warmup", str(args.warmup), "--decks", *args.decks,
               "--batches", *map(str, args.batches)]
        subprocess.run(cmd, env=env, check=True)
        with open(tmp) as f:
            result["layouts"][layout] = json.load(f)
        os.remove(tmp)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
