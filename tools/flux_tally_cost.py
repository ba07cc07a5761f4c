"""What the track-length flux tally costs: csp, split, stream and scatter at full size, resident on
one GPU and run with Simulation.run_pipelined, without and with a flux array attached
(nb200_bank_set_flux_tally). The two configurations alternate run by run in the same process:
each deck run restarts both banks from the same injected snapshot, and after --warmup warm-up
runs of each the next --runs are timed with CUDA events. Reported: median ms per deck run and
events/s of each, their ratio, and the tally and flux totals (the tally totals of the two must
agree to summation order).

With --tally-batches B both banks have B tally batches (option tally_batches), and the flux of
the second is batched too (nb200_bank_set_batched_flux_tally): what the flux batches cost on top
of the energy batches.

With --groups G [G ...] each G adds one more configuration to the alternation: a group flux
(nb200_bank_set_group_flux_tally) over G logarithmic energy groups from 1e-3 eV to twice the
deck's initial energy, which cover every energy the deck reaches. Its rows carry the flux summed
over the groups, and their ratio to the run without flux. With --tally-batches B as well, every
bank of the alternation is batched: no flux, a batched plain flux, and one batched group flux per
G (nb200_bank_set_batched_group_flux_tally), whose slab holds (B + 1) * G * ncells doubles.

    python tools/flux_tally_cost.py --out profiles/r04/flux_tally_cost.json
    python tools/flux_tally_cost.py --tally-batches 16 --out flux_batches_cost_b16.json
    python tools/flux_tally_cost.py --groups 8 32 --out profiles/r05/group_flux_cost.json
    python tools/flux_tally_cost.py --tally-batches 16 --groups 8 --out batched_group_b16.json

The GPU's name and power limit are written into the same output. Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tally_batches_cost import gpu_identity  # noqa: E402  (tools/ is the script's directory)


def measure(args) -> dict:
    import numpy as np
    import torch

    from neutral_b200.decks import build_problem
    from neutral_b200.host import Simulation, _check, _soa_p, load_library

    lib = load_library(build=True)
    if lib.nb200_device_count() <= 0:
        raise SystemExit("flux_tally_cost.py needs a CUDA device")
    out = {}
    for deck in args.decks:
        prob = build_problem(deck)
        e0 = prob.deck.initial_energy
        sims = {flux: Simulation(prob, per_particle_counters=False, flux_tally=flux,
                                 tally_batches=args.tally_batches)
                for flux in (False, True)}
        for g in args.groups:
            sims[f"groups_{g}"] = Simulation(prob, per_particle_counters=False,
                                             flux_groups=np.geomspace(1.0e-3, 2.0 * e0, g + 1),
                                             tally_batches=args.tally_batches,
                                             group_flux_batches=args.tally_batches > 0)
        for sim in sims.values():
            sim.inject()
        injected = sims[False].bank_to_host()
        st = injected.as_struct()
        snap = _soa_p()
        _check(lib.nb200_bank_create(C.byref(st), len(injected), 0, C.byref(snap)), "snapshot")
        ms = {k: [] for k in sims}
        events = {k: [] for k in sims}
        for i in range(args.warmup + args.runs):
            for flux, sim in sims.items():
                _check(lib.nb200_bank_copy(sim.bank, snap), "bank_copy")
                sim.tally.zero()
                if flux:
                    sim.flux.zero()
                torch.cuda.synchronize()
                ev0 = torch.cuda.Event(enable_timing=True)
                ev1 = torch.cuda.Event(enable_timing=True)
                ev0.record()
                res = sim.run_pipelined()
                ev1.record()
                torch.cuda.synchronize()
                if i >= args.warmup:
                    ms[flux].append(ev0.elapsed_time(ev1))
                    events[flux].append(sum(r.events for r in res))
        row = {}
        for flux, sim in sims.items():
            med = statistics.median(ms[flux])
            name = flux if isinstance(flux, str) else "flux" if flux else "no_flux"
            row[name] = {
                "ms_per_deck_run": med, "ms_min": min(ms[flux]), "ms_max": max(ms[flux]),
                "events_per_s": statistics.median(events[flux]) / (med / 1e3),
                "runs": len(ms[flux]), "tally_total": float(np.sum(sim.tally_to_host()))}
            if flux is True:
                row[name]["flux_total"] = float(np.sum(sim.flux_to_host()))
            elif flux:
                row[name]["flux_total"] = float(np.sum(sim.group_flux_to_host()))
                row[name]["ratio"] = med / statistics.median(ms[False])
        row["ratio"] = row["flux"]["ms_per_deck_run"] / row["no_flux"]["ms_per_deck_run"]
        out[deck] = row
        print(deck, json.dumps(row), flush=True)
        lib.nb200_bank_free(snap)
        for sim in sims.values():
            sim.free()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--decks", nargs="+", default=["csp", "split", "stream", "scatter"])
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--tally-batches", type=int, default=0,
                    help="B > 0: both banks batched, the flux of the second batched too")
    ap.add_argument("--groups", type=int, nargs="*", default=[],
                    help="G ...: one more configuration per G, a group flux over G log groups "
                         "(batched with --tally-batches)")
    ap.add_argument("--out", default=None, help="JSON file for the results")
    args = ap.parse_args()
    result = {"what": "ms per resident deck run (run_pipelined, CUDA events, median) without "
                      "and with a flux array attached (plain, and a group flux per --groups G), "
                      "alternating run by run; events/s",
              **gpu_identity(), "runs": args.runs, "warmup": args.warmup,
              "tally_batches": args.tally_batches, "groups": args.groups,
              "decks": measure(args)}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
