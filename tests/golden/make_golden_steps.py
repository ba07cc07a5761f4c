#!/usr/bin/env python3
"""Generates the step-by-step reference vectors the reference-parity tests compare against, so
that they run without the reference library:

    OMP_NUM_THREADS=8 python tests/golden/make_golden_steps.py   # ~5 CPU-minutes on 8 cores

* ``steps.json``: per problem, sha256 of every particle field after injection and after every
  timestep, the per-timestep (facets, collisions) and the tally's sum after every timestep - for the small decks, the variants of
  tests/variants.py and the 50 000-particle banks of test_device_inject_equals_host_inject;
* ``tally_samples.npz``: the final tally of every variant and of the full csp and split decks
  on a fixed, seeded sample of its non-zero cells, with its sum and its number of non-zero
  cells.

The vectors come from the unmodified reference omp3 library (oracle/_ref) where it is built,
else from the oracle port, which reproduces it bit for bit: the script then checks every
particle state, count and tally it can against the vectors recorded from the reference library
itself (tests/golden/<deck>.npz, tests/golden/full_decks.json) and refuses to write on any
difference.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from neutral_b200.bank import ALL_FIELDS, HostBank  # noqa: E402
from neutral_b200.decks import build_problem  # noqa: E402
from oracle.oracle import OraclePort, ReferenceOmp3  # noqa: E402
from variants import VARIANTS  # noqa: E402

SMALL_DECKS = ["csp_small", "split_small", "scatter_small", "stream_small", "mixed_small"]
INJECT_ONLY = {"csp_small@50000": ("csp_small", 50_000), "split_small@50000": ("split_small", 50_000)}
FULL_DECKS = ["csp", "split"]
TALLY_SAMPLE = 1024


def field_hashes(bank: HostBank):
    return [hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
            for k in ALL_FIELDS]


def tally_sample(out, name, tally):
    nonzero = np.flatnonzero(tally)
    pick = np.random.default_rng(0).choice(nonzero.size, min(TALLY_SAMPLE, nonzero.size),
                                           replace=False)
    cells = np.sort(nonzero[pick])
    out[f"{name}_cells"] = cells.astype(np.int32)
    out[f"{name}_tally"] = tally[cells]
    out[f"{name}_sum"] = np.float64(tally.sum())
    out[f"{name}_nonzero"] = np.int64(nonzero.size)


def close(a, b, rtol):
    return bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b))))


class Engine:
    """The reference library when built, else the oracle port, behind one bank type."""

    def __init__(self):
        self.ref = ReferenceOmp3() if ReferenceOmp3.available() else None
        self.port = OraclePort()
        self.source = "reference omp3 library" if self.ref else "oracle port"

    def inject(self, prob):
        return self.ref.inject(prob) if self.ref else self.port.inject(prob)

    def step(self, prob, bank, tt, tally):
        if self.ref:
            return self.ref.step(prob, bank, tt, tally)
        return self.port.step(prob, bank, tt, tally)[:2]

    def host(self, bank):
        return HostBank.from_aos(bank) if self.ref else bank


def run(eng, prob, quiet=False):
    d = prob.deck
    bank = eng.inject(prob)
    hashes = [field_hashes(eng.host(bank))]
    tally = np.zeros(d.nx * d.ny)
    counts, sums = [], []
    devnull, saved = os.open(os.devnull, os.O_WRONLY), os.dup(1)
    if quiet:
        os.dup2(devnull, 1)  # the reference prints "Particles N" every timestep
    try:
        for tt in range(1, d.iterations + 1):
            counts.append([int(x) for x in eng.step(prob, bank, tt, tally)])
            hashes.append(field_hashes(eng.host(bank)))
            sums.append(float(tally.sum()))
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)
    return {"counts": counts, "hashes": hashes, "tally_sums": sums}, tally, eng.host(bank)


def main():
    eng = Engine()
    steps = {"source": eng.source}
    for name in SMALL_DECKS:
        rec, tally, _ = run(eng, build_problem(name))
        g = np.load(os.path.join(HERE, f"{name}.npz"))
        assert np.array_equal(np.array(rec["counts"], dtype=np.uint64), g["counts"][:, :2]), name
        assert rec["hashes"][0] == list(g["inject_hashes"]), name
        assert rec["hashes"][1] == list(g["step1_hashes"]), name
        assert rec["hashes"][-1] == list(g["final_hashes"]), name
        assert close(tally, g["tally"], 1e-12), name
        steps[name] = rec
    sample = {}
    for name, make in VARIANTS.items():
        steps[name], tally, _ = run(eng, make())
        tally_sample(sample, name, tally)
    for key, (base, n) in INJECT_ONLY.items():
        steps[key] = {"hashes": [field_hashes(eng.host(eng.inject(build_problem(base, nparticles=n))))]}
    full = json.load(open(os.path.join(HERE, "full_decks.json")))
    for name in FULL_DECKS:
        prob = build_problem(name)
        d = prob.deck
        rec, tally, bank = run(eng, prob, quiet=True)
        g = full[name]
        assert rec["counts"] == g["counts"], name
        assert dict(zip(ALL_FIELDS, rec["hashes"][-1])) == g["final_hashes"], name
        t = tally.reshape(d.ny, d.nx)
        img = t[:d.ny // 64 * 64, :d.nx // 64 * 64].reshape(64, d.ny // 64, 64, d.nx // 64)
        assert close(img.sum(axis=(1, 3)).ravel(), np.array(g["tally_block_sums"]), 1e-10), name
        tally_sample(sample, name, tally)
    with open(os.path.join(HERE, "steps.json"), "w") as f:
        json.dump(steps, f, indent=0)
    np.savez_compressed(os.path.join(HERE, "tally_samples.npz"), **sample)
    print(f"recorded from the {eng.source}")


if __name__ == "__main__":
    main()
