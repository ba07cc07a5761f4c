"""The reference omp3 runs recorded step by step (test infrastructure): what the reference-parity
tests compare against, written by tests/golden/make_golden_steps.py."""
from __future__ import annotations

import hashlib
import json
import os
from functools import lru_cache

import numpy as np

from neutral_b200.bank import ALL_FIELDS

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def field_hashes(bank):
    """sha256 of each of the 11 particle fields, in ALL_FIELDS order."""
    return [hashlib.sha256(np.ascontiguousarray(bank.arrays[k]).tobytes()).hexdigest()
            for k in ALL_FIELDS]


@lru_cache(maxsize=None)
def _steps():
    with open(os.path.join(GOLDEN, "steps.json")) as f:
        return json.load(f)


def reference_run(name: str) -> dict:
    """``counts``: per-timestep [facets, collisions]; ``hashes``: field_hashes of the bank after
    injection (index 0) and after every timestep."""
    return _steps()[name]


def reference_tally_sample(name: str):
    """(cells, values, sum, number of non-zero cells) of the final tally: a fixed, seeded sample
    of its non-zero cells."""
    with np.load(os.path.join(GOLDEN, "tally_samples.npz")) as g:
        return (g[f"{name}_cells"], g[f"{name}_tally"], float(g[f"{name}_sum"]),
                int(g[f"{name}_nonzero"]))


def tally_matches_sample(tally, name: str, rtol: float) -> bool:
    """The sampled cells within rtol, the same non-zero cell count, the sum within rtol."""
    cells, want, total, nonzero = reference_tally_sample(name)
    got = tally[cells]
    return bool(np.all(np.abs(got - want) <= rtol * np.maximum(np.abs(got), np.abs(want)))
                and np.count_nonzero(tally) == nonzero
                and abs(float(tally.sum()) - total) <= rtol * abs(total))
