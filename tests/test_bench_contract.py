"""The bench.py contract. Without a GPU: the reference arm (`--impl reference`) prints ONE JSON
line with the keys the driver reads, times the CPU checker with the threads it reports - also
when the launcher exported OMP_NUM_THREADS=1, as torchrun does - and the b200 arm refuses to
run N > 1 outside torchrun or without a timed step. On the GPU: `--steps` timed runs, and
`--dump-outputs` writes what the last of them computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT,
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_line():
    res = _run(["--impl", "reference", "--deck", "csp_small", "--steps", "1", "--warmup", "0"],
               {"OMP_NUM_THREADS": "1", "NB200_REF_THREADS": "2"})
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "particle_events_per_sec"
    assert d["unit"] == "events/s" and d["higher_is_better"] is True and d["value"] > 0
    for key in ("n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["dtype"] == "f64" and d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 2 and cb["value"] == d["value"]
    assert "OMP threads=2" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    res = _run(["--impl", "reference", "--deck", "csp_small", "--steps", "1", "--warmup", "0"],
               {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_multi_gpu_needs_torchrun():
    res = _run(["--gpus", "2", "--steps", "1", "--warmup", "0"])
    assert res.returncode != 0 and "torch.distributed.run" in (res.stderr + res.stdout)


def test_steps_must_be_positive():
    res = _run(["--steps", "0"])
    assert res.returncode != 0 and "--steps" in res.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_run(tmp_path):
    """Two timed runs of csp_small: the dumped counts, bank and tally are the reference run's
    (tests/golden/csp_small.npz), in float64, well under 64 MB."""
    out = tmp_path / "dump"
    res = _run(["--deck", "csp_small", "--steps", "2", "--warmup", "1", "--no-e2e", "--no-decks",
                "--no-cpu-baseline", "--dump-outputs", str(out)])
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["roofline"]["launches_timed"] == 2 * 10
    g = np.load(os.path.join(ROOT, "tests", "golden", "csp_small.npz"))
    files = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert all(a.dtype == np.float64 for a in files.values())
    assert sum(p.stat().st_size for p in out.glob("*.npy")) <= 64 << 20
    assert np.array_equal(files["counts"][:, :3], g["counts"].astype(np.float64))
    assert np.array_equal(files["bank_sample_index"][:256], np.arange(256))
    for k in g["sample"].dtype.names:
        assert np.array_equal(files[f"bank_{k}"][:256], g["sample"][k].astype(np.float64)), k
    t, got = g["tally"], files["tally_sample"]
    assert np.array_equal(files["tally_sample_index"], np.arange(t.size))
    assert np.all(np.abs(got - t) <= 1e-10 * np.maximum(np.abs(got), np.abs(t)))
    assert abs(files["tally_block_sums"].sum() - t.sum()) <= 1e-10 * t.sum()
