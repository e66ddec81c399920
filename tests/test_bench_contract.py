"""bench.py's command line: the reference arm (`--impl reference`, no GPU) prints one JSON line with the contract keys;
`--dump-outputs` writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _util import ROOT


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "samples/s" and d["n_gpus"] == 1
    assert d["metric"].startswith("train samples/sec") and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("cfg5") and d["config"]["rows"] > 30_000_000 and d["config"]["batch_per_gpu"] == 8192
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # a non-zero rank of a torchrun launch exits 0 without output
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         env=dict(env, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2"), capture_output=True, text=True, timeout=300,
                         cwd=ROOT)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_repeat_for_the_same_arguments(tmp_path):
    """--dump-outputs writes the last timed step's outputs (float32 / float64, 64 MB at most): its rows are the rows of the
    last timed batch, the same arguments give the same files, and one more timed step changes exactly the rows its batch
    hits."""
    import bench
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    # run_ours' schedule: 16 rotating batches (seed 1234 on rank 0), max(warm-up, 3, 2 * 16 + 2) untimed steps, then the
    # timed ones; the last timed step of a K-step run is step 34 + K - 1
    sizes = bench.feature_sizes("cfg4")
    batches = bench.synth_batches(sizes, 8192, 16, 1234)
    offsets = np.concatenate([[0], np.cumsum(sizes)])[:-1]
    last_rows = lambda steps: np.unique(batches[(34 + steps - 1) % 16][0] + offsets[None, :])
    dumps = {}
    for run, steps in (("a", 3), ("b", 3), ("c", 4)):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg4", "--steps", str(steps),
                              "--warmup", "1", "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path / run)],
                             env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == steps
        dumps[run] = {f[:-4]: np.load(tmp_path / run / f) for f in sorted(os.listdir(tmp_path / run))}
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert sorted(a) == ["bias", "loss", "sample_row_ids", "sample_rows", "updated_row_ids", "updated_rows"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["updated_rows"].shape == (len(a["updated_row_ids"]), 11) and np.isfinite(a["loss"]).all()
    assert np.array_equal(a["updated_row_ids"], last_rows(3)) and np.array_equal(c["updated_row_ids"], last_rows(4))
    assert sorted(b) == sorted(a) and all(np.array_equal(a[n], b[n]) for n in a)
    assert not np.array_equal(a["loss"], c["loss"])
    assert np.array_equal(a["sample_row_ids"], c["sample_row_ids"])
    hit = np.isin(a["sample_row_ids"], last_rows(4))
    assert np.array_equal(a["sample_rows"][~hit], c["sample_rows"][~hit])
    assert hit.any() and not np.array_equal(a["sample_rows"][hit], c["sample_rows"][hit])
