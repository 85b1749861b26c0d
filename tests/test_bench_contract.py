"""bench.py's reference arm runs on the CPU (it times the oracle port of the reference's algorithm): its ONE JSON line must carry
the same keys as the GPU arm's line, so that the two can be compared (same metric, unit and direction). --dump-outputs writes
the last timed step's results, bounded in size and the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "impl", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "leaf_candidates_scored_per_sec" and d["unit"] == "candidates/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["gpu_launches"] == 0 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "extrapolation" in d["cpu_baseline"] and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # other ranks of a torchrun launch print nothing and exit 0
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_writes_a_bounded_seeded_sample(tmp_path):
    """bench.dump_outputs: float32 stays float32, integers become exact float64; above the byte limit every array keeps the
    same seeded sample of rows, and the sample's row indices are written too."""
    import bench
    rng = np.random.RandomState(0)
    arrays = dict(idx=rng.randint(0, 50, size=1000).astype(np.int32), feat=rng.standard_normal((1000, 64)).astype(np.float32))
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["feat.npy", "idx.npy"]
    idx, feat = np.load(tmp_path / "all" / "idx.npy"), np.load(tmp_path / "all" / "feat.npy")
    assert idx.dtype == np.float64 and np.array_equal(idx, arrays["idx"]) and feat.dtype == np.float32 and np.array_equal(feat, arrays["feat"])
    limit = 100 * 1024
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["feat.npy", "idx.npy", "rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit + 3 * 128        # + the .npy headers
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "feat.npy"), arrays["feat"][rows])
    assert np.array_equal(np.load(tmp_path / "a" / "idx.npy"), arrays["idx"][rows])
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_are_identical(tmp_path):
    """bench.py --dump-outputs: the last timed step's winners and features, the same in two runs with the same arguments, and
    --steps is the number of timed steps the line reports."""
    outs = []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--batch", "16", "--rho", "20",
                              "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-library-baseline", "--no-train-step",
                              "--no-dense77", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 3 and line["value"] > 0
        assert sorted(os.listdir(d)) == ["best_character.npy", "best_features.npy", "best_position.npy"]
        outs.append({f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)})
    a, b = outs
    assert a["best_position"].shape == a["best_character"].shape == (16,) and a["best_features"].shape == (16, 64)
    assert a["best_position"].dtype == np.float64 and a["best_features"].dtype == np.float32
    assert ((a["best_position"] >= 0) & (a["best_position"] < 20)).all() and np.isfinite(a["best_features"]).all()
    for f in a:
        assert np.array_equal(a[f], b[f]), f
