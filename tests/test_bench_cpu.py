"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port on the host cores at the workload's full
size -- here cut down with the development switch --n) prints one JSON line with the expected keys; argument checks;
the writer behind --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _run(kind, extra=()):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--n", "1536", "--ref-kind", kind, *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_reference_arm_prints_contract_line():
    line = _run("port")
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "s" and line["higher_is_better"] is False
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "sample" in line["cpu_baseline"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]
    assert line["steps_run"] == 1 and line["config"]["N"] == 1536
    assert len(line["config"]["labels_sha256"]) == 64 and "scal" not in line["cpu_baseline"]["sample"].replace("no scaling", "")
    # thread pinning does not depend on what the launcher exported (torchrun sets OMP_NUM_THREADS=1)
    assert line["cpu_baseline"]["threads"]["blas"] == os.cpu_count()


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--n", "512"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_rejected_arguments():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=600, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, extra


def test_dump_outputs_types_sample_and_limit(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    big = rng.standard_normal((bench.DUMP_ARRAY_BYTES // (4 * 64) + 1000, 64)).astype(np.float32)
    arrays = {"labels": np.arange(-1, 99, dtype=np.int64), "core": np.ones(100, np.uint8), "count": np.int64(7),
              "keys": big, "half": np.ones((3, 2), np.float16), "wide": np.zeros(5, np.float64)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(["labels.npy", "core.npy", "count.npy", "keys.npy", "keys_rows.npy", "half.npy", "wide.npy"])
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    d = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert np.array_equal(d["labels"], np.arange(-1, 99)) and d["labels"].dtype == np.float64
    assert d["count"].tolist() == [7.0] and d["half"].dtype == np.float32 and d["wide"].dtype == np.float64
    rows = d["keys_rows"].astype(np.int64)
    assert d["keys"].nbytes + d["keys_rows"].nbytes <= bench.DUMP_ARRAY_BYTES and np.all(np.diff(rows) > 0)
    assert np.array_equal(d["keys"], big[rows])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
