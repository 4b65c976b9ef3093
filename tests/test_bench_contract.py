"""CPU: the `bench.py --impl reference` arm (the oracle port timed on host cores) prints ONE JSON line carrying the keys
of the bench line and times exactly --steps steps; `--dump-outputs` stays within its size limit.  The GPU arm needs a B200
(tests/test_gpu_bench.py)."""
import json
import os
import subprocess
import sys

from _util import ROOT


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("tasks/sec") and d["unit"] == "tasks/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"] == "convcnp1d_b256_c128_t128" and d["data"] == "synthetic" and d["vs_baseline"] is None
    cb, e2e = d["cpu_baseline"], d["e2e"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"].startswith("2 steps")
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_dump_outputs_samples_down_to_the_size_limit(tmp_path):
    import numpy as np
    import bench
    big = np.arange(40000, dtype=np.float64).reshape(200, 200)
    outs = {"loss": np.float32(1.5), "grad.b": np.arange(100, dtype=np.float32), "grad.w": big}
    limit = 20000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs, limit_bytes=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["grad.b.npy", "grad.w.npy", "loss.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["loss.npy"].shape == () and got["loss.npy"] == 1.5 and np.array_equal(got["grad.b.npy"], outs["grad.b"])   # small: whole
    w = got["grad.w.npy"]
    assert 4000 < w.size < big.size and (np.diff(w) > 0).all() and np.isin(w, big).all()      # distinct entries in index order
    assert all(np.array_equal(got[f], np.load(tmp_path / "b" / f)) for f in files)             # the same sample every run
    bench.dump_outputs(str(tmp_path / "c"), outs)                                               # under the limit: whole arrays
    assert np.array_equal(np.load(tmp_path / "c" / "grad.w.npy"), big.astype(np.float32))
