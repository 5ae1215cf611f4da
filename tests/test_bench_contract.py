"""bench.py's reference arm runs without a GPU (it times the oracle port on the host cores): its one JSON line must carry
the keys the driver reads, on the same metric / unit / config shape as the CUDA arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "20000",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "bbfmm_matvec_throughput" and d["unit"] == "Mpts/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1
    assert d["config"]["points"] == 20000 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--n",
                          "20000", "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_times_the_requested_steps_and_dumps_its_result(tmp_path):
    from oracle import kernels as ok
    n = 5000
    d = _bench("--impl", "reference", "--n", str(n), "--steps", "3", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 3 and len(d["cpu_baseline"]["step_seconds"]) == 3
    assert sorted(os.listdir(tmp_path)) == ["matvec.npy"]
    got = np.load(tmp_path / "matvec.npy")
    assert got.dtype == np.float64 and got.shape == (n, 1)
    rng = np.random.default_rng(1000)  # bench.make_workload(n, 1000)
    pts, w = rng.random((n, 3)), rng.random((n, 1))
    dense = ok.dense_matvec(ok.Kernel(ok.LINEAR), pts, pts, w)
    assert np.linalg.norm(got - dense) / np.linalg.norm(dense) <= 1e-5


def test_dump_outputs_keeps_the_same_sampled_rows_under_the_size_cap(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 8000)
    a = np.arange(2000, dtype=np.float64).reshape(1000, 2)
    bench.dump_outputs(str(tmp_path), {"a": a, "b": -a.astype(np.float32)})
    ga, gb = np.load(tmp_path / "a.npy"), np.load(tmp_path / "b.npy")
    assert ga.dtype == gb.dtype == np.float64 and ga.nbytes + gb.nbytes <= 8000 and ga.shape == (250, 2)
    assert np.array_equal(gb, -ga) and np.all(np.diff(ga[:, 0]) > 0) and np.array_equal(ga[:, 1], ga[:, 0] + 1)
    bench.dump_outputs(str(tmp_path), {"a": a, "b": -a})
    assert np.array_equal(np.load(tmp_path / "a.npy"), ga)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_step_of_each_timed_path(tmp_path):
    """The CUDA arm and the reference arm dump matvec.npy for the same seeded workload; they agree to the FMM parity
    bar.  The third e2e step evaluates the original weights again, so e2e.npy equals the resident result."""
    n = 20000
    ours, ref = tmp_path / "ours", tmp_path / "ref"
    d = _bench("--n", str(n), "--steps", "3", "--warmup", "3", "--no-fit", "--no-cpu-baseline", "--dump-outputs",
               str(ours))
    assert d["steps"] == 3
    _bench("--impl", "reference", "--n", str(n), "--steps", "1", "--warmup", "0", "--dump-outputs", str(ref))
    assert sorted(os.listdir(ours)) == ["e2e.npy", "matvec.npy", "matvec_sqrt_exact.npy"]
    got = {k: np.load(ours / (k + ".npy")) for k in ("matvec", "matvec_sqrt_exact", "e2e")}
    want = np.load(ref / "matvec.npy").reshape(n)  # the oracle port returns (n, 1)
    rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))
    for a in got.values():
        assert a.dtype == np.float64 and a.shape == (n,)  # one column comes back 1-D, as from FmmTree.evaluate
    assert rel(got["matvec"], want) <= 1e-10
    assert rel(got["matvec_sqrt_exact"], want) <= 1e-10
    assert rel(got["e2e"], got["matvec"]) <= 1e-12
