"""Persistent-evaluator throughput with host arrays against CUDA tensors: `evaluate_targets` (numpy in, numpy out)
against `evaluate_targets_cuda` (torch CUDA tensor in and out, no host round trip) on two fitted models:
  - "latency": the tools/evaluator_latency.py model (N = 200 000 uniform points, linear kernel, evaluator on [0, 1]^3);
  - "c4": the BASELINE.json C4 model (albatite signed-distance points, cubic kernel, linear drift).
Batches: 10^3 and 10^5 random targets in the evaluator box, and the 256^3 grid over it (16.7 M targets; for C4 the
grid of tools/c4_albatite.py), the grid built with torch on the device.  Each timing is a host clock around a call
that ends in torch.cuda.synchronize(), after warm-up; the median of the repeats is reported, with the card's name
and power limit read in the same run.

    python tools/device_eval_bench.py [--grid 256] [--out result.json]
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import ferreus_rbf_rs_b200 as fb  # noqa: E402


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": line}


def median_s(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def grid_cuda(lo, hi, g):
    """g^3 nodes over [lo, hi], x fastest (tools/c4_albatite.py), built on the device"""
    import torch
    ax = [torch.linspace(float(lo[k]), float(hi[k]), g, dtype=torch.float64, device="cuda") for k in range(3)]
    zz, yy, xx = torch.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
    return torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], dim=1).contiguous()


def bench_model(name, model, lo, hi, g):
    import torch
    rng = np.random.default_rng(7)
    rows = []
    for label, m in (("1e3", 1000), ("1e5", 100_000), (f"grid{g}^3", g ** 3)):
        if m == g ** 3:
            x = grid_cuda(lo, hi, g)
            xh = x.cpu().numpy()
        else:
            xh = np.ascontiguousarray(rng.random((m, 3)) * (hi - lo) + lo)
            x = torch.as_tensor(xh, device="cuda")
        reps, warm = (10, 3) if m <= 100_000 else (3, 1)
        if m <= 1000:
            reps = 50
        host_s, host_all = median_s(lambda: model.evaluate_targets(xh), reps, warm)
        dev_s, dev_all = median_s(lambda: model.evaluate_targets_cuda(x), reps, warm)
        vh = np.asarray(model.evaluate_targets(xh))
        vd = model.evaluate_targets_cuda(x).cpu().numpy()
        rows.append({"model": name, "batch": label, "targets": m,
                     "evaluate_targets_median_ms": host_s * 1e3, "evaluate_targets_cuda_median_ms": dev_s * 1e3,
                     "host_over_device": host_s / dev_s,
                     "evaluate_targets_ms_all": [t * 1e3 for t in host_all],
                     "evaluate_targets_cuda_ms_all": [t * 1e3 for t in dev_all],
                     "device_vs_host_rel_l2": float(np.linalg.norm(vd - vh) / np.linalg.norm(vh))})
        del x, xh
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    ic = fb.interpolant_config
    rows = []
    # latency model (tools/evaluator_latency.py)
    rng = np.random.default_rng(0)
    pts = rng.random((200_000, 3))
    vals = np.sin(4 * pts[:, 0]) * np.cos(3 * pts[:, 1]) + pts[:, 2]
    model = fb.RBFInterpolator(pts, vals, ic.InterpolantSettings(ic.RBFKernelType.Linear))
    model.build_evaluator([0.0, 0.0, 0.0, 1.0, 1.0, 1.0])
    rows += bench_model("latency", model, np.zeros(3), np.ones(3), a.grid)
    del model
    # C4 (tools/c4_albatite.py)
    d = np.load("tests/golden/albatite_SD_points.npz")
    model = fb.RBFInterpolator(d["points"], d["values"], ic.InterpolantSettings(ic.RBFKernelType.Cubic))
    lo, hi = np.floor(d["points"].min(0)), np.ceil(d["points"].max(0))
    model.build_evaluator(list(lo) + list(hi))
    rows += bench_model("c4", model, lo, hi, a.grid)
    out = {"card": card(), "timing": "host clock around call + torch.cuda.synchronize(), median after warm-up",
           "results": rows}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
