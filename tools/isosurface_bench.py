"""Isosurface extraction (RBFInterpolator.extract_isosurfaces_cuda over fr_isosurface_extract) on two fitted models:
  - "latency": the tools/evaluator_latency.py model (N = 200 000 uniform points, linear kernel) on [0, 1]^3, isovalue
    0.5;
  - "c4": the BASELINE.json C4 model (albatite signed-distance points, cubic kernel, linear drift) on the box of
    tools/c4_albatite.py, isovalue 0 (the geological boundary).
at 128^3 and 256^3 lattices.  Reported per case: the stage times of fr_isosurface_timing (lattice evaluation with its
tree, extraction, refinement, normals) and a host clock around the synchronous call (median of the repeats after a
warm-up), vertex / face counts, mean and maximum refinement iterations, max |f(v) - iso| by the one-shot evaluate_cuda
at the refined and the unrefined vertices, the algorithmic bytes of the extraction passes and the device memory the
call leaves in the allocation cache (emptied before).  The card's name and power limit are read in the same run.

    python tools/isosurface_bench.py [--grids 128 256] [--reps 3] [--out profiles/r4_isosurface_bench.json]
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


def extraction_bytes(nodes, cubes, nv, nf):
    """compulsory DRAM traffic of the extraction passes: crossing masks (8 B value read, 1 B mask written), node scan
    (1 B in, 8 B out), cube counts (1 B classes in, 1 B count out), cube scan (1 B in, 8 B out), vertices (mask, and per
    vertex the node base, both end values, 24 B position and 8 B edge id written), triangles (classes and face base per
    cube, per face 24 B written and three vertex look-ups of 8 B base + 1 B mask)"""
    return int(nodes * (8 + 1 + 1 + 8 + 1) + cubes * (1 + 1 + 1 + 8) + nodes * (1 + 8) + nv * (8 + 16 + 24 + 8)
               + cubes * (1 + 8) + nf * (24 + 3 * 9))


def bench_case(name, model, ext, g, iso, reps):
    import torch
    res = (g, g, g)
    lib = fb._lib.lib()
    torch.cuda.synchronize()
    lib.fb_trim_memory()
    free0 = torch.cuda.mem_get_info()[0]
    model._isosurfaces([iso], ext, 32, 0, True, torch.device("cuda"))     # warm-up: module loads, first launches
    walls, runs = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        meshes, stats = model._isosurfaces([iso], ext, res, 0, True, torch.device("cuda"))
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
        runs.append(stats)
    held = free0 - torch.cuda.mem_get_info()[0]
    k = int(np.argsort(walls)[len(walls) // 2])
    v, f, n = meshes[0]
    nv, nf = v.shape[0], f.shape[0]
    ev, iters = runs[k]["refine"][0]
    v0, f0, _ = model._isosurfaces([iso], ext, res, 0, False, torch.device("cuda"))[0][0]
    r = (model.evaluate_cuda(v) - iso).abs().max().item() if nv else 0.0
    r0 = (model.evaluate_cuda(v0) - iso).abs().max().item() if nv else 0.0
    nodes, cubes = g ** 3, (g - 1) ** 3
    ms = runs[k]["ms"]
    return {"model": name, "lattice": list(res), "isovalue": iso, "extents": [float(x) for x in ext],
            "stage_ms": {"lattice_eval": ms[0], "extraction": ms[1], "refinement": ms[2], "normals": ms[3]},
            "stage_ms_all": [r_["ms"] for r_ in runs],
            "wall_ms_median": walls[k], "wall_ms_all": walls,
            "vertices": nv, "faces": nf, "faces_equal_unrefined": bool(torch.equal(f, f0)),
            "refine_iterations_mean": ev / nv if nv else 0.0, "refine_iterations_max": iters,
            "max_abs_residual_refined": r, "max_abs_residual_unrefined": r0,
            "extraction_bytes": extraction_bytes(nodes, cubes, nv, nf),
            "extraction_gbps": extraction_bytes(nodes, cubes, nv, nf) / (ms[1] * 1e-3) / 1e9 if ms[1] > 0 else None,
            "device_bytes_held_after_call": int(held), "device_bytes_per_node": held / nodes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[128, 256])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    ic = fb.interpolant_config
    rows = []
    rng = np.random.default_rng(0)
    pts = rng.random((200_000, 3))
    vals = np.sin(4 * pts[:, 0]) * np.cos(3 * pts[:, 1]) + pts[:, 2]
    model = fb.RBFInterpolator(pts, vals, ic.InterpolantSettings(ic.RBFKernelType.Linear))
    for g in a.grids:
        rows.append(bench_case("latency", model, [0.0, 0.0, 0.0, 1.0, 1.0, 1.0], g, 0.5, a.reps))
        print(json.dumps(rows[-1]), flush=True)
    del model
    d = np.load("tests/golden/albatite_SD_points.npz")
    model = fb.RBFInterpolator(d["points"], d["values"], ic.InterpolantSettings(ic.RBFKernelType.Cubic))
    lo, hi = np.floor(d["points"].min(0)), np.ceil(d["points"].max(0))
    for g in a.grids:
        rows.append(bench_case("c4", model, list(lo) + list(hi), g, 0.0, a.reps))
        print(json.dumps(rows[-1]), flush=True)
    out = {"card": card(),
           "timing": "stage_ms: fr_isosurface_timing (host clock, each stage ends in a stream synchronise); "
                     "wall_ms: host clock around the synchronous call; median of the repeats after a warm-up",
           "results": rows}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
