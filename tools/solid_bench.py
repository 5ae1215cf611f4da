"""Cost of closing and measuring: RBFInterpolator.extract_solids_cuda (fr_isosurface_extract_solid) against
extract_isosurfaces_cuda (fr_isosurface_extract) on the models of tools/isosurface_bench.py ("latency": N = 200 000
uniform points, linear kernel, isovalue 0.5 on [0, 1]^3; "c4": the albatite signed-distance points, cubic kernel,
isovalue 0 on their box) at 128^3 and 256^3.  The two calls alternate, open first, after one warm-up of each; per
case the medians of the host clock around the synchronous call and of the fr_isosurface_timing stages (for solids
the refinement stage includes the volume and area reductions, the extraction stage the cap), the cap's vertex and
face counts, the volumes of both sides with their sum against the box volume, the isosurface area and the closedness
check (every directed edge once, none open).  The card's name and power limit are read in the same run.

    python tools/solid_bench.py [--grids 128 256] [--reps 5] [--out profiles/r6_solid_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ferreus_rbf_rs_b200 as fb  # noqa: E402
from isosurface_bench import card  # noqa: E402
from tests import isosurface_oracle as oi  # noqa: E402


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out, stats = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out, stats


def bench_case(name, model, ext, g, iso, reps):
    import torch
    dev = torch.device("cuda")
    res = (g, g, g)
    open_call = lambda: model._isosurfaces([iso], ext, res, 0, True, dev)  # noqa: E731
    solid_call = lambda: model._isosurfaces([iso], ext, res, 0, True, dev, 0)  # noqa: E731
    open_call()
    solid_call()
    w_open, w_solid, s_open, s_solid = [], [], [], []
    for _ in range(reps):
        t, _, st = timed(open_call)
        w_open.append(t)
        s_open.append(st["ms"])
        t, below, st = timed(solid_call)
        w_solid.append(t)
        s_solid.append(st["ms"])
    below = below[0]
    above = model._isosurfaces([iso], ext, res, 0, True, dev, 1)[0][0]
    box = float(np.prod(np.subtract(ext[3:], ext[:3])))
    closed = {}
    for side, s in (("below", below), ("above", above)):
        once, open_edges = oi.edge_use(s.faces.cpu().numpy())
        closed[side] = bool(once and not open_edges)
    med = lambda a: float(np.median(a))  # noqa: E731
    return {"model": name, "lattice": list(res), "isovalue": iso, "extents": [float(x) for x in ext],
            "open_wall_ms_median": med(w_open), "solid_wall_ms_median": med(w_solid),
            "solid_over_open": med(w_solid) / med(w_open),
            "open_wall_ms_all": w_open, "solid_wall_ms_all": w_solid,
            "open_stage_ms_median": [med([s[i] for s in s_open]) for i in range(4)],
            "solid_stage_ms_median": [med([s[i] for s in s_solid]) for i in range(4)],
            "surface_vertices": below.n_surface_vertices, "surface_faces": below.n_surface_faces,
            "cap_vertices_below": int(below.vertices.shape[0]) - below.n_surface_vertices,
            "cap_faces_below": int(below.faces.shape[0]) - below.n_surface_faces,
            "cap_vertices_above": int(above.vertices.shape[0]) - above.n_surface_vertices,
            "cap_faces_above": int(above.faces.shape[0]) - above.n_surface_faces,
            "volume_below": below.volume, "volume_above": above.volume, "box_volume": box,
            "volume_sum_rel_error": (below.volume + above.volume - box) / box,
            "surface_area": below.surface_area, "surface_area_above": above.surface_area, "closed": closed}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[128, 256])
    ap.add_argument("--reps", type=int, default=5)
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
           "timing": "wall_ms: host clock around the synchronous call, open and solid calls alternating after one "
                     "warm-up of each; stage_ms: fr_isosurface_timing (lattice evaluation with its tree, extraction, "
                     "refinement, normals); medians of the repeats",
           "results": rows}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
