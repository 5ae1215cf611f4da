"""A/B of the W/X pass (P2L + fused M2P): the order-templated kernel k_p2l_grid_t against the generic k_p2l_grid.

    python tools/wx_ab.py [--runs 3] [--c5-runs 1] [--out profiles/r3_wx_ab.json]

Runs `bench.py --no-cpu-baseline` --runs times per arm in one process tree, alternating FB_GENERIC_P2L=1 (generic) and
the default (templated), so both arms see the same card, clocks and neighbours.  Stage times come from the bench's CUDA
events.  The first run of each arm also dumps its outputs (--dump-outputs), and the relative L2 distance of the two
`matvec` results is recorded.  --c5-runs > 0 adds alternating `tools/config_bench.py C5` runs (10M clustered points,
spheroidal, 8 right-hand sides: the NR = 4 instantiations).  The card's name and power limit are read with a read-only
nvidia-smi query in the same call.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARMS = (("generic", {"FB_GENERIC_P2L": "1"}), ("templated", {}))


def last_json(stdout):
    for line in reversed(stdout.splitlines()):
        line = line.strip()
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in output:\n" + stdout[-2000:])


def run(cmd, extra_env):
    env = dict(os.environ)
    env.pop("FB_GENERIC_P2L", None)
    env.update(extra_env)
    t0 = time.perf_counter()
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} failed ({p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
    return last_json(p.stdout), time.perf_counter() - t0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    name, power = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "count": len(q)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--c5-runs", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_wx_ab.json"))
    args = ap.parse_args()
    result = {"gpu": gpu_info(), "arms": {a: {"bench": [], "c5": []} for a, _ in ARMS},
              "what": "bench.py --no-cpu-baseline, arms alternated in one call; generic = FB_GENERIC_P2L=1 "
                      "(k_p2l_grid), templated = default (k_p2l_grid_t at order 7, 3-D)"}
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(args.runs):
            for arm, env in ARMS:
                cmd = [sys.executable, "bench.py", "--no-cpu-baseline"]
                if i == 0:
                    cmd += ["--dump-outputs", os.path.join(tmp, arm)]
                line, wall = run(cmd, env)
                rec = {k: line.get(k) for k in ("value", "ms_per_step", "sqrt_exact", "fit", "clocks")}
                rec["stages_ms"] = line["stages"]["ms"]
                rec["wx_roofline_frac"] = line.get("roofline", {}).get("frac")
                rec["wall_s"] = wall
                result["arms"][arm]["bench"].append(rec)
                print(f"run {i} {arm}: {line['value']:.2f} Mpts/s, wx {line['stages']['ms']['wx']:.3f} ms",
                      flush=True)
        ref = np.load(os.path.join(tmp, "generic", "matvec.npy"))
        new = np.load(os.path.join(tmp, "templated", "matvec.npy"))
        result["matvec_rel_l2_templated_vs_generic"] = float(np.linalg.norm(new - ref) / np.linalg.norm(ref))
        result["matvec_bitwise_equal"] = bool(np.array_equal(new, ref))
    for i in range(args.c5_runs):
        for arm, env in ARMS:
            line, wall = run([sys.executable, "tools/config_bench.py", "C5"], env)
            line["wall_s"] = wall
            result["arms"][arm]["c5"].append(line)
            print(f"C5 run {i} {arm}: {json.dumps(line)[:300]}", flush=True)
    for arm, _ in ARMS:
        b = result["arms"][arm]["bench"]
        result["arms"][arm]["summary"] = {
            "value": [r["value"] for r in b], "wx_ms": [r["stages_ms"]["wx"] for r in b],
            "total_ms": [r["stages_ms"].get("total") for r in b],
            "sqrt_exact_value": [(r["sqrt_exact"] or {}).get("value") for r in b],
            "fit_wall_s": [(r["fit"] or {}).get("wall_s") for r in b]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({a: result["arms"][a]["summary"] for a, _ in ARMS}))
    print("matvec rel L2 templated vs generic:", result["matvec_rel_l2_templated_vs_generic"])


if __name__ == "__main__":
    main()
