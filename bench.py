#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: BBFMM matvec throughput (Mpts/s), 3-D N = 1M.

One "step" = one matvec = set_weights(w) + evaluate(w, targets = sources) on a pre-built tree
(exactly one solver matvec of the reference, ferreus_rbf/src/rbf.rs:1357-1364).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n POINTS] [--dump-outputs DIR]

* `--dump-outputs DIR`: after the timed steps, what each timed path returned in its last step goes to DIR/<name>.npy
             (float64): `matvec` (the resident matvec of `value`; the oracle port's result with --impl reference),
             `matvec_sqrt_exact` and `e2e` (the host-buffer result of the last e2e step), each shaped as its caller
             receives it.  The workload is seeded, so two builds run with the same arguments can be compared output for
             output.  The device sums are not bit-reproducible: compare with a tolerance (two runs of the default
             workload on one B200 differ by 3e-16 in relative L2 norm, at most 2.2e-15 relative per row).

* `value`  : whole-job Mpts/s with inputs resident in HBM (fb_tree_matvec_resident), device time from CUDA
             events on the library's launch stream, max over ranks.
* `e2e`    : same metric through the reference-facing API with HOST buffers: FmmTree.set_weights(w) +
             FmmTree.evaluate(w, points) (H2D of weights and targets, target check / binning, D2H of the result
             inside the timed region).
* `roofline`: dominant kernel = k_p2l_grid<FUSE> (the fused W/X pass: P2L and the M2P transpose from one kernel
             evaluation per point-node pair), algorithmic FLOPs of both passes / CUDA-event time against the FP64
             FMA peak measured in the same run (MEASURED_PEAKS.json has no FP64 entry); the other stages are in
             `stages`.
* `cpu_baseline`: the oracle port (oracle/fast.py + oracle/csrc/oracle_passes.c, OpenMP) on this host.
* `sqrt_exact`: the same resident matvec with the third-order (~1 ulp) square root (fb_set_sqrt_mode(0)); the
             default is the second-order one (<= 1.3e-12 per kernel value, see include/ferreus_b200.h).
N > 1: one process per GPU (torchrun), ONE shared 1M-point cloud partitioned by Morton-contiguous leaf ranges
(csrc/comm.cu): owned-leaf upward pass and ncclAllReduce of the multipoles with the near-field pass beside them on a
low-priority stream, downward / leaf passes of the share (every kernel evaluation of the unpartitioned matvec is made by exactly one rank: the symmetric halves for
foreign rows travel in the result), ncclAllReduce of the full-length result.  `value` = N / (device time of that step, max
over ranks): strong scaling.  Every rank checks the partitioned result against the unpartitioned matvec on its own GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ORDER = 7
KERNEL_FLOPS = {"linear": 1}  # c_k of SURVEY.md §8(d)
# DRAM bytes per launch (read + write) from the committed ncu captures of the default workload: profiles/ncu_traffic.json
# names the capture every figure comes from
try:
    _TRAFFIC = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
except Exception:
    _TRAFFIC = {}
NCU_DRAM_BYTES = {k: v["bytes"] for k, v in _TRAFFIC.items() if isinstance(v, dict)}
NCU_CAPTURE = {k: v["capture"] for k, v in _TRAFFIC.items() if isinstance(v, dict)}
DUMP_BYTES = 60 << 20  # --dump-outputs budget: the .npy files stay under 64 MB in all, headers included


def make_workload(n, seed):
    rng = np.random.default_rng(seed)
    pts = rng.random((n, 3))
    w = rng.random((n, 1))
    return pts, w


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy in float64.  Beyond DUMP_BYTES in all, each array keeps the same fixed,
    seeded sample of its rows (in ascending order), so that two runs stay comparable row for row."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.shape[0] * DUMP_BYTES // total
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([s.strip() for s in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
                for nme, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        # keep the samples taken under load (upper half of the clock distribution)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(pts, w, leaf_fraction):
    """Oracle port on the host cores (kind = "port": restatement of the reference algorithm, not the Rust
    binary — no cargo/rustc on this image).  torchrun exports OMP_NUM_THREADS=1: the OpenMP team is set explicitly
    to every core this process may run on, as the reference's rayon pool would be."""
    from oracle import bbfmm as obb
    from oracle import fast
    from oracle import kernels as okern
    fast.lib().orc_set_num_threads(host_threads())
    t0 = time.perf_counter()
    ot = obb.FmmTree(pts, ORDER, okern.Kernel(okern.LINEAR), True, True, None,
                     obb.FmmParams(256, 2, 10.0 ** -ORDER, 1024))
    ff = fast.FastFmm(ot)
    build_s = time.perf_counter() - t0
    return ff, build_s, fast.lib().orc_num_threads()


def full_fit(n):
    """second half of BASELINE.json's metric: full RBF fit wall time (config C3: clustered 3-D points, linear
    kernel, tol 1e-6 relative, default Params), through RBFInterpolator with host buffers."""
    import ferreus_rbf_rs_b200 as fb
    rng = np.random.default_rng(0)
    centres = rng.random((64, 3))
    pts = centres[rng.integers(0, 64, n)] + 0.02 * rng.standard_normal((n, 3))
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    vals = 0.75 * np.exp(-((9 * x - 2) ** 2 + (9 * y - 2) ** 2 + (9 * z - 2) ** 2) / 4) + \
        0.5 * np.exp(-((9 * x - 7) ** 2 + (9 * y - 3) ** 2 + (9 * z - 5) ** 2) / 4)
    ic = fb.interpolant_config
    # warm-up: a 30k-point fit loads the solver's kernels (CUDA loads modules lazily) before the timed construction
    wp = rng.random((30000, 3))
    fb.RBFInterpolator(wp, wp[:, 0] + wp[:, 1] * wp[:, 2], ic.InterpolantSettings(ic.RBFKernelType.Linear))
    # three complete constructions, each model released outside the timed region; the MEDIAN wall time is reported
    walls, infos = [], []
    for _ in range(3):
        t0 = time.perf_counter()
        model = fb.RBFInterpolator(pts, vals, ic.InterpolantSettings(ic.RBFKernelType.Linear))
        walls.append(time.perf_counter() - t0)
        infos.append(model.info())
        del model
    mid = int(np.argsort(walls)[1])
    info = infos[mid]
    return {"workload": f"ferreus_rbf 3D global fit, linear kernel, tol 1e-6, N={n} clustered (64 Gaussian blobs); "
                        "timed after one 30k-point warm-up fit; median of three constructions",
            "wall_s": walls[mid], "wall_s_all": walls, "setup_s": info["setup_seconds"], "solve_s": info["solve_seconds"],
            "iterations": info["iterations"], "fmm_matvecs": info["matvecs"], "ddm_domains": info["ddm_domains"],
            "final_relative_residual": info["last_residual"]}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port, all host threads) on the same workload.  Every
    step is one complete, fully timed 1M-point matvec (upward pass, M2L, P2L, L2L and the whole leaf pass; nothing is
    extrapolated); --steps of them are timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pts, w = make_workload(args.n, 1000)
    ff, build_s, cores = cpu_baseline(pts, w, args.cpu_leaf_fraction)
    times = []
    warm = min(args.warmup, 1)
    for it in range(warm + args.steps):
        t0 = time.perf_counter()
        out = ff.matvec(w)
        sec = time.perf_counter() - t0
        if it >= warm:
            times.append(sec)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"matvec": out})
    ms = 1e3 * float(np.mean(times))
    val = args.n / (ms * 1e-3) / 1e6
    sample = (f"{len(times)} complete {args.n}-point matvecs of the oracle port (oracle/fast.py + "
              f"oracle/csrc/oracle_passes.c, OpenMP, {cores} threads), every stage timed in full")
    line = {"impl": "reference", "metric": "bbfmm_matvec_throughput", "value": val, "unit": "Mpts/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.n, 1),
            "cpu_baseline": {"value": val, "unit": "Mpts/s", "cores": cores, "kind": "port", "sample": sample,
                             "tree_build_s": build_s, "step_seconds": times},
            "e2e": {"value": val, "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(n, n_gpus):
    par = ("one GPU" if n_gpus == 1 else
           f"one {n}-point cloud partitioned over {n_gpus} GPUs by Morton-contiguous leaf ranges balanced by work; "
           "ncclAllReduce of the multipoles (under the near-field pass) + ncclAllReduce of the full-length result per matvec")
    return {"workload": f"ferreus_bbfmm 3D LinearRbf matvec, N={n} uniform points in the unit cube, "
                        f"Chebyshev order {ORDER}, 1 RHS, adaptive sparse tree, 256 pts/leaf, ACA eps=1e-{ORDER} "
                        "(BASELINE.md headline H)",
            "points": n, "order": ORDER, "nrhs": 1, "kernel": "LinearRbf", "compression": "ACA",
            "sqrt_mode": "second-order (default; <= 1.3e-12 per kernel value; sqrt_exact holds the ~1 ulp variant)",
            "l2_policy": "256 MiB buffer written between timed iterations (L2 flush)",
            "parallelism": par}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--cpu-leaf-fraction", type=float, default=0.02)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fit", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what each timed path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to stdout when the first communicator is created: point fd 1 at stderr
        # until that has happened so that stdout carries exactly one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    import ferreus_rbf_rs_b200 as fb
    from ferreus_rbf_rs_b200 import _lib
    L = _lib.lib()
    L.fb_set_device(local_rank)

    n = args.n
    pts, w = make_workload(n, 1000)  # the same cloud on every rank: N > 1 partitions it
    t0 = time.perf_counter()
    tree = fb.FmmTree(pts, ORDER, fb.KernelParams(fb.FmmKernelType.LinearRbf), True, True)
    build_s = time.perf_counter() - t0
    info = tree.info()
    tree.set_timing(True)
    tree.upload_weights(w)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    partition_err = None
    if world > 1:
        comm = fb.Communicator.from_torch_distributed(dist)
        tree.matvec_resident()
        unpartitioned = np.array(tree.download_result()).reshape(n, -1)
        tree.shard(comm)
        tree.matvec_sharded()
        got = np.array(tree.sharded_download()).reshape(n, -1)
        partition_err = float(np.linalg.norm(got - unpartitioned) / np.linalg.norm(unpartitioned))
        assert partition_err <= 1e-12, f"rank {rank}: partitioned matvec differs from the unpartitioned one: {partition_err}"
        del got, unpartitioned

    def step():
        if world > 1:
            tree.matvec_sharded()
            t = tree.sharded_timing()
            t.update({"k_" + k: v for k, v in tree.last_timing().items()})  # this rank's per-kernel times
            return sum(v for k, v in t.items() if not k.startswith("k_")), t
        tree.matvec_resident()
        return tree.last_matvec_ms(), tree.last_timing()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = L.fb_kernel_launch_count()
    for _ in range(args.warmup):
        step()
    launches_per_step = (L.fb_kernel_launch_count() - launches0) // max(args.warmup, 1)

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    # ---- timed: K resident matvecs, device time (CUDA events on the library stream) per step
    barrier()
    dev_ms, stage_ms = [], []
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms, st = step()
        dev_ms.append(ms)
        stage_ms.append(st)
    barrier()
    wall_s = time.perf_counter() - wall0
    total_ms = float(np.sum(dev_ms))
    dumps = {}
    if args.dump_outputs and rank == 0:  # read back before the e2e calls below reuse the tree's result buffer
        dumps["matvec"] = np.array(tree.sharded_download() if world > 1 else tree.download_result())

    # ---- the same resident matvec with the third-order square root (tree rebuilt in that mode)
    exact = None
    if world == 1:
        fb.set_sqrt_mode(False)
        tree_x = fb.FmmTree(pts, ORDER, fb.KernelParams(fb.FmmKernelType.LinearRbf), True, True)
        fb.set_sqrt_mode(True)
        tree_x.set_timing(True)
        tree_x.upload_weights(w)
        for _ in range(args.warmup):
            tree_x.matvec_resident()
        xs = []
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            tree_x.matvec_resident()
            xs.append(tree_x.last_matvec_ms())
        if args.dump_outputs:
            dumps["matvec_sqrt_exact"] = np.array(tree_x.download_result())
        exact = {"ms_per_step": float(np.mean(xs)), "value": n / (float(np.mean(xs)) * 1e-3) / 1e6, "unit": "Mpts/s",
                 "what": "fb_set_sqrt_mode(0): ~1 ulp square roots in the direct sums"}
        del tree_x

    # ---- e2e: reference-facing calls with host buffers (H2D + D2H inside the timed region).  The weights change
    #      every step, as in a solver: set_weights(w) uploads them, evaluate(w, points) recognises on the host that
    #      w is the vector just set and that the targets are the source points, so neither is sent again.
    w_alt = [w, np.ascontiguousarray(w[::-1])]

    def e2e_step(i):
        if world > 1:  # host weights in, partitioned matvec, full result out to the host on every rank
            tree.upload_weights(w_alt[i % 2])
            tree.matvec_sharded()
            return tree.sharded_download()
        tree.set_weights(w_alt[i % 2])
        return tree.evaluate(w_alt[i % 2], pts)

    for i in range(2):
        e2e_step(i)
    barrier()
    e0 = time.perf_counter()
    for i in range(args.steps):
        out = e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - e0
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:
        dumps["e2e"] = out
        dump_outputs(args.dump_outputs, dumps)

    tms = torch.tensor([total_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    per_rank = None
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        med_r = {k: float(np.median([s_[k] for s_ in stage_ms])) for k in stage_ms[0]}
        a, b = tree.shard_rows(rank)
        kernel_keys = ["p2m", "m2m", "m2l", "wx", "l2l", "l2p", "leaf"]
        mine = torch.tensor([float(b - a), med_r["upward_exchange"], med_r["downward"], med_r["near_field_join_l2p"],
                             med_r["result_allreduce"], partition_err] + [med_r["k_" + k] for k in kernel_keys],
                            dtype=torch.float64, device="cuda")
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        names = ["rows", "upward_exchange_ms", "downward_ms", "near_field_join_l2p_ms", "result_allreduce_ms",
                 "rel_l2_vs_unpartitioned"] + ["kernel_" + k + "_ms" for k in kernel_keys]
        per_rank = [dict(zip(names, v.cpu().tolist())) for v in allv]
    total_ms_max, e2e_ms_max = [float(v) for v in tms.tolist()]

    if rank == 0:
        ms_per_step = total_ms_max / args.steps
        value = n / (ms_per_step * 1e-3) / 1e6
        e2e_val = n / (e2e_ms_max / args.steps * 1e-3) / 1e6
        # ---- roofline of the dominant kernel
        fp64_peak, dmma_peak = np.zeros(1), np.zeros(1)
        L.fb_measure_fp64_tflops(_lib.dptr(fp64_peak))
        L.fb_measure_fp64_dmma_tflops(_lib.dptr(dmma_peak))
        fp64_peak[0] = max(fp64_peak[0], dmma_peak[0])  # one FP64 datapath: the higher of the two readings is the peak
        m2l_flops = np.zeros(1)
        L.fb_tree_m2l_flops(tree._h, _lib.dptr(m2l_flops))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        P = ORDER ** 3
        f_pair = (3 * 3 - 1) + KERNEL_FLOPS["linear"] + 2 * 1          # SURVEY.md §8(d): (3d-1) + c_k + 2K
        pairs_p2p = info["p2p_pairs"]
        pairs_m2p = info["m2p_pairs"] * P
        pairs_p2l = info["p2l_pairs"] * P
        if world == 1:
            med = {k: float(np.median([s[k] for s in stage_ms])) for k in stage_ms[0]}
        else:  # slowest rank per kernel: the time the whole-job FLOP counts below are divided by
            med = {k: max(r["kernel_" + k + "_ms"] for r in per_rank) for k in kernel_keys}
            med["total"] = ms_per_step
        wx_flops = (pairs_m2p + pairs_p2l) * f_pair
        wx_tf = wx_flops / max(med["wx"] * 1e-3, 1e-9) / 1e12
        p2p_tf = pairs_p2p * f_pair / max(med["leaf"] * 1e-3, 1e-9) / 1e12
        direct_tf = (wx_flops + pairs_p2p * f_pair) / max((med["wx"] + med["leaf"]) * 1e-3, 1e-9) / 1e12
        peak = float(fp64_peak[0]) * world  # whole-job FLOPs against the FP64 peak of all GPUs used
        roofline = {"kernel": "k_p2l_grid<FUSE> (W/X pass: P2L + M2P transpose, one kernel evaluation per pair)",
                    "bound": "fp64", "achieved": wx_tf, "peak": peak, "unit": "TFLOP/s", "frac": wx_tf / peak,
                    "traffic": NCU_DRAM_BYTES.get("k_p2l_grid") if n == 1_000_000 and world == 1 else None,
                    "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this "
                                      "kernel at this workload; compute-bound: 81 MB",
                    "peak_source": "in-run DFMA and DMMA micro-benchmarks (fb_measure_fp64_tflops / "
                                   "fb_measure_fp64_dmma_tflops), the higher reading; MEASURED_PEAKS.json has no FP64 entry",
                    "traffic_capture": NCU_CAPTURE.get("k_p2l_grid"),
                    "algorithmic_flops_per_launch": wx_flops, "flops_per_pair": f_pair, "launch_ms": med["wx"],
                    "note": "algorithmic count = SURVEY.md §8(d): M2P and P2L pairs x 11 FLOP; the kernel evaluates the "
                            "symmetric kernel once per (point, node) and uses it for both passes",
                    "p2p": {"kernel": "k_p2p_sym (P2P, targets == sources: each unordered U-list pair evaluated once, "
                                      "both rows updated)",
                            "achieved": p2p_tf, "frac": p2p_tf / peak,
                            "launch_ms": med["leaf"], "algorithmic_flops_per_launch": pairs_p2p * f_pair,
                            "traffic": NCU_DRAM_BYTES.get("k_p2p_sym") if n == 1_000_000 and world == 1 else None,
                            "traffic_capture": NCU_CAPTURE.get("k_p2p_sym"),
                            "note": "algorithmic count = every ordered (target, source) pair of the reference's U lists "
                                    "x 11 FLOP (SURVEY.md 8(d)); the kernel evaluates half of them"},
                    "pipe_note": "FP64 tensor instructions (DMMA) share the DFMA datapath on B200 (tools/dmma_bench.cu mix "
                                 "test, profiles/r1_dmma_dfma_mix.txt: 4 DMMA + 32 DFMA per trip take the sum of the two "
                                 "times), so this one FP64 peak bounds P2P, W/X and M2L alike",
                    "direct_sums_total": {"achieved": direct_tf, "frac": direct_tf / peak},
                    "m2l": {"kernel": "k_m2l_stream (TMA bulk gathers, register-resident operator slices, DMMA, TMA "
                                      "scatter-adds)",
                            "achieved": float(m2l_flops[0]) / max(med["m2l"] * 1e-3, 1e-9) / 1e12,
                            "frac": float(m2l_flops[0]) / max(med["m2l"] * 1e-3, 1e-9) / 1e12 / peak,
                            "launch_ms": med["m2l"], "algorithmic_flops_per_launch": float(m2l_flops[0]),
                            "traffic": NCU_DRAM_BYTES.get("k_m2l_stream") if n == 1_000_000 and world == 1 else None,
                            "traffic_capture": NCU_CAPTURE.get("k_m2l_stream"),
                            "note": "algorithmic count = sum over V-list entries of 4 r P with the reference's truncation "
                                    "ranks r (SURVEY.md 8(d)); rank tiles are padded to 8"},
                    "stage_fractions": {k: med[k] / max(med["total"], 1e-9) for k in med if k != "total"},
                    "peaks": {"dfma_tflops": float(fp64_peak[0]) if dmma_peak[0] <= fp64_peak[0] else None,
                              "dmma_tflops": float(dmma_peak[0]), "per_gpu_peak_used": float(fp64_peak[0]),
                              "measured": "in this run, after the timed region, 8 repetitions each (the first two bring the "
                                          "clocks up), best of the rest"}}
        stages = {"ms": med, "hbm_peak_gbs": hbm_peak,
                  "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                  "pairs": {"p2p": pairs_p2p, "m2p_nodes": pairs_m2p, "p2l_nodes": pairs_p2l,
                            "m2l_entries": info["n_v"]}}
        line = {"metric": "bbfmm_matvec_throughput", "value": value, "unit": "Mpts/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(n, world),
                "e2e": {"value": e2e_val, "unit": "Mpts/s", "h2d_bytes_per_step": int(w.nbytes) * world,
                        "d2h_bytes_per_step": int(out.nbytes) * world,
                        "api": ("FmmTree.set_weights + FmmTree.evaluate" if world == 1 else
                                "FmmTree.upload_weights + FmmTree.matvec_sharded + FmmTree.sharded_download on every rank"),
                        "note": "weights alternate between two vectors; N = 1: the second copy of w (evaluate) and the "
                                "targets (== source points) are compared on the host instead of being re-sent; N > 1: "
                                "every rank uploads the full weight vector and downloads the full result"},
                "gpu_launches": int(launches_per_step * args.steps),
                "clocks": clocks, "roofline": roofline, "stages": stages, "sqrt_exact": exact,
                "tree": {"build_s": build_s, "cells": info["n_cells"], "leaves": info["n_leaves"],
                         "depth": info["depth"]},
                "wall_s_timed_region": wall_s}
        if per_rank is not None:
            line["partition"] = {"per_rank": per_rank,
                                 "what": "device time per stage and per kernel on every rank (median over the timed steps); "
                                         "upward_exchange = weight sort, owned-leaf upward pass and the multipole all-reduce on the "
                                         "high-priority stream (the symmetric P2P of the owned chunks runs beside them and "
                                         "beside the downward pass on a low-priority stream); near_field_join_l2p = what is "
                                         "left of the P2P when the downward pass is done, plus L2P"}
        if world == 1 and not args.no_fit:
            line["fit"] = full_fit(n)
        if world == 1 and not args.no_cpu_baseline:
            ff, cpu_build_s, cores = cpu_baseline(pts, w, args.cpu_leaf_fraction)
            t0 = time.perf_counter()
            cpu_out = ff.matvec(w)
            sec = time.perf_counter() - t0
            # the timed CPU result doubles as a parity check of the timed GPU path (bar: 1e-10, tests/test_gpu_configs.py)
            tree.set_weights(w)
            gpu_out = np.asarray(tree.evaluate(w, pts)).reshape(n, 1)
            line["cpu_baseline"] = {
                "value": n / sec / 1e6, "unit": "Mpts/s", "cores": cores, "kind": "port",
                "sample": "one complete 1M-point matvec of the oracle port (OpenMP over cells / leaves like the "
                          "reference's rayon loops), every stage timed in full, nothing extrapolated",
                "seconds_per_matvec": sec, "tree_build_s": cpu_build_s,
                "rel_l2_gpu_vs_cpu": float(np.linalg.norm(gpu_out - cpu_out) / np.linalg.norm(cpu_out))}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
