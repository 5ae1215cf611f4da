"""Instruction budget of the W/X inner loop at the headline shape (order 7, 3-D, linear kernel, 1 RHS, fused M2P,
second-order square root), read from the built library's SASS: no spills, no local-memory traffic and no branch
other than the back edge inside the loop, at most 10 warp-instructions per kernel evaluation (6 of them FP64 and one
MUFU are the arithmetic itself)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sass_loop_mix  # noqa: E402

LIB = os.path.join(ROOT, "ferreus_rbf_rs_b200", "libferreus_b200.so")
KERNEL = "_ZN2fb12k_p2l_grid_tILi0ELi1ELi7ELi3ELb1ELb1EEEvNS_7P2LArgsE"  # k_p2l_grid_t<KF_LINEAR, 1, 7, 3, true, true>
EVALS_PER_TRIP = 4 * 7  # kP2LJB sources x 7 nodes of the thread's column


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_headline_wx_loop_within_budget():
    assert os.path.exists(LIB), "build the library first (__graft_entry__.build())"
    text = subprocess.run(["cuobjdump", "-sass", "-fun", KERNEL, LIB], check=True, capture_output=True,
                          text=True).stdout
    insns = sass_loop_mix.parse_sass(text)
    assert insns, f"{KERNEL} not in {LIB}"
    ops = [sass_loop_mix.opcode(i) for _, i in insns]
    assert "LDL" not in ops and "STL" not in ops  # no spills anywhere in the kernel
    inner = [(lo, hi) for lo, hi in sass_loop_mix.loops(insns) if sass_loop_mix.mix(insns, lo, hi)[1]["MUFU"] > 0]
    assert inner, "no loop with kernel evaluations"
    lo, hi = inner[0]
    n, mix, _ = sass_loop_mix.mix(insns, lo, hi)
    assert mix["MUFU"] == EVALS_PER_TRIP, mix
    assert mix["BRA"] == 1, mix  # the back edge only
    assert n / EVALS_PER_TRIP <= 10.0, (n, mix)
