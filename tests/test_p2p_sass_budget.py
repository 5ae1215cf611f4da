"""Instruction budget of the one-column symmetric P2P kernel at the headline shape (linear kernel, second-order square
root, four targets per lane), read from the built library's SASS: no spills, no local-memory traffic, the back edge as
the only branch of the source loop, 11 FP64 instructions and one MUFU per kernel evaluation, and at most 15.75
warp-instructions per evaluation in all (the two-target body of k_p2p_sym runs 16.4)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sass_loop_mix  # noqa: E402

LIB = os.path.join(ROOT, "ferreus_rbf_rs_b200", "libferreus_b200.so")
KERNEL = "_ZN2fb17k_p2p_sym_blockedILi0ELb1EEEvNS_10DirectArgsEi"  # k_p2p_sym_blocked<KF_LINEAR, true>
EVALS_PER_TRIP = 2 * 4  # two sources per trip (unroll 2) x four targets per lane
FP64 = ("DADD", "DMUL", "DFMA")


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_headline_p2p_loop_within_budget():
    assert os.path.exists(LIB), "build the library first (__graft_entry__.build())"
    text = subprocess.run(["cuobjdump", "-sass", "-fun", KERNEL, LIB], check=True, capture_output=True,
                          text=True).stdout
    insns = sass_loop_mix.parse_sass(text)
    assert insns, f"{KERNEL} not in {LIB}"
    ops = [sass_loop_mix.opcode(i) for _, i in insns]
    assert "LDL" not in ops and "STL" not in ops  # no spills anywhere in the kernel
    # the source loop of the four-target body: one partial-sum store per source, every evaluation's FP64 work (the
    # diagonal loops evaluate fewer source-side terms and so fewer FP64 instructions per MUFU)
    body = []
    for lo, hi in sass_loop_mix.loops(insns):
        n, mix, _ = sass_loop_mix.mix(insns, lo, hi)
        if mix["MUFU"] == EVALS_PER_TRIP and mix["STS"] == 2 and sum(mix[k] for k in FP64) == 11 * EVALS_PER_TRIP:
            body.append((n, mix))
    assert body, "no four-target source loop with 11 FP64 instructions per evaluation"
    n, mix = body[0]
    assert mix["BRA"] == 1, mix  # the back edge only
    assert mix["LDS"] == 4, mix  # {x, y}, {z, w} of two sources: one broadcast per source for four evaluations
    assert n / EVALS_PER_TRIP <= 15.75, (n, mix)
