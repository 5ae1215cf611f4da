"""Per-loop opcode counts of a kernel's SASS.

    python tools/sass_loop_mix.py <object or library> <mangled kernel name> [--evals N]

Runs `cuobjdump -sass -fun <kernel>` and reports every loop of the kernel: a backward branch at address B to target A
< B closes the loop [A, B].  For each loop it prints the instruction count, the opcode histogram (by base opcode, e.g.
`LDS.128` counts under `LDS`) and, with --evals N (kernel evaluations per trip), instructions per evaluation for the
innermost loop that contains a MUFU (the kernel evaluations).  The loops are listed innermost first (shortest span).
"""
import argparse
import collections
import re
import subprocess
import sys

_INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")
_BRA_TARGET = re.compile(r"\bBRA\b.*?(0x[0-9a-f]+)\s*$")


def parse_sass(text):
    """[(address, full instruction text without predicate)] in program order."""
    out = []
    for line in text.splitlines():
        m = _INSN.search(line)
        if not m:
            continue
        insn = m.group(2).strip()
        if insn.startswith("@"):
            insn = insn.split(None, 1)[1] if " " in insn else insn
        out.append((int(m.group(1), 16), insn))
    return out


def opcode(insn):
    return insn.split()[0].split(".")[0]


def loops(insns):
    """[(start, end)] address ranges closed by backward branches, shortest first."""
    found = set()
    for addr, insn in insns:
        if opcode(insn) != "BRA":
            continue
        m = _BRA_TARGET.search(insn)
        if m and int(m.group(1), 16) <= addr:
            found.add((int(m.group(1), 16), addr))
    return sorted(found, key=lambda r: (r[1] - r[0], r[0]))


def mix(insns, lo, hi):
    body = [i for a, i in insns if lo <= a <= hi]
    return len(body), collections.Counter(opcode(i) for i in body), collections.Counter(
        i.split()[0] for i in body if opcode(i) in ("LDS", "STS", "LDL", "STL"))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("binary")
    ap.add_argument("kernel", help="mangled kernel name (cuobjdump -fun)")
    ap.add_argument("--evals", type=float, default=0.0, help="kernel evaluations per trip of the innermost loop")
    args = ap.parse_args(argv)
    text = subprocess.run(["cuobjdump", "-sass", "-fun", args.kernel, args.binary], check=True, capture_output=True,
                          text=True).stdout
    insns = parse_sass(text)
    if not insns:
        sys.exit(f"no SASS for {args.kernel} in {args.binary}")
    print(f"kernel {args.kernel}: {len(insns)} instructions")
    inner_done = False
    for lo, hi in loops(insns):
        n, ops, mem = mix(insns, lo, hi)
        line = f"loop [{lo:#06x}, {hi:#06x}]: {n} instructions"
        if args.evals > 0 and ops["MUFU"] > 0 and not inner_done:
            line += f", {n / args.evals:.2f} per evaluation ({args.evals:g} per trip)"
            inner_done = True
        print(line)
        print("  " + "  ".join(f"{k} {v}" for k, v in ops.most_common()))
        if mem:
            print("  memory: " + "  ".join(f"{k} {v}" for k, v in sorted(mem.items())))


if __name__ == "__main__":
    main()
