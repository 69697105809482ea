"""Count the SASS instructions of the Chamfer filter scan's inner loop, by pipe, per 16 evaluations per query.

    python tools/chamfer_sass_count.py [LIB_OR_CUBIN] [--kernel SUBSTRING] [--all]

Runs on the CPU: it disassembles the built library (default active-3d-vision-and-touch_b200/lib/libptk_b200.so) with
`cuobjdump -sass`.  For every instantiation of the kernel it finds the innermost loop (backward branch) that holds the
FFMA2 instructions of the 3-FFMA filter and counts what that loop issues.  One evaluation costs 1.5 FFMA2, so the loop
is normalised to 24 FFMA2 = 16 evaluations of one query; the same factor scales every other class.

Pipe classes follow the sm_100 issue model: FFMA2 and the other FP32 arithmetic go to the FMA pipe, FMNMX/FMNMX3,
compares, selects and integer logic to the ALU pipe, shared and global memory to the LSU, U* instructions to the
uniform datapath, branches and barriers to the branch unit.
"""
import argparse
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "active-3d-vision-and-touch_b200", "lib", "libptk_b200.so")
CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")

FMA = {"FFMA2", "FADD2", "FMUL2", "FFMA", "FADD", "FMUL", "IMAD", "HFMA2"}
ALU = {"FMNMX", "FMNMX3", "FSETP", "FSEL", "SEL", "ISETP", "LOP3", "IADD3", "MOV", "SHF", "LEA", "PLOP3", "IMNMX",
       "VIADD", "VIADDMNMX", "FSET", "P2R", "R2P", "PRMT", "LEA.HI"}
LSU = {"LDS", "LDG", "STS", "STG", "LD", "ST", "ATOM", "ATOMS", "RED", "SHFL", "LDSM"}
BRANCH = {"BRA", "EXIT", "BAR", "BSSY", "BSYNC", "WARPSYNC", "RET", "CALL", "SYNCS"}

INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def pipe_of(op):
    base = op.split(".")[0]
    if base.startswith("U") and base not in ("UBLKCP",):
        return "uniform"
    for cls, names in (("fma", FMA), ("alu", ALU), ("lsu", LSU), ("branch", BRANCH)):
        if base in names or op in names:
            return cls
    return "other"


def functions(sass):
    for block in re.split(r"\n\s*Function : ", sass)[1:]:
        name = block.split("\n", 1)[0].strip()
        insns = []
        for line in block.split("\n"):
            m = INSN.search(line)
            if m:
                text = re.sub(r"^@!?U?P\w+\s+", "", m.group(2))  # drop the guard predicate
                insns.append((int(m.group(1), 16), text))
        yield name, insns


BRANCH_TARGET = re.compile(r"BRA(?:\.\S+)*\s+(?:!?U?P\w+,\s*)?0x([0-9a-f]+)")


def inner_loop(insns):
    """Smallest backward-branch range holding the most FFMA2: the scan's innermost loop."""
    best = None
    for addr, text in insns:
        m = BRANCH_TARGET.match(text)
        if not m or int(m.group(1), 16) >= addr:
            continue
        body = [t for a, t in insns if int(m.group(1), 16) <= a <= addr]
        n2 = sum(t.startswith("FFMA2") for t in body)
        if n2 and (best is None or n2 > best[0] or (n2 == best[0] and len(body) < len(best[1]))):
            best = (n2, body)
    return best[1] if best else None


def demangle_short(name):
    m = re.search(r"(chamfer_\w+?)ILi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)E", name)
    return f"{m.group(1)}<{','.join(m.groups()[1:])}>" if m else name[:90]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("path", nargs="?", default=DEFAULT_LIB)
    ap.add_argument("--kernel", default="chamfer_nn_filter_tma_kernel")
    ap.add_argument("--all", action="store_true", help="list every mnemonic of the loop, not only the totals")
    args = ap.parse_args()
    sass = subprocess.run([CUOBJDUMP, "-sass", args.path], check=True, capture_output=True, text=True).stdout
    found = False
    for name, insns in functions(sass):
        if args.kernel not in name:
            continue
        body = inner_loop(insns)
        if body is None:
            continue
        found = True
        ops = collections.Counter(t.split()[0] for t in body)
        n_ffma2 = ops["FFMA2"]
        scale = 24.0 / n_ffma2  # -> per 16 evaluations of one query
        pipes = collections.Counter()
        for op, n in ops.items():
            pipes[pipe_of(op)] += n
        print(f"{demangle_short(name)}: inner loop {len(body)} instructions, {n_ffma2} FFMA2 "
              f"= {n_ffma2 / 24.0:g} x (16 evaluations x 1 query)")
        print("  per 16 evaluations per query: " + ", ".join(f"{p} {pipes[p] * scale:.2f}" for p in
                                                           ("fma", "alu", "lsu", "uniform", "branch", "other")))
        print(f"    FFMA2 {n_ffma2 * scale:.2f}, FMNMX3 {ops['FMNMX3'] * scale:.2f}, "
              f"ALU other than FMNMX3 {(pipes['alu'] - ops['FMNMX3']) * scale:.2f}")
        skips = sum(1 for t in body[:-1] if BRANCH_TARGET.match(t))
        if skips:
            print(f"    note: {skips} branch(es) inside the loop: these are static counts, and code a branch skips "
                  f"does not run on every iteration")
        if args.all:
            for op, n in ops.most_common():
                print(f"      {op:<22} {pipe_of(op):<8} {n:5d}  {n * scale:7.3f}")
    if not found:
        sys.exit(f"no {args.kernel} with an FFMA2 loop in {args.path}")


if __name__ == "__main__":
    main()
