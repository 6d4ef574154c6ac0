#!/usr/bin/env python3
"""Count the instructions of a matvec kernel's consumer loop, per chunk and by opcode class.

usage: tools/sass_loop_count.py <object | cubin | library> <kernel-name substring> [--paths N]

The consumer loop is the innermost loop (a backward branch and its target) that contains both an mbarrier wait
(SYNCS.PHASECHK.TRANS64.TRYWAIT) and dp4a instructions (IDP.4A).  Its steady state is every path from the loop
head to the back-branch that
  * does not retry the mbarrier wait (backward edges are dropped),
  * does not take a BRA.DIV edge (the compiler's fall-back for a diverged warp),
  * does not enter the tile flush (blocks with warp shuffles: once per tile, not per chunk).
Each such path is printed with its instruction count divided by the number of mbarrier waits on it (= chunks per
iteration), so a loop that handles two chunks per trip is comparable with one that handles one.  A dual-format kernel
has one path per format.  Needs cuobjdump (CUDA toolkit); no GPU.
"""
import argparse
import re
import subprocess
import sys
from collections import Counter

INSN = re.compile(r"^\s*/\*([0-9a-f]+)\*/\s+(.*?)\s*;")
TARGET = re.compile(r"\b0x([0-9a-f]+)\b")

CLASSES = [
    ("dot", ("IDP",)),
    ("shared load", ("LDS", "LDSM")),
    ("fp / convert", ("FMUL", "FADD", "FFMA", "FHFMA", "HADD2", "HFMA2", "HMUL2", "I2FP", "I2F", "F2F", "F2I", "DFMA", "DADD",
                      "DMUL", "FSEL", "FMNMX")),
    ("int alu", ("LOP3", "IADD3", "IMAD", "VIADD", "IADD", "SEL", "ISETP", "LEA", "SHF", "PRMT", "MOV", "CS2R", "UMOV", "ULOP3",
                 "UIADD3", "USEL", "UISETP", "BMSK", "SGXT", "IABS", "IMNMX", "VIMNMX", "R2UR", "UMOV", "PLOP3", "P2R", "R2P")),
    ("const / special", ("LDC", "LDCU", "ULDC", "S2R", "S2UR", "CS2R")),
    ("sync / control", ("SYNCS", "YIELD", "BSSY", "BSYNC", "BRA", "NOP", "WARPSYNC", "ELECT", "VOTE", "VOTEU", "BAR", "EXIT",
                        "DEPBAR", "WARPGROUP")),
]


def opcode(text):
    t = text
    if t.startswith("@"):
        t = t.split(None, 1)[1]
    return t.split()[0]


def op_class(op):
    base = op.split(".")[0]
    for name, ops in CLASSES:
        if base in ops:
            return name
    return "other"


def functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :", 1)[1].strip()
            funcs[name] = []
            continue
        m = INSN.match(line)
        if name and m:
            funcs[name].append((int(m.group(1), 16), m.group(2)))
    return funcs


def branch_target(text):
    op = opcode(text)
    if not op.startswith("BRA"):
        return None
    m = TARGET.search(text.split(op, 1)[1])
    return int(m.group(1), 16) if m else None


def consumer_loops(insns):
    addr_idx = {a: k for k, (a, _) in enumerate(insns)}
    loops = []
    for k, (a, t) in enumerate(insns):
        tgt = branch_target(t)
        if tgt is None or tgt > a or tgt not in addr_idx:
            continue
        body = insns[addr_idx[tgt]:k + 1]
        ops = [opcode(x) for _, x in body]
        if any(o.startswith("SYNCS.PHASECHK") for o in ops) and any(o.startswith("IDP") for o in ops):
            loops.append((addr_idx[tgt], k))
    # innermost first: a loop that encloses another candidate is not the consumer loop
    return [l for l in loops if not any(o != l and l[0] <= o[0] and o[1] <= l[1] for o in loops)]


def steady_paths(insns, lo, hi, limit):
    """every head -> back-branch path through [lo, hi] under the rules in the module docstring"""
    addr_idx = {a: k for k, (a, _) in enumerate(insns)}
    # basic-block leaders
    leaders = {lo}
    for k in range(lo, hi + 1):
        t = insns[k][1]
        tgt = branch_target(t)
        if tgt is not None or opcode(t) in ("EXIT", "RET"):
            if k + 1 <= hi:
                leaders.add(k + 1)
            if tgt is not None and tgt in addr_idx and lo <= addr_idx[tgt] <= hi:
                leaders.add(addr_idx[tgt])
    starts = sorted(leaders)
    blocks = {s: (s, (starts[n + 1] - 1) if n + 1 < len(starts) else hi) for n, s in enumerate(starts)}

    def succ(s):
        b0, b1 = blocks[s]
        last = insns[b1][1]
        op, tgt = opcode(last), branch_target(last)
        res = []
        if tgt is not None and not op.startswith("BRA.DIV") and tgt in addr_idx:
            ti = addr_idx[tgt]
            if b1 < ti <= hi:  # forward edges inside the loop only
                res.append(ti)
        unconditional = (op in ("BRA", "EXIT", "RET") or op.startswith("BRA.")) and not last.startswith("@") and not op.startswith("BRA.DIV")
        if not unconditional and b1 + 1 <= hi:
            res.append(b1 + 1)
        return res

    def flush(s):
        b0, b1 = blocks[s]
        return any(opcode(x).startswith("SHFL") for _, x in insns[b0:b1 + 1])

    paths, stack = [], [(lo, [lo])]
    while stack and len(paths) < limit:
        s, path = stack.pop()
        if flush(s):
            continue
        if blocks[s][1] == hi:
            paths.append(path)
            continue
        for n in succ(s):
            stack.append((n, path + [n]))
    return [[k for s in p for k in range(blocks[s][0], blocks[s][1] + 1)] for p in paths]


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("obj")
    ap.add_argument("kernel", help="substring of the mangled kernel name, e.g. matvec_kernelINS_6FmtQ4KELi1ELb1ELb0ELi2E")
    ap.add_argument("--paths", type=int, default=16, help="at most this many steady-state paths")
    ap.add_argument("--opcodes", action="store_true", help="also list every opcode of each path")
    args = ap.parse_args()
    funcs = {n: v for n, v in functions(args.obj).items() if args.kernel in n}
    if not funcs:
        sys.exit(f"no kernel matching {args.kernel!r} in {args.obj}")
    if len(funcs) > 1:
        sys.exit("ambiguous kernel substring, matches:\n  " + "\n  ".join(sorted(funcs)))
    (name, insns), = funcs.items()
    loops = consumer_loops(insns)
    if not loops:
        sys.exit(f"{name}: no loop with an mbarrier wait and dp4a found")
    print(name)
    for lo, hi in loops:
        print(f"loop 0x{insns[lo][0]:x} .. 0x{insns[hi][0]:x}")
        paths = sorted(steady_paths(insns, lo, hi, args.paths), key=len)
        for p in paths:
            ops = [opcode(insns[k][1]) for k in p]
            chunks = sum(o.startswith("SYNCS.PHASECHK") for o in ops) or 1
            by_class = Counter(op_class(o) for o in ops)
            print(f"  path: {len(ops)} instructions, {chunks} chunk(s) -> {len(ops) / chunks:.1f} per chunk")
            for cls, _ in CLASSES + [("other", ())]:
                if by_class[cls]:
                    print(f"    {cls:16s} {by_class[cls] / chunks:6.1f}")
            if args.opcodes:
                for o, c in sorted(Counter(ops).items(), key=lambda x: -x[1]):
                    print(f"      {o:32s} {c / chunks:6.1f}")


if __name__ == "__main__":
    main()
