"""Static SASS instructions per source line of one kernel, from the cubin's line table (nvdisasm -gi): what
ncu_lines.py reports for executed instructions, without a profiler.  Counts are instructions in the binary,
not instructions executed: a line inside a loop counts once, a branch that is rarely taken counts in full.

    python scratch/sass_lines.py LIB.so KERNEL_MANGLED [--cubin NAME] [--file rt_warp.cuh]
                                 [--region NAME=LO-HI ...] [--within LO-HI] [--top N] [--dump]

Per line, each instruction is charged to the innermost frame of its inline chain that lies in --file (default
rt_warp.cuh), so that code inlined from other headers counts at the line of --file that calls it.  --region
NAME=LO-HI sums under NAME the instructions with a frame on lines LO..HI of --file, the innermost such frame
deciding (so a helper called from two regions counts in each where it is called); the rest is "other".
--within LO-HI keeps only the instructions with a frame on lines LO..HI of --file: one loop of the kernel,
including what is inlined into it."""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

FRAME = re.compile(r'"([^"]+)", line (\d+)')


def disassemble(lib, cubin, mangled):
    tmp = tempfile.mkdtemp()
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
    names = [f for f in os.listdir(tmp) if f.endswith(".cubin") and cubin in f]
    for name in sorted(names):
        dis = subprocess.run(["nvdisasm", "-gi", os.path.join(tmp, name)], capture_output=True, text=True, check=True).stdout.splitlines()
        head = ".text." + mangled + ":"
        if head in dis:
            return dis[dis.index(head) + 1:]
    sys.exit(f"{mangled} not found in {names}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib")
    ap.add_argument("kernel")
    ap.add_argument("--cubin", default="rt_kernels_f32")
    ap.add_argument("--file", default="rt_warp.cuh")
    ap.add_argument("--region", action="append", default=[])
    ap.add_argument("--within", help="LO-HI: only instructions with a frame on these lines of --file")
    ap.add_argument("--top", type=int, default=40)
    ap.add_argument("--dump", action="store_true", help="every instruction with its line")
    args = ap.parse_args()

    regions = []
    for r in args.region:
        name, span = r.split("=")
        lo, hi = (int(x) for x in span.split("-"))
        regions.append((name, lo, hi))

    def region_of(chain):
        for f, n in chain:
            for name, lo, hi in regions:
                if f == args.file and lo <= n <= hi:
                    return name
        return "other"

    within = tuple(int(x) for x in args.within.split("-")) if args.within else None
    # nvdisasm -gi writes an instruction's inline chain as consecutive "//## File" lines, innermost first
    insts = []  # (chain, text)
    chain, fresh = [("?", 0)], True
    for l in disassemble(args.lib, args.cubin, args.kernel):
        if l.startswith("\t.section") or l.startswith(".text."):
            break
        if "//## File" in l:
            f, n = FRAME.search(l).groups()
            chain = [(os.path.basename(f), int(n))] if fresh else chain + [(os.path.basename(f), int(n))]
            fresh = False
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
        if m:
            if not within or any(f == args.file and within[0] <= n <= within[1] for f, n in chain):
                insts.append((chain, m.group(2)))
            fresh = True
    line_of = lambda chain: next((fr for fr in chain if fr[0] == args.file), chain[-1])
    if args.dump:
        for chain, txt in insts:
            f, n = line_of(chain)
            print(f"{f}:{n:<5d} {region_of(chain):12s} {' < '.join(f'{a}:{b}' for a, b in chain):60s} {txt}")
        return

    per_line = collections.Counter(line_of(chain) for chain, _ in insts)
    per_region = collections.Counter(region_of(chain) for chain, _ in insts)
    total = len(insts)
    op = lambda t: t.split()[1] if t.startswith("@") else t.split()[0]
    print(f"{args.kernel}: {total} SASS instructions, {sum(op(t).startswith('STL') for _, t in insts)} STL, "
          f"{sum(op(t).startswith('LDL') for _, t in insts)} LDL, {sum(op(t).startswith('CALL') for _, t in insts)} CALL")
    # FP32-pipe opcodes per region: packed (FFMA2 / FMUL2 / FADD2) against scalar, and the moves that form pairs
    fp_classes = (("packed", ("FFMA2", "FMUL2", "FADD2")), ("scalar", ("FFMA", "FMUL", "FADD")), ("mov", ("MOV", "PRMT")))
    fp_of = lambda t: next((c for c, ops in fp_classes if op(t).split(".")[0] in ops), None)
    per_region_fp = collections.Counter((region_of(chain), fp_of(t)) for chain, t in insts)
    if regions:
        for name, lo, hi in regions + [("other", 0, 0)]:
            span = f"{args.file}:{lo}-{hi}" if name != "other" else ""
            fp = "  ".join(f"{c} {per_region_fp[(name, c)]:4d}" for c, _ in fp_classes)
            print(f"  region {name:12s} {per_region[name]:6d}  {fp}  {span}")
    for (f, n), k in sorted(per_line.items(), key=lambda kv: -kv[1])[:args.top]:
        print(f"  {f}:{n:<5d} {k:6d}")


if __name__ == "__main__":
    main()
