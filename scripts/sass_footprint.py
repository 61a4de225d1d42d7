#!/usr/bin/env python
"""Code footprint of the fused small-batch kernels in a built libmppi_b200.so (runs on the CPU, needs cuobjdump/nvdisasm).

  python scripts/sass_footprint.py [path/to/libmppi_b200.so] [--lines 25] [--bucket 20] [--match tile_fused]

For every tile_fused_kernel / tile_fused_batch_kernel instance: registers and stack frame (cuobjdump -res-usage), the SASS
instruction count of the kernel's text section (which holds its __noinline__ callees too: all of it can be fetched by one
launch), the CALL, LDL / STL, SHFL and BAR counts, and where the instructions come from (nvdisasm --print-line-info-inline):
  - by the innermost source line (device helpers show as themselves), the largest --lines entries;
  - by --bucket-line range of mppi_kernels.cuh, taking the innermost frame that lies in that file (a helper's code is
    charged to the kernel line that calls it).
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)")
LOC = re.compile(r'^\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')
SECTION = re.compile(r"^\s*\.section\s+\.text\.(\S+?),")


def disassemble(lib):
    with tempfile.TemporaryDirectory() as d:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=d, check=True, capture_output=True)
        cubins = sorted(f for f in os.listdir(d) if f.endswith(".cubin"))
        if not cubins:
            sys.exit("no cubin in %s" % lib)
        # one cubin per architecture; the library is built for sm_100a only
        return subprocess.run(["nvdisasm", "--print-line-info-inline", os.path.join(d, cubins[0])], check=True,
                              capture_output=True, text=True).stdout


def resources(lib):
    out = subprocess.run(["cuobjdump", "-res-usage", lib], check=True, capture_output=True, text=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            res[name] = dict(re.findall(r"(REG|STACK):(\d+)", line))
            name = None
    return res


def parse(text, match):
    """{kernel: [(opcode, [(file, line), ...innermost first])]}"""
    kernels, cur, chain, fresh = {}, None, [], True
    for line in text.splitlines():
        m = SECTION.match(line)
        if m:
            cur = m.group(1) if match in m.group(1) else None
            if cur:
                kernels[cur] = []
            chain, fresh = [], True
            continue
        if cur is None:
            continue
        m = LOC.match(line)
        if m:
            # a group of location lines precedes each run of instructions: the first line of the group is the innermost
            if fresh:
                chain = []
                fresh = False
            chain.append((os.path.basename(m.group(1)), int(m.group(2))))
            continue
        m = INSN.match(line)
        if m:
            kernels[cur].append((m.group(1), chain))
            fresh = True
    return kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", nargs="?", default=os.path.join(ROOT, "mpcholonavigation_b200", "libmppi_b200.so"))
    ap.add_argument("--match", default="tile_fused")
    ap.add_argument("--lines", type=int, default=25, help="innermost source lines listed per kernel")
    ap.add_argument("--bucket", type=int, default=20, help="mppi_kernels.cuh line range per bucket")
    a = ap.parse_args()
    res = resources(a.lib)
    kernels = parse(disassemble(a.lib), a.match)
    print("%-72s %5s %5s %6s %5s %4s %4s %5s %4s" % ("kernel", "REG", "STACK", "SASS", "CALL", "LDL", "STL", "SHFL", "BAR"))
    for name, insns in sorted(kernels.items()):
        ops = collections.Counter(op.split(".")[0] for op, _ in insns)
        r = res.get(name, {})
        print("%-72s %5s %5s %6d %5d %4d %4d %5d %4d" % (
            name[:72], r.get("REG", "?"), r.get("STACK", "?"), len(insns), ops["CALL"], ops["LDL"], ops["STL"],
            ops["SHFL"], ops["BAR"]))
    for name, insns in sorted(kernels.items()):
        print("\n== %s: %d instructions" % (name, len(insns)))
        inner = collections.Counter(chain[0] if chain else ("?", 0) for _, chain in insns)
        print("  innermost source line                          insns")
        for (f, ln), n in inner.most_common(a.lines):
            print("  %-44s %6d" % ("%s:%d" % (f, ln), n))
        buckets = collections.Counter()
        for _, chain in insns:
            ln = next((l for f, l in chain if f == "mppi_kernels.cuh"), None)
            buckets[None if ln is None else (ln - 1) // a.bucket * a.bucket + 1] += 1
        print("  mppi_kernels.cuh lines                         insns")
        for lo in sorted(buckets, key=lambda k: -1 if k is None else k):
            label = "(no line)" if lo is None else "%d-%d" % (lo, lo + a.bucket - 1)
            print("  %-44s %6d" % (label, buckets[lo]))


if __name__ == "__main__":
    main()
