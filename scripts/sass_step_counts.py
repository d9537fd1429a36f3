"""Instruction budget of the fused small-N kernels, read from the compiled objects (no GPU needed).

For every instantiation of small_fit_kernel and small_sweep_kernel in gpcc_b200/csrc/build/small_{fit,sweep}_k*.o it prints
  * registers, spill stores / loads and stack frame, from the ptxas log that the Makefile writes next to each object;
  * per sweep step segment, the counts of all instructions, LDL, STL, register moves (MOV and IMAD.MOV) and LDS;
  * the code size.
A sweep step segment is the code between two BAR.SYNC that holds the reciprocal of the next pivot (MUFU.RCP64H) and
64 to 79 DFMA (64 for the tile update, six for the Newton steps of the reciprocal); the eight specialised steps of
small_eval.cuh are eight such segments.  The stretches that hold the assembly, the gradient or thread 0's optimiser
hold many more DFMA (inlined exp, log, divisions).

    python scripts/sass_step_counts.py [--build DIR] [--kernel SUBSTRING]

--kernel keeps the instantiations whose short name (e.g. "small_fit_kernel<2,192,2,0>") contains SUBSTRING.
"""
import argparse
import glob
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = ("small_fit_kernel", "small_sweep_kernel")

_INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)(\.[A-Z0-9_.]+)?")
_FUNC = re.compile(r"^\s*Function : (\S+)")
_PTXAS_ENTRY = re.compile(r"Compiling entry function '(\S+)'")
_PTXAS_SPILL = re.compile(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads")
_PTXAS_REGS = re.compile(r"Used (\d+) registers")


def short_name(mangled):
    """small_fit_kernel<2,192,2,0> from the mangled name (the template arguments are all ints)."""
    for k in KERNELS:
        m = re.search(k + r"I((?:Li-?\d+E)+)E", mangled)
        if m:
            return "%s<%s>" % (k, ",".join(re.findall(r"Li(-?\d+)E", m.group(1))))
    return None


def ptxas_info(log):
    """{mangled name: (registers, spill store bytes, spill load bytes, stack frame bytes)} from one ptxas -v log."""
    out, cur = {}, None
    with open(log) as f:
        for line in f:
            m = _PTXAS_ENTRY.search(line)
            if m:
                cur = m.group(1)
                out[cur] = [None, 0, 0, 0]
                continue
            m = _PTXAS_SPILL.search(line)
            if m and cur:
                out[cur][1:] = [int(m.group(2)), int(m.group(3)), int(m.group(1))]
            m = _PTXAS_REGS.search(line)
            if m and cur:
                out[cur][0] = int(m.group(1))
    return {k: tuple(v) for k, v in out.items()}


def sass_functions(obj):
    """{mangled name: [(address, opcode, modifiers)]} of the kernels of interest in one object."""
    text = subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = _FUNC.match(line)
        if m:
            cur = m.group(1) if short_name(m.group(1)) else None
            if cur:
                funcs[cur] = []
            continue
        if cur is None:
            continue
        m = _INSN.match(line)
        if m:
            funcs[cur].append((int(m.group(1), 16), m.group(2), m.group(3) or ""))
    return funcs


def step_segments(insns):
    """Per sweep step segment: dict of instruction counts."""
    segs, seg = [], []
    for ins in insns:
        if ins[1] == "BAR" and ins[2].startswith(".SYNC"):
            segs.append(seg)
            seg = []
        else:
            seg.append(ins)
    out = []
    for s in segs[1:]:   # code before the first barrier is not between two of them
        ops = [o for _, o, _ in s]
        if 64 <= ops.count("DFMA") < 80 and any(o == "MUFU" and m.startswith(".RCP64H") for _, o, m in s):
            out.append({"insts": len(ops), "DFMA": ops.count("DFMA"), "LDL": ops.count("LDL"), "STL": ops.count("STL"),
                        "MOV": sum(o == "MOV" or (o == "IMAD" and m.startswith(".MOV")) for _, o, m in s),
                        "LDS": ops.count("LDS")})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--build", default=os.path.join(ROOT, "gpcc_b200", "csrc", "build"),
                    help="directory with small_{fit,sweep}_k*.o and their .ptxas.log")
    ap.add_argument("--kernel", default="", help="only instantiations whose short name contains this")
    a = ap.parse_args()
    objs = sorted(glob.glob(os.path.join(a.build, "small_fit_k*.o")) + glob.glob(os.path.join(a.build, "small_sweep_k*.o")))
    if not objs:
        sys.exit("no small_fit_k*.o / small_sweep_k*.o under %s: run make -C gpcc_b200/csrc first" % a.build)
    for obj in objs:
        info = ptxas_info(obj[:-2] + ".ptxas.log")
        for mangled, insns in sass_functions(obj).items():
            name = short_name(mangled)
            if a.kernel not in name:
                continue
            regs, sst, sld, stack = info.get(mangled, (None, None, None, None))
            size = (insns[-1][0] + 16) if insns else 0
            print("%-32s %-17s regs %3s  spill st/ld %4s/%4s B  stack %4s B  code %6.1f KB" % (
                name, os.path.basename(obj), regs, sst, sld, stack, size / 1024))
            for i, s in enumerate(step_segments(insns)):
                print("    step segment %d: %3d insts  DFMA %2d  LDL %2d  STL %2d  MOV %2d  LDS %2d" % (
                    i, s["insts"], s["DFMA"], s["LDL"], s["STL"], s["MOV"], s["LDS"]))


if __name__ == "__main__":
    main()
