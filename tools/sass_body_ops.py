"""Static SASS opcode count of one inlined device function inside one kernel, from a -lineinfo build.

    python tools/sass_body_ops.py OBJ KERNEL_SUBSTRING SOURCE.cu FUNCTION [FUNCTION ...]

OBJ is an object file or cubin compiled with -lineinfo (fiksi_b200/csrc/build/lm_sketch.o).  An instruction counts for
FUNCTION when its inline chain (nvdisasm -gi) passes through a line of FUNCTION's definition in SOURCE.cu, so the loads and
stores of helpers it calls count with it.  Example (the warp-pair kernel's column body):
    python tools/sass_body_ops.py fiksi_b200/csrc/build/lm_sketch.o sketch_pair_kernel fiksi_b200/csrc/lm_sketch.cu sk_column_half"""
import collections
import os
import re
import subprocess
import sys
import tempfile

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def line_range(src, func):
    lines = open(src).read().split("\n")
    for i, l in enumerate(lines):
        if re.match(r"__device__ .*\b" + re.escape(func) + r"\(", l):
            for j in range(i, len(lines)):
                if lines[j] == "}":
                    return i + 1, j + 1
    raise SystemExit(f"{func}: no definition in {src}")


def disassemble(obj):
    if obj.endswith(".cubin"):
        cubins = [obj]
    else:
        tmp = tempfile.mkdtemp()
        subprocess.run([f"{CUDA}/bin/cuobjdump", "-xelf", "all", os.path.abspath(obj)], cwd=tmp, check=True, capture_output=True)
        cubins = [os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin")]
    out = []
    for c in cubins:
        out += subprocess.run([f"{CUDA}/bin/nvdisasm", "-gi", "-c", c], check=True, capture_output=True, text=True).stdout.split("\n")
    return out


def count(asm, kernel, src_name, lo, hi):
    on = inr = False
    in_group = False
    c = collections.Counter()
    for l in asm:
        if ".section" in l and ".text." in l:
            on = kernel in l
        if "//##" in l:  # one instruction's inline chain, innermost frame first
            if not in_group:
                inr = False
            in_group = True
            for m in re.finditer(re.escape(src_name) + r'", line (\d+)', l):
                inr = inr or lo <= int(m.group(1)) <= hi
            continue
        in_group = False
        if on and inr:
            m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_]+)", l)
            if m:
                c[m.group(1)] += 1
    return c


def main():
    obj, kernel, src, funcs = sys.argv[1], sys.argv[2], sys.argv[3], sys.argv[4:]
    asm = disassemble(obj)
    for f in funcs:
        lo, hi = line_range(src, f)
        c = count(asm, kernel, os.path.basename(src), lo, hi)
        print(f"{f} (lines {lo}-{hi}) in *{kernel}*: {sum(c.values())} instructions  " + " ".join(f"{k} {v}" for k, v in c.most_common()))


if __name__ == "__main__":
    main()
