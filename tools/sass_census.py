"""Instruction census of the render kernel's instantiations, compiled for sm_100a (CPU only, needs nvcc).

  python tools/sass_census.py                       # this tree
  python tools/sass_census.py --rev HEAD~1          # ... and the difference to a git revision
  python tools/sass_census.py -D RT_NODE_PLANAR=1   # extra nvcc defines (applied to both builds)

For every render_kernel instantiation: registers, stack frame and spill stores / loads (ptxas -v), the number of
SASS instructions, the FP32 opcodes (FFMA / FFMA2 / FMUL / FMUL2 / FADD / FADD2 / FMNMX / FMNMX3), and the same
FP32 counts for the instructions whose source line is inside load_node or node_step (rt_device.cuh), the node step: the packed slab arithmetic
that must not silently fall back to scalar FFMA.  The compile flags are build()'s (__graft_entry__.NVCC_FLAGS)."""
import argparse
import collections
import os
import re
import subprocess
import sys
import tarfile
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = ("FFMA", "FFMA2", "FMUL", "FMUL2", "FADD", "FADD2", "FMNMX", "FMNMX3")
FLAGS = ("COUNT", "ALL_SMEM", "SSTACK", "AOV", "COOP", "VIEWS")
PRODUCTION = "render_kernel<0,1,0,0,0,0>"  # the plan of the headline scene: staged BVH and leaves, local stack


def _nvcc_flags():
    sys.path.insert(0, ROOT)
    from __graft_entry__ import NVCC_FLAGS
    out, skip = [], False
    for f in NVCC_FLAGS:  # a cubin: no host compiler flags, no shared library
        if skip:
            skip = False
        elif f == "-Xcompiler":
            skip = True
        elif f != "-shared":
            out.append(f)
    return out


def _region(src_file, func):
    """(first, last) source line of the definition of device function `func` in `src_file`."""
    lines = open(src_file).read().splitlines()
    first = next(i for i, l in enumerate(lines) if re.search(r"\b%s\(" % func, l) and "__device__" in l)
    last = next(i for i in range(first, len(lines)) if lines[i].startswith("}"))
    return first + 1, last + 1


def _pretty(mangled):
    args = re.findall(r"Lb([01])E", mangled)
    return "render_kernel<%s>" % ",".join(args)


def census(tree, defines=()):
    """{instantiation: {field: count}} of the render kernels of the sources under `tree`."""
    csrc = os.path.join(tree, "raytracing-practice_b200", "csrc")
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "rt_b200.cubin")
        cmd = ["nvcc", "-cubin", *_nvcc_flags(), "-Xptxas", "-v", *["-D" + d for d in defines], "-I", os.path.join(tree, "include"),
               os.path.join(csrc, "rt_b200.cu"), "-o", cubin]
        ptxas = subprocess.run(cmd, check=True, capture_output=True, text=True).stderr
        sass = subprocess.run(["nvdisasm", "--print-line-info", cubin], check=True, capture_output=True, text=True).stdout
    res = {}
    for block in re.split(r"Compiling entry function", ptxas)[1:]:
        name = re.search(r"'(\w+)'", block).group(1)
        if "render_kernel" not in name:
            continue
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        frame, sst, sld = map(int, re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block).groups())
        res[name] = collections.Counter(regs=regs, stack=frame, spill_st=sst, spill_ld=sld)
    # a node step is load_node + node_step; load_node does no FP arithmetic, but the packed FFMA2 that follow its loads
    # carry the line of their CUDA header and so inherit its region
    regions = [_region(os.path.join(csrc, "rt_device.cuh"), f) for f in ("load_node", "node_step")]
    fn, in_step = None, False
    for line in sass.splitlines():
        m = re.match(r"\.text\.(\w+):", line)
        if m:
            fn = m.group(1) if m.group(1) in res else None
            continue
        if fn is None:
            continue
        m = re.search(r'## File "([^"]+)", line (\d+)', line)
        if m:
            # an intrinsic's instructions carry the line of its CUDA header (crt/sm_100_rt.hpp): they stay in the region
            # of the project line that precedes them
            if "/crt/" not in m.group(1):
                in_step = m.group(1).endswith("rt_device.cuh") and any(lo <= int(m.group(2)) <= hi for lo, hi in regions)
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9]*)", line)
        if not m:
            continue
        op = m.group(1)
        c = res[fn]
        c["instrs"] += 1
        if op in OPS:
            c[op] += 1
            if in_step:
                c["step_" + op] += 1
    return {_pretty(k): v for k, v in res.items()}


def _revision_tree(rev, tmp):
    data = subprocess.run(["git", "-C", ROOT, "archive", rev], check=True, capture_output=True).stdout
    path = os.path.join(tmp, "tree")
    os.makedirs(path)
    with tempfile.TemporaryFile() as f:
        f.write(data)
        f.seek(0)
        with tarfile.open(fileobj=f) as t:
            t.extractall(path, filter="data")
    return path


COLS = ["regs", "stack", "spill_st", "spill_ld", "instrs", *OPS, *("step_" + o for o in OPS if o.startswith(("FFMA", "FMNMX")))]


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rev", help="git revision to compare against")
    ap.add_argument("-D", dest="defines", action="append", default=[], help="extra preprocessor define, e.g. RT_NODE_PLANAR=1")
    args = ap.parse_args()
    cur = census(ROOT, args.defines)
    old = None
    if args.rev:
        with tempfile.TemporaryDirectory() as tmp:
            old = census(_revision_tree(args.rev, tmp), args.defines)
    print("instantiation <" + ",".join(FLAGS) + ">" + (f"   (new, or old->new against {args.rev})" if old else ""))
    print(f"{'':28s}" + "".join(f"{c:>12s}" for c in COLS))
    for name in sorted(cur):
        row = []
        for c in COLS:
            v = cur[name][c]
            if old is not None and name in old and old[name][c] != v:
                row.append(f"{old[name][c]}->{v}")
            else:
                row.append(str(v))
        mark = " *" if name == PRODUCTION else ""
        print(f"{name + mark:28s}" + "".join(f"{r:>12s}" for r in row))
    if old is not None:
        for name in sorted(set(old) - set(cur)):
            print(f"{name:28s} only in {args.rev}")


if __name__ == "__main__":
    main()
