#!/usr/bin/env python3
"""What the region stage's kernel compiles to, without a GPU.

Compiles linesegmentdetector-slam_b200/csrc/grow.cu with the package Makefile's flags (or reads a given object file and,
optionally, its ptxas log) and prints, for every instantiation of lsdb_grow_kernel:
  * instructions and bytes of the kernel and of the __noinline__ functions it calls (the call graph of CALL.REL targets);
  * stack frame and spills reported by ptxas (-Xptxas -v), for the kernel and per callee;
  * counts of LDL*, STL*, generic LD.E* (LD without a state space), LD.E.STRONG.SYS, LDG*, LDS* and CALL;
  * instructions, LDL and generic loads per source function of grow.cu, from nvdisasm -g line info (an inlined helper's
    instructions count for the helper, where its source lines are).

  python3 tools/sass_census.py                      # compile the tree's grow.cu into a temporary directory
  python3 tools/sass_census.py --obj grow.o [--log grow.ptxas.log]
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "linesegmentdetector-slam_b200")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def makefile_flags():
    """NVFLAGS of the package Makefile, with $(ARCH) expanded."""
    text = open(os.path.join(PKG, "Makefile")).read()
    arch = re.search(r"^ARCH\s*:=\s*(.*)$", text, re.M).group(1).strip()
    flags = re.search(r"^NVFLAGS\s*:=\s*(.*)$", text, re.M).group(1).strip()
    return flags.replace("$(ARCH)", arch).split()


def compile_grow(out_dir):
    obj = os.path.join(out_dir, "grow.o")
    cmd = [os.path.join(CUDA, "bin", "nvcc")] + makefile_flags() + ["-c", "-o", obj, os.path.join(PKG, "csrc", "grow.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.exit(r.stdout + r.stderr)
    return obj, r.stdout + r.stderr


def ptxas_props(log):
    """mangled name -> (stack frame, spill stores, spill loads, registers or None)"""
    props, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            props[cur] = [int(m.group(1)), int(m.group(2)), int(m.group(3)), None]
            continue
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in props:
            props[cur][3] = int(m.group(1))
    return props


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return dict(zip(names, r.stdout.splitlines())) if r.returncode == 0 else {n: n for n in names}


def source_functions(path):
    """[(first line, name)] of the functions (and structs) defined at column 0 of a source file"""
    out, pending = [], None
    for i, line in enumerate(open(path).read().splitlines(), 1):
        if line.startswith("template"):
            pending = pending or i
            continue
        m = re.match(r"struct (\w+)\s*\{", line)
        if m:
            out.append((pending or i, m.group(1)))
        elif re.match(r"(__device__|__global__|__host__|static|void|int|size_t|LSDM_FN)\b", line) and "(" in line and not line.rstrip().endswith(";"):
            name = re.findall(r"(\w+)\s*\(", line.split("(")[0] + "(")
            if name and name[-1] not in ("__launch_bounds__",):
                out.append((pending or i, name[-1]))
            else:
                m2 = re.search(r"(\w+)\s*\(int nImgs", line)
                if m2:
                    out.append((pending or i, m2.group(1)))
        pending = None
    return sorted(out)


def classify(op):
    c = []
    if op.startswith("LDL"): c.append("LDL")
    if op.startswith("STL"): c.append("STL")
    if op.startswith("LDG"): c.append("LDG")
    if op.startswith("LDS"): c.append("LDS")
    if op == "LD" or op.startswith("LD."):
        c.append("LD.E")   # generic: no state space in the opcode
        if ".STRONG.SYS" in op: c.append("LD.E.STRONG.SYS")
    if op.startswith("CALL"): c.append("CALL")
    return c


def disassemble(obj, work):
    subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", os.path.abspath(obj)], cwd=work, check=True, capture_output=True)
    cubins = [f for f in os.listdir(work) if f.endswith(".cubin") and "grow" in f]
    if not cubins:
        sys.exit("no cubin in " + obj)
    r = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-g", "-c", os.path.join(work, cubins[0])],
                       capture_output=True, text=True, check=True)
    funcs = collections.OrderedDict()   # mangled -> list of (opcode, file, line, call target)
    cur, loc = None, (None, 0)
    for line in r.stdout.splitlines():
        m = re.match(r"\s*\.section\s+\.text\.(\S+?),", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)', line)
        if m:
            loc = (os.path.basename(m.group(1)), int(m.group(2)))
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)(.*);", line)
        if m and cur is not None:
            op, rest = m.group(1), m.group(2)
            tgt = None
            if op.startswith("CALL"):
                t = re.search(r"`\(([^)]+)\)", rest)
                tgt = t.group(1) if t else None
            funcs[cur].append((op, loc[0], loc[1], tgt))
    return funcs


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--obj", help="an object file built from grow.cu (default: compile the tree's grow.cu)")
    ap.add_argument("--log", help="the ptxas -v log of that object (the Makefile writes build/grow.ptxas.log)")
    ap.add_argument("--src", default=os.path.join(PKG, "csrc", "grow.cu"), help="grow.cu the object was built from (line info)")
    ap.add_argument("--top", type=int, default=14, help="source functions listed per instantiation")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as work:
        if a.obj:
            obj, log = a.obj, open(a.log).read() if a.log else ""
        else:
            obj, log = compile_grow(work)
        funcs = disassemble(obj, work)
    props = ptxas_props(log)
    names = demangle(list(funcs))
    srcf = source_functions(a.src)
    src_name = os.path.basename(a.src)

    def owner(fname, line):
        if fname != src_name:
            return fname
        best = "?"
        for first, nm in srcf:
            if first <= line:
                best = nm
            else:
                break
        return best

    def closure(root):
        seen, todo = [], [root]
        while todo:
            f = todo.pop()
            if f in seen or f not in funcs:
                continue
            seen.append(f)
            todo.extend(t for (_, _, _, t) in funcs[f] if t)
        return seen

    kernels = [f for f in funcs if names[f].startswith("void lsdb_grow_kernel")]
    for k in kernels:
        fs = closure(k)
        tot = collections.Counter()
        n = 0
        per_src = collections.defaultdict(collections.Counter)
        print("== %s" % names[k].split("(")[0])
        p = props.get(k)
        if p:
            print("   kernel: %d registers, %d B stack frame, %d B spill stores, %d B spill loads" % (p[3] or 0, p[0], p[1], p[2]))
        print("   %-44s %7s %5s %5s %5s %5s %5s %5s %5s %5s  %s" % ("function (SASS)", "instr", "LDL", "STL", "LD.E", ".SYS", "LDG", "LDS", "CALL", "frame", "spill st/ld"))
        for f in fs:
            c = collections.Counter()
            for op, fn, ln, _ in funcs[f]:
                for cl in classify(op):
                    c[cl] += 1
                    per_src[owner(fn, ln)][cl] += 1
                per_src[owner(fn, ln)]["instr"] += 1
            tot.update(c)
            n += len(funcs[f])
            pf = props.get(f)
            frame = "%d" % pf[0] if pf else "-"
            spill = "%d/%d" % (pf[1], pf[2]) if pf else "-"
            nm = names[f].split("(")[0] if f != k else "(kernel body)"
            print("   %-44s %7d %5d %5d %5d %5d %5d %5d %5d %5s  %s" % (nm[:44], len(funcs[f]), c["LDL"], c["STL"], c["LD.E"], c["LD.E.STRONG.SYS"],
                                                                   c["LDG"], c["LDS"], c["CALL"], frame, spill))
        print("   %-44s %7d %5d %5d %5d %5d %5d %5d %5d   (%d bytes)" % ("total", n, tot["LDL"], tot["STL"], tot["LD.E"], tot["LD.E.STRONG.SYS"],
                                                                  tot["LDG"], tot["LDS"], tot["CALL"], 16 * n))
        print("   per source function (line info):  %-26s %7s %5s %5s %5s %5s" % ("", "instr", "LDL", "STL", "LD.E", "LDG"))
        for nm, c in sorted(per_src.items(), key=lambda kv: -kv[1]["instr"])[:a.top]:
            print("     %-58s %7d %5d %5d %5d %5d" % (nm, c["instr"], c["LDL"], c["STL"], c["LD.E"], c["LDG"]))
        print()


if __name__ == "__main__":
    main()
