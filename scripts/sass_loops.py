"""Registers, spills and per-loop SASS opcode counts of one kernel of one translation unit.

    python scripts/sass_loops.py kern_step_pcp.cu "step_thread_kernel<0,4>" "step_thread_kernel<0,3>"

Compiles the unit with marbler_b200/build.py's flags (plus -Xptxas -v) into a temporary directory, disassembles the
cubin with line information and lists every loop of the kernel: the instructions between a backward branch and its
target.  Each loop is named by the source line of its backward branch (e.g. the `for` of the IPM iteration in
qp_dual.cuh), so a census can be compared across builds without reading the SASS.  Needs nvcc, cuobjdump, nvdisasm
and cu++filt from the CUDA toolkit, no GPU.
"""
import argparse
import collections
import os
import re
import shutil
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from marbler_b200 import build as mb  # noqa: E402

OPS = ("DFMA", "DMUL", "DADD", "MUFU", "DSETP", "FSEL", "LDL", "STL", "LDS", "STS")
INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)(\.[\w.]+)?\s*([^;]*);")
LABEL = re.compile(r"^(\.L_x_\d+):")
LINE = re.compile(r'//## File "([^"]+)", line (\d+)')
TARGET = re.compile(r"`\((\.L_x_\d+)\)")


def tool(name):
    path = shutil.which(name) or os.path.join("/usr/local/cuda/bin", name)
    if not os.path.exists(path):
        sys.exit("sass_loops: %s not found" % name)
    return path


def demangle(names):
    out = subprocess.run([tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def norm(s):
    """'void mrb::k<(int)0, (int)4>(...)' -> 'mrb::k<0,4>'"""
    s = re.sub(r"\((int|bool|unsigned int|long)\)", "", s.replace(" ", "").replace("void", "", 1))
    return s.split("(")[0]


def compile_unit(unit, tmp):
    src = unit if os.path.isabs(unit) else os.path.join(mb.CSRC, unit)
    obj = os.path.join(tmp, "unit.o")
    flags = [f for f in mb.NVCC_FLAGS if f != "-shared"]
    res = subprocess.run([tool("nvcc")] + flags + ["-Xptxas", "-v", "-c", "-o", obj, src], capture_output=True, text=True)
    if res.returncode != 0:
        sys.exit(res.stdout + res.stderr)
    # ptxas -v: "Compiling entry function 'X'" / "Function properties for X", then "N bytes stack frame, S bytes spill
    # stores, L bytes spill loads" and "Used R registers"
    info, cur = {}, None
    for ln in res.stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?(\w+)'?", ln)
        if m:
            cur = m.group(1)
            info.setdefault(cur, {})
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", ln)
        if m:
            info[cur].update(stack=int(m.group(1)), spill_st=int(m.group(2)), spill_ld=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", ln)
        if m:
            info[cur]["regs"] = int(m.group(1))
    subprocess.run([tool("cuobjdump"), "-xelf", "all", obj], cwd=tmp, capture_output=True, check=True)
    cubin = next(os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin"))
    sass = subprocess.run([tool("nvdisasm"), "-g", "-c", cubin], capture_output=True, text=True, check=True).stdout
    return info, sass


def kernel_text(sass, mangled):
    lines, on = [], False
    for ln in sass.splitlines():
        if ln.startswith(".text."):
            on = ln[len(".text."):].rstrip(":") == mangled
            continue
        if on:
            lines.append(ln)
    return lines


def parse(lines):
    """-> list of (addr, opcode, operands, src) and {label: addr}"""
    insns, labels, pending, src = [], {}, [], ("?", 0)
    for ln in lines:
        m = LINE.search(ln)
        if m:
            src = (os.path.basename(m.group(1)), int(m.group(2)))
            continue
        m = LABEL.match(ln.strip())
        if m:
            pending.append(m.group(1))
            continue
        m = INSN.search(ln)
        if m:
            addr = int(m.group(1), 16)
            for lb in pending:
                labels[lb] = addr
            pending = []
            insns.append((addr, m.group(3), m.group(5), src))
    return insns, labels


def census(insns):
    c = collections.Counter(op for _, op, _, _ in insns)
    return len(insns), c


def fmt(total, c):
    return "%5d insns  " % total + "  ".join("%s %d" % (op, c[op]) for op in OPS)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("unit", help="translation unit under marbler_b200/csrc (or a path)")
    ap.add_argument("kernel", nargs="+", help="demangled name without parameters, spaces ignored: 'step_thread_kernel<0,4>'")
    ap.add_argument("--min", type=int, default=20, help="list loops of at least this many instructions (default 20)")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory(prefix="sass_loops_") as tmp:
        info, sass = compile_unit(a.unit, tmp)
    names = demangle([k for k, d in info.items() if "regs" in d])
    for want in a.kernel:
        hits = [k for k, d in names.items() if norm(d) == norm(want) or norm(d).endswith("::" + norm(want))]
        if len(hits) != 1:
            sys.exit("sass_loops: %d kernels match %r; kernels of this unit:\n  %s"
                     % (len(hits), want, "\n  ".join(sorted(norm(d) for d in names.values()))))
        report(names[hits[0]], info[hits[0]], kernel_text(sass, hits[0]), a.min)


def report(name, d, text, min_len):
    print("%s\n  %d registers, %d bytes stack, %d bytes spill stores, %d bytes spill loads"
          % (name, d.get("regs", -1), d.get("stack", -1), d.get("spill_st", -1), d.get("spill_ld", -1)))
    insns, labels = parse(text)
    print("  whole kernel  " + fmt(*census(insns)))
    index = {addr: i for i, (addr, _, _, _) in enumerate(insns)}
    for i, (addr, op, args, src) in enumerate(insns):
        if op != "BRA":
            continue
        t = TARGET.search(args)
        if not (t and t.group(1) in labels and labels[t.group(1)] <= addr):
            continue
        lo = index[labels[t.group(1)]]
        body = insns[lo:i + 1]
        if len(body) >= min_len:
            print("  loop %s:%d [%04x-%04x]  %s" % (src[0], src[1], insns[lo][0], addr, fmt(*census(body))))


if __name__ == "__main__":
    main()
