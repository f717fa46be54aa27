"""SASS opcode histogram, registers / spills and the geodesic step loop of kernels in a built object (CPU only).

    python tools/sass_ops.py bendy_tracer_b200/csrc/kernels.o 'render_pool_kernel<true, false, 1, 25>' 'integrate_kernel<false, 1>'

A kernel is picked by a substring of its demangled name (all kernels when none is given).  Registers and spills come
from the ptxas log next to the object (`kernels.o` -> `kernels.ptxas.log`; `--log` to name another).  For each loop
(a backward branch and its target) that holds at least four MUFU.RSQ -- the RK4 stages of a step -- and 40 FFMA / FFMA2,
the smallest such loop is the step loop: the script prints its size and the instructions from its first to its last MUFU.RSQ ("rsq span"), with their opcode histograms:
for integrate_kernel the loop is one bare M-mass step, for the render kernels the span is the step with its bookkeeping.
"""
import argparse
import collections
import os
import re
import subprocess
import sys

INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_]+)(\.[A-Z0-9_.]+)?\s*([^;]*);")
FUNC = re.compile(r"Function : (\S+)")
FP = ("FFMA", "FFMA2", "FMUL", "FMUL2", "FADD", "FADD2", "MUFU", "MOV", "IMAD.MOV", "FMNMX")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def short(name):
    m = re.search(r"(\w+<[^>]*>)\(", name)
    return m.group(1) if m else name


def sass_functions(obj):
    text = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = FUNC.search(line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = INSN.search(line)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), m.group(3), (m.group(4) or ""), m.group(5)))
    return funcs


def ptxas_info(log):
    info, name, spill = {}, None, None
    if not os.path.exists(log):
        return info
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            spill = (int(m.group(1)), int(m.group(2)), int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            info[name] = (int(m.group(1)),) + (spill or (0, 0, 0))
            spill = None
    return info


def hist(insns):
    # IMAD.MOV is a register move issued on the FMA pipe: counted with the moves, not the multiplies
    return collections.Counter("IMAD.MOV" if op == "IMAD" and mod.startswith(".MOV") else op for _, op, mod, _ in insns)


def fmt(h):
    keys = [k for k in FP if h.get(k)] + sorted(k for k in h if k not in FP and k != "NOP")
    return ", ".join(f"{k} {h[k]}" for k in keys)


def step_loop(insns):
    """the smallest loop (backward branch -> target) holding >= 4 MUFU.RSQ and >= 40 FFMA / FFMA2: the STEP loop"""
    addr_ix = {a: i for i, (a, _, _, _) in enumerate(insns)}
    loops = []
    for i, (a, op, mod, args) in enumerate(insns):
        if op != "BRA":
            continue
        m = re.search(r"0x([0-9a-f]+)\s*$", args)
        if not m:
            continue
        t = int(m.group(1), 16)
        if t <= a and t in addr_ix:
            body = insns[addr_ix[t]:i + 1]
            h = hist(body)
            rsq = sum(1 for x in body if x[1] == "MUFU" and x[2].startswith(".RSQ"))
            if rsq >= 4 and h["FFMA"] + h["FFMA2"] >= 40:
                loops.append((i - addr_ix[t], addr_ix[t], i))
    return [min(loops)[1:]] if loops else []


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("obj", help="a built .o or .so")
    ap.add_argument("kernels", nargs="*", help="substrings of demangled kernel names (default: all)")
    ap.add_argument("--log", help="ptxas -v log (default: <obj stem>.ptxas.log)")
    a = ap.parse_args()
    funcs = sass_functions(a.obj)
    names = demangle(list(funcs))
    info = ptxas_info(a.log or os.path.splitext(a.obj)[0] + ".ptxas.log")
    found = False
    for mangled, insns in funcs.items():
        dem = names[mangled]
        if a.kernels and not any(k in dem for k in a.kernels):
            continue
        found = True
        insns = [x for x in insns if x[1] != "NOP"]
        print(f"== {short(dem)}")
        if mangled in info:
            r, stack, ss, sl = info[mangled]
            print(f"   registers {r}, stack {stack} B, spill stores {ss} B, spill loads {sl} B")
        print(f"   kernel: {len(insns)} instructions: {fmt(hist(insns))}")
        for s, e in step_loop(insns):
            body = insns[s:e + 1]
            rsq = [i for i, x in enumerate(body) if x[1] == "MUFU" and x[2].startswith(".RSQ")]
            span = body[rsq[0]:rsq[-1] + 1]
            print(f"   loop {body[0][0]:#x}-{body[-1][0]:#x}: {len(body)} instructions, {len(rsq)} MUFU.RSQ: {fmt(hist(body))}")
            print(f"     rsq span: {len(span)} instructions: {fmt(hist(span))}")
    if not found:
        sys.exit(f"no kernel matches {a.kernels}")


if __name__ == "__main__":
    main()
