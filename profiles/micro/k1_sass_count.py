"""Static instruction count of K1's steady loop, no GPU needed.

Compiles csrc/step_global_d2.cu for sm_100a with the build's flags, disassembles
k_global_mcmc<2, 1, false, false, LAYOUT, false> (d = 2, ABS_NORMAL, FAST, native RNG, no dump) for
LAYOUT = TRACE_NONE, TRACE_TIME_MAJOR and TRACE_CHAIN_MAJOR and prints, per chain-step:
  steady   the 8-step ping-pong body (the innermost loop with the most MUFU), instructions outside
           BSSY..BSYNC regions divided by 8: the path without a trace flush;
  flushed  the chain-major tile loop around it: four bodies plus the fall-through path of the
           tile's flush (full warp, 16-byte aligned runs), divided by 32.  Equal to steady for the
           layouts without a tile.
plus the body's LDC / LDCU / S2R counts and ptxas' registers and spills of each kernel.

    python profiles/micro/k1_sass_count.py
"""
import collections
import importlib
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
build = importlib.import_module("gl-abc-mcmc_b200.build")
LAYOUTS = {"TRACE_NONE": 0, "TRACE_TIME_MAJOR": 1, "TRACE_CHAIN_MAJOR": 2}


def mangled(layout):
    return f"_ZN5glabc13k_global_mcmcILi2ELi1ELb0ELb0ELi{layout}ELb0EEEvNS_12GlobalConstsENS_9RunParamsE"


def opcode(text):
    t = text.split()
    return (t[1] if t[0].startswith("@") else t[0]).split(".")[0]


def parse(sass):
    ins = []
    for line in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2).strip()))
    return ins


def branch_target(text):
    m = re.search(r"\bBRA(?:\.\w+)*\s+(?:!?U?P\w+,\s*)?(0x[0-9a-f]+)", text)
    return int(m.group(1), 16) if m else None


def loops(ins):
    """(head index, back-edge index) of every backward branch"""
    where = {a: i for i, (a, _) in enumerate(ins)}
    out = []
    for i, (a, t) in enumerate(ins):
        tgt = branch_target(t)
        if tgt is not None and tgt < a and tgt in where:
            out.append((where[tgt], i))
    return out


def outside_bssy(body):
    depth, n = 0, []
    for t in body:
        op = opcode(t)
        if op == "BSSY":
            depth += 1
        elif op == "BSYNC":
            depth -= 1
        elif depth == 0:
            n.append(t)
    return n


def fall_through_path(ins, lo, hi, skip):
    """instructions executed from ins[lo] to the back-edge ins[hi], taking unconditional branches,
    falling through conditional ones and stepping over the index range `skip`"""
    where = {a: i for i, (a, _) in enumerate(ins)}
    i, n = lo, 0
    while i < hi:
        if skip[0] <= i <= skip[1]:
            i = skip[1] + 1
            continue
        a, t = ins[i]
        n += 1
        tgt = branch_target(t)
        if tgt is not None and re.match(r"BRA(\.U)?\s+0x", t):
            i = where[tgt]
        else:
            i += 1
    return n


def count(ins):
    ls = loops(ins)
    mufu = lambda lo, hi: sum(opcode(t) == "MUFU" for _, t in ins[lo:hi + 1])  # noqa: E731
    best = max(mufu(lo, hi) for lo, hi in ls)
    step = min((l for l in ls if mufu(*l) == best), key=lambda l: l[1] - l[0])
    body = [t for _, t in ins[step[0]:step[1] + 1]]
    steady = len(outside_bssy(body)) / 8
    enclosing = [l for l in ls if l[0] <= step[0] and l[1] > step[1]]
    flushed = steady
    if enclosing:
        lo, hi = min(enclosing, key=lambda l: l[1] - l[0])
        flushed = (4 * len(body) + fall_through_path(ins, lo, hi, step) + 1) / 32
    ops = collections.Counter(opcode(t) for t in body)
    return steady, flushed, {k: ops[k] for k in ("LDC", "LDCU", "S2R")}


def main():
    src = os.path.join(build.CSRC, "step_global_d2.cu")
    flags = [f for f in build.NVCC_FLAGS if f not in ("-Xcompiler", "-fPIC", "-fvisibility=hidden")]
    cuobjdump = os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "d2.cubin")
        p = subprocess.run([build._nvcc(), *flags, "-cubin", "-o", cubin, src], capture_output=True, text=True, check=True)
        ptxas = p.stderr + p.stdout
        print(f"{'layout':<20}{'steady':>8}{'flushed':>9}{'LDC':>5}{'LDCU':>6}{'S2R':>5}{'regs':>6}{'spill st/ld':>13}")
        for name, lay in LAYOUTS.items():
            fn = mangled(lay)
            sass = subprocess.run([cuobjdump, "-sass", "-fun", fn, cubin], capture_output=True, text=True, check=True).stdout
            steady, flushed, ops = count(parse(sass))
            m = re.search(re.escape(fn) + r"\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads"
                          r"[\s\S]*?Used (\d+) registers", ptxas)
            print(f"{name:<20}{steady:>8.2f}{flushed:>9.2f}{ops['LDC']:>5}{ops['LDCU']:>6}{ops['S2R']:>5}{m.group(4):>6}"
                  f"{m.group(2) + '/' + m.group(3):>13}")


if __name__ == "__main__":
    main()
