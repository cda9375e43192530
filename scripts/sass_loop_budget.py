#!/usr/bin/env python3
"""Instruction budget of the f32 event loop of the simulate kernel, read from the SASS (no GPU needed).

Cross-compiles the f32 translation units of the simulate kernel for sm_100a with the library's nvcc flags (which include
`-Xptxas -v`) into a temporary directory. In each selected `pf_sim_weight_kernel` instantiation it finds the event loop:
the innermost backward branch whose body contains the warp vote of the work queue (`VOTE.ANY`). It then prints the loop's
SASS instruction count, the kernel's registers and its spill bytes.

    python scripts/sass_loop_budget.py                   # the working tree, plain-mode f32 kernels
    python scripts/sass_loop_budget.py --rev HEAD~1      # the same for a commit (git archive into the temporary directory)
    python scripts/sass_loop_budget.py --match "SIR I8 plain ilp1" --show   # also print the loop's SASS

The count is static: every instruction of the loop body once, whether or not a path is taken in a given iteration.
"""
from __future__ import annotations

import argparse
import importlib.util
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TUS = ["pf_sim_f32.cu", "pf_sim_count_f32.cu"]
MODELS = {0: "generic", 1: "SI", 2: "SIR", 3: "SIS", 4: "SEI", 5: "SEIR", 6: "SEIS", 7: "LOTKA", -1: "count"}
MODES = {0: "plain", 1: "fused", 2: "persist"}
KERNEL = "_ZN5dpomp20pf_sim_weight_kernelI"


def load_build(src: str):
    spec = importlib.util.spec_from_file_location("dpomp_build_src", os.path.join(src, "discretepomp.jl_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def compile_tu(build, src: str, tu: str, out: str):
    obj = os.path.join(out, tu.replace(".cu", ".o"))
    cmd = [build._nvcc(), *build.NVCC_FLAGS, *build._host_cxx_args(), "-c",
           os.path.join(src, "discretepomp.jl_b200", "csrc", tu), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed for {tu}:\n{res.stderr}")
    sass = subprocess.run([os.path.join(os.path.dirname(build._nvcc()), "cuobjdump"), "-sass", obj],
                          capture_output=True, text=True, check=True).stdout
    return res.stdout + res.stderr, sass


def ptxas_resources(log: str) -> dict:
    """entry function -> (registers, spill store bytes, spill load bytes)"""
    out, cur, spill = {}, None, (0, 0)
    for line in log.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            spill = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out[cur] = (int(m.group(1)), *spill)
            cur, spill = None, (0, 0)
    return out


def sass_functions(sass: str) -> dict:
    """function -> [(address, instruction text)]"""
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), m.group(2).strip()))
    return funcs


def event_loop(ins):
    """(first, last) index of the innermost backward-branch loop containing VOTE.ANY, or None"""
    addr = {a: i for i, (a, _) in enumerate(ins)}
    best = None
    for j, (a, text) in enumerate(ins):
        m = re.search(r"\bBRA(?:\.\w+)*\s+(?:!?U?P\d,\s*)?(0x[0-9a-f]+)", text)
        if not m or int(m.group(1), 16) > a:
            continue
        i = addr.get(int(m.group(1), 16))
        if i is None or not any("VOTE.ANY" in t for _, t in ins[i:j + 1]):
            continue
        if best is None or j - i < best[1] - best[0]:
            best = (i, j)
    return best


def label(name: str) -> str:
    # template arguments <Real, C, E, ITEMS, MODEL, MODE, ILP>: "fLi3ELi2ELi8ELi2ELi0ELi1EEEv..." ("n" = minus)
    tpl = name[len(KERNEL):].split("EEv")[0]
    c, e, items, model, mode, ilp = [int(v.replace("n", "-")) for v in re.findall(r"Li(n?\d+)", tpl)][:6]
    real = "f32" if tpl[0] == "f" else "f64"
    return f"{real} C{c} E{e} I{items} {MODELS.get(model, model)} {MODES.get(mode, mode)} ilp{ilp}"


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rev", help="git revision to measure instead of the working tree")
    ap.add_argument("--match", action="append", default=[],
                    help="substring of the label ('f32 C3 E2 I8 SIR plain ilp1'); repeatable; default: every plain-mode kernel")
    ap.add_argument("--all-modes", action="store_true", help="include the fused and persistent instantiations")
    ap.add_argument("--show", action="store_true", help="print the SASS of each selected loop")
    args = ap.parse_args()

    with tempfile.TemporaryDirectory(prefix="sass_loop_budget_") as tmp:
        src = ROOT
        if args.rev:
            src = os.path.join(tmp, "src")
            os.makedirs(src)
            subprocess.run(f"git -C '{ROOT}' archive '{args.rev}' | tar -x -C '{src}'", shell=True, check=True)
        build = load_build(src)
        with ThreadPoolExecutor(max_workers=len(TUS)) as ex:
            results = list(ex.map(lambda tu: compile_tu(build, src, tu, tmp), TUS))
    rows = []
    for log, sass in results:
        res = ptxas_resources(log)
        for name, ins in sass_functions(sass).items():
            if not name.startswith(KERNEL + "f"):
                continue
            lab = label(name)
            if args.match and not any(m in lab for m in args.match):
                continue
            if not args.match and not args.all_modes and " plain " not in lab:
                continue
            loop = event_loop(ins)
            regs, st, ld = res.get(name, (None, None, None))
            rows.append((lab, loop[1] - loop[0] + 1 if loop else None, regs, st, ld, name, ins, loop))
    print(f"source: {args.rev or 'working tree'}; nvcc flags: {' '.join(build.NVCC_FLAGS)}")
    print(f"{'kernel':40s} {'loop':>5s} {'regs':>5s} {'spill st/ld':>12s}")
    for lab, n, regs, st, ld, name, ins, loop in sorted(rows):
        print(f"{lab:40s} {n if n is not None else '-':>5} {regs if regs is not None else '-':>5} {f'{st}/{ld}':>12s}")
        if args.show and loop:
            print(f"  {name}")
            for a, t in ins[loop[0]:loop[1] + 1]:
                print(f"    {a:05x}  {t}")
    return 0 if rows else 1


if __name__ == "__main__":
    sys.exit(main())
