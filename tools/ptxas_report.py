#!/usr/bin/env python
"""Compile csrc/capi.cu with -Xptxas -v and print registers / spills per k_step_fused<NOISE, RATE1, FULL, NT, REF> variant.
usage: tools/ptxas_report.py [-o out.so] [extra nvcc flags ...]"""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "binary-fluctuating-lattice-boltzmann_b200")
args = sys.argv[1:]
out = os.path.join(PKG, "libbflbm.so")
if "-o" in args:
    i = args.index("-o")
    out = args[i + 1]
    del args[i:i + 2]
cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--shared", "-Xcompiler", "-fPIC",
       "-Xptxas", "-v"] + args + [os.path.join(PKG, "csrc", "capi.cu"), os.path.join(PKG, "csrc", "multi.cu"), "-o", out]
r = subprocess.run(cmd, capture_output=True, text=True)
if r.returncode:
    sys.stderr.write(r.stderr)
    sys.exit(r.returncode)
cur = None
rows = {}
for ln in r.stderr.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", ln)
    if m:
        cur = m.group(1)
        rows[cur] = {}
        continue
    if cur is None:
        continue
    m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", ln)
    if m and "stack" not in rows[cur]:
        rows[cur]["stack"], rows[cur]["st"], rows[cur]["ld"] = map(int, m.groups())
    m = re.search(r"Used (\d+) registers", ln)
    if m:
        rows[cur]["regs"] = int(m.group(1))
for k, v in rows.items():
    m = re.search(r"k_step_fusedILb([01])ELb([01])ELb([01])ELi(\d+)ELb([01])E", k)
    if m:
        print(f"fused noise={m.group(1)} rate1={m.group(2)} full={m.group(3)} nt={m.group(4)} ref={m.group(5)}: regs {v.get('regs')} "
              f"stack {v.get('stack')} spill st/ld {v.get('st')}/{v.get('ld')}")
