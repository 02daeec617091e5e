"""Registers, stack and spill instructions of every kernel in the shipped libkrotov_cuda.so (cuobjdump; no GPU needed).

    python tools/resource_usage.py > profiles/r2_resource_usage.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "krotov.jl_b200", "libkrotov_cuda.so")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    clean = [re.sub(r"\(anonymous namespace\)::|kr::|<unnamed>::", "", x) for x in out]
    return [re.sub(r"\((?:[^()]|\([^()]*\))*\)$", "", x) for x in clean]  # drop the parameter list


res = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
funcs, cur = [], None
for line in res.splitlines():
    m = re.match(r"\s*Function (\S+):", line)
    if m:
        cur = m.group(1)
        continue
    m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", line)
    if m and cur:
        funcs.append((cur,) + tuple(int(x) for x in m.groups()))
        cur = None

# spill instructions per function from the SASS
sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
spills, ops, cur = collections.Counter(), collections.defaultdict(collections.Counter), None
for line in sass.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        cur = m.group(1)
        continue
    m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", line)
    if m and cur:
        op = m.group(1)
        if op.startswith(("LDL", "STL")):
            spills[cur] += 1
        base = op.split(".")[0]
        if base in ("DFMA", "DMMA", "UBLKCP", "SYNCS", "LDS", "STS", "ATOMG", "REDG", "RED", "ATOM"):
            ops[cur][base] += 1

names = demangle([f[0] for f in funcs])
print(f"{len(funcs)} kernels in {os.path.relpath(LIB, ROOT)} (sm_100a); LDL/STL = local-memory (spill or stack-array) instructions in the SASS")
print(f"{'kernel':78s} {'REG':>4s} {'STACK':>6s} {'LDL/STL':>8s}  DFMA  DMMA  LDS  STS  bulk-copy  atom/red")
for (mangled, reg, stack, shared, local), name in sorted(zip(funcs, names), key=lambda t: t[1]):
    o = ops[mangled]
    print(f"{name[:78]:78s} {reg:4d} {stack:6d} {spills[mangled]:8d} {o['DFMA']:5d} {o['DMMA']:5d} {o['LDS']:4d} {o['STS']:4d} {o['UBLKCP']:10d} "
          f"{o['ATOMG'] + o['REDG'] + o['RED'] + o['ATOM']:9d}")
worst = max(spills.values()) if spills else 0
print(f"\nlargest LDL/STL count in one kernel: {worst}")

# ---- where the local-memory instructions of the C4 instance sit: address histogram of its SASS --------------------------
KEY = "_ZN2kr18krotov_warp_kernelILi6ELi2ELi256ELi32ELb0ELb0ELb0EEEvNS_10WarpParamsE"
k = subprocess.run(["cuobjdump", "-sass", "-fun", KEY, LIB], capture_output=True, text=True).stdout
ins = []
for line in k.splitlines():
    m = re.match(r"\s*/\*([0-9a-f]+)\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", line)
    if m:
        ins.append((int(m.group(1), 16), m.group(2)))
if ins:
    nb, top = 24, ins[-1][0] + 16
    H = [[0, 0, 0, 0] for _ in range(nb)]
    for a, op in ins:
        b = a * nb // top
        H[b][0] += op.startswith(("DFMA", "DMUL", "DADD"))
        H[b][1] += op.startswith(("LDL", "STL"))
        H[b][2] += op.startswith(("BAR", "WARPSYNC"))
        H[b][3] += op.startswith(("CALL", "RET"))
    print(f"\nkrotov_warp_kernel<6, 2, 256, 32> (the C4 instance), {len(ins)} instructions: where the LDL/STL sit.  The FP64-dense "
          "address ranges (the two sweeps of the trajectory warps) hold none; they belong to the comm warp's out-of-line exchange "
          "protocols (call ABI saves, small stack arrays) and the prologue.")
    print("bin  address range         FP64  LDL/STL  BAR/WARPSYNC  CALL/RET")
    for i, h in enumerate(H):
        print(f"{i:3d}  {hex(i * top // nb):>8s}-{hex((i + 1) * top // nb):>8s} {h[0]:6d} {h[1]:8d} {h[2]:13d} {h[3]:9d}")
    dense = [h for h in H if h[0] >= 60]
    print(f"bins with >= 60 FP64 instructions: {len(dense)}, LDL/STL inside them: {sum(h[1] for h in dense)}")

print("\nReading the table.  Every warp-kernel instance carries the comm warp and its out-of-line exchange protocols: 159-260 LDL/STL and "
      "192-370 bytes of stack come from there (see the histogram above), not from the sweeps.  The RF instances (last template flag "
      "true: backward sweep only, no comm warp) show the sweeps alone: 0 LDL/STL, STACK 0.  Instances ABOVE that baseline spill in the "
      "sweeps: the 64- and 128-thread-per-trajectory instances with 16-24 off-diagonal slots, which run 512 threads per CTA and are "
      "capped at 128 registers (306-609 LDL/STL).  They serve Hilbert spaces of 33-128 levels with unusually wide rows; narrow rows "
      "(W <= 12, the transmon cases of DESIGN.md 4.1) stay at the baseline.")
