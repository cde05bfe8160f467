"""Opcode histogram per kernel of libbdlm.so (cuobjdump -sass), committed under profiles/.

    python tools/sass_histogram.py > profiles/r2_sass_opcodes.txt
    python tools/sass_histogram.py [lib.so] --loops 'kf_small_kernel<2, true, 3, false>'

--loops SUBSTRING: for each kernel whose name contains SUBSTRING, the same columns for every loop
body (a backward branch and the instructions it jumps back over) instead of the whole kernel.

What to look for (B200_PROFILING.md): LDGSTS = cp.async staging, UTMALDG / UBLKCP = TMA,
UTC*MMA / LDTM = tcgen05, HMMA / DMMA = legacy tensor path.  This path is fp64 recursions at
0.6 flop/B (config 2) or small dense fp64 chains (configs 3, 4): no tensor-core instruction is
expected; the FP64 pipe (DADD / DMUL / DFMA) and the memory pipes are what matter."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
args = sys.argv[1:]
loops = None
if "--loops" in args:
    i = args.index("--loops")
    loops = args[i + 1]
    del args[i:i + 2]
so = args[0] if args else os.path.join(ROOT, "bayesian_dlms_b200", "libbdlm.so")
out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
kern, code = None, collections.OrderedDict()  # kernel -> [(address, opcode, branch target)]
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        kern = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        kern = re.sub(r"\(anonymous namespace\)::|bdlm::", "", kern)
        code[kern] = []
        continue
    m = re.search(r"/\*([0-9a-f]{4,6})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)([^;]*)", line)
    if m and kern:
        tgt = re.search(r"0x([0-9a-f]+)\s*$", m.group(3)) if m.group(2) == "BRA" else None
        code[kern].append((int(m.group(1), 16), m.group(2), int(tgt.group(1), 16) if tgt else None))
hist = collections.OrderedDict()
for k, ins in code.items():
    if loops is None:
        hist[k] = collections.Counter(op for _, op, _ in ins)
    elif loops in k:
        for a, _, tgt in ins:
            if tgt is not None and tgt < a:
                hist[f"loop {tgt:#06x}-{a:#06x} of {k}"] = collections.Counter(
                    op for x, op, _ in ins if tgt <= x <= a)
FLAG = ("LDGSTS", "UTMALDG", "UTMASTG", "UBLKCP", "UTCHMMA", "UTCQMMA", "LDTM", "STTM", "HMMA", "DMMA")
print("# cuobjdump -sass of", os.path.relpath(so, ROOT), "(sm_100a): static instruction counts per",
      "kernel" if loops is None else "loop")
print("# columns: total | FP64 (DADD+DMUL+DFMA+DSETP+MUFU) | LDG/STG | LDS/STS | SHFL | LDL/STL | flagged opcodes")
for k, h in hist.items():
    tot = sum(h.values())
    if tot == 0:
        continue
    f64 = sum(h[o] for o in ("DADD", "DMUL", "DFMA", "DSETP", "MUFU"))
    g = h["LDG"] + h["STG"] + h["LD"] + h["ST"]
    sh = h["LDS"] + h["STS"]
    lo = h["LDL"] + h["STL"]
    flags = " ".join(f"{o}={h[o]}" for o in FLAG if h[o])
    print(f"{tot:7d} | {f64:6d} | {g:5d} | {sh:5d} | {h['SHFL']:5d} | {lo:5d} | {flags or '-':24s} | {k[:110] if loops is None else k}")
