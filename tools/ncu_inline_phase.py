#!/usr/bin/env python3
"""Executed warp-instructions and stall samples of the v5 tokenize kernel per PHASE and per SOURCE LINE of latok_tok5.cuh,
with inlined helpers (latok_bits.h, latok_device.cuh, CUDA intrinsics headers) charged to the line of latok_tok5.cuh
that called them.  ncu's own source page charges an instruction to the innermost inlined function only.

    python tools/ncu_inline_phase.py <rep.ncu-rep> <kernel-substring> <input bytes> [first-line last-line]
        kernel-substring  e.g. Lb1ELb0E (default rules: split mask + spans), Lb1ELb1E (with token features)
        LATOK_SHORT=0     the report is of the long geometry (4 KB ranges); default: short (3 KB ranges)

How: the translation unit of that geometry (latok_tok5_short.cu or latok_tok5.cu) is compiled to a cubin with the
library's flags, `nvdisasm -gi` gives every SASS instruction its chain of inlined call sites, and the n-th instruction of
the kernel in the disassembly is the n-th row of `ncu --page source --print-source sass` (checked: same count, same
opcodes).  The source must be the one the profiled library was built from."""
import collections, csv, os, re, subprocess, sys, tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "latok_b200" / "csrc"
SRC = CSRC / "latok_tok5.cuh"
rep, kern, nbytes = sys.argv[1], sys.argv[2], float(sys.argv[3])
lohi = (int(sys.argv[4]), int(sys.argv[5])) if len(sys.argv) > 5 else None
short = os.environ.get("LATOK_SHORT", "1") != "0"
RS = 3 if short else 4
NSTEP = nbytes / (RS * 1024 - 128) * RS                   # warp-steps (1 KB each) per launch

tmp = Path(tempfile.mkdtemp())
tu = CSRC / ("latok_tok5_short.cu" if short else "latok_tok5.cu")
subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-cubin",
                "-o", str(tmp / "k.cubin"), str(tu)], check=True, capture_output=True)
sass = subprocess.run(["nvdisasm", "-gi", "-c", str(tmp / "k.cubin")], check=True, capture_output=True, text=True).stdout.split("\n")
start = end = None
for i, l in enumerate(sass):
    if l.startswith(".text.") and kern in l: start = i
    elif start is not None and l.startswith("//-----"): end = i; break
assert start is not None, "kernel not found in the cubin"
pat_file = re.compile(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')
pat_ins = re.compile(r'^\s+/\*([0-9a-f]{4,})\*/\s+(.*?);')
chain, fresh, last_in, recs = [], True, None, []
for l in sass[start:end]:
    m = pat_file.search(l)
    if m:
        if fresh: chain, fresh = [], False
        chain.append((os.path.basename(m.group(1)), int(m.group(2))))
        last_in = (os.path.basename(m.group(3)), int(m.group(4))) if m.group(3) else None
        continue
    m = pat_ins.match(l)
    if m:
        if not fresh and last_in: chain.append(last_in)
        fresh = True
        ins = m.group(2).strip()
        recs.append((tuple(chain), (ins.split()[1] if ins.startswith("@") else ins.split()[0]).split(".")[0]))
out = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(out.splitlines()))
hdr, data = rows[1], rows[2:]
assert len(data) == len(recs), f"the report has {len(data)} instructions, this source compiles to {len(recs)}: not the profiled build"
iE, iS = hdr.index("Instructions Executed"), hdr.index("# Samples")
stalls = [h for h in hdr if h.startswith("stall_") and "Not Issued" not in h]
sidx = {n: hdr.index(n) for n in stalls}
src = SRC.read_text().split("\n")
# the lambdas' call sites are not "the line": skip them when walking the chain outwards-in
calls = {i + 1 for i, l in enumerate(src) if re.search(r"\b(analyze|output|finish_tile|begin_load)\(", l) and "auto " not in l}
by, sm, ops, st = collections.Counter(), collections.Counter(), collections.defaultdict(collections.Counter), collections.defaultdict(collections.Counter)
for (ch, op), r in zip(recs, data):
    tag = next((ln for f, ln in reversed(ch) if f == "latok_tok5.cuh" and ln not in calls), None)
    e = int(r[iE]); by[tag] += e; sm[tag] += int(r[iS]); ops[tag][op] += e
    for n in stalls:
        v = int(r[sidx[n]] or 0)
        if v: st[n][tag] += v
markers = [("setup", "template <class Geom, bool kDefault, bool kFeats>"), ("analysis: head", "auto analyze = [&]"), ("analysis: base planes", "for (int j = 0; j <= RS; ++j) {"),
           ("analysis: context + rules + block mask", "context + rules of step j-1"), ("analysis: guess", "PROF5(1);"),
           ("pass C", "pass C: blanked chunks, values, tokens"), ("service warp", "// service warp: tile aggregate"),
           ("output: head + CSR", "auto output = [&]"), ("output: step head", "for (int js = 0; js < RS; ++js) {\n            const uint32_t *t = SA("),
           ("output: split bytes", "split mask bytes"), ("output: spans", "// latest owned string start in the lanes before"),
           ("output: token features", "per-token feature sums (latok.c:342-354)"), ("main loop", "================= main loop"), ("end", "static cudaError_t launch_one")]
text = "\n".join(src)
pos = [(name, text[:text.index(mk)].count("\n") + 1) for name, mk in markers]
phases = [(pos[i][0], pos[i][1], pos[i + 1][1] - 1) for i in range(len(pos) - 1)]
tot, ts = sum(by.values()), sum(sm.values())
print(f"{tot / 1e6:.1f} M warp-instructions = {tot / NSTEP:.0f} per 1 KB step; {ts} stall samples")
for name, lo, hi in phases:
    e = sum(v for k, v in by.items() if k and lo <= k <= hi); s = sum(v for k, v in sm.items() if k and lo <= k <= hi)
    print(f"  {name:40s} {e / NSTEP:7.1f} per step {100 * e / tot:5.1f} %   samples {100 * s / ts:5.1f} %")
T = sum(sum(c.values()) for c in st.values())
print("stall reasons: " + "  ".join(f"{n[6:]} {100 * sum(c.values()) / T:.1f}" for n, c in sorted(st.items(), key=lambda kv: -sum(kv[1].values())) if sum(c.values()) > 0.01 * T))
if lohi:
    for tag in sorted(k for k in by if k and lohi[0] <= k <= lohi[1]):
        if by[tag] / NSTEP < 0.5: continue
        o = " ".join(f"{k}:{v / NSTEP:.0f}" for k, v in ops[tag].most_common(5))
        top = max(stalls, key=lambda n: st[n][tag])[6:]
        print(f"{tag:5d} {by[tag] / NSTEP:6.1f} {100 * sm[tag] / ts:5.2f}% {top[:10]:10s}| {src[tag - 1].strip()[:64]:64s} | {o}")
