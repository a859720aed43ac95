#!/usr/bin/env python3
"""Where the fixed cost of a tokenize step goes (config-#2 text, data on the device).  Needs a GPU.

    python tools/step_cost.py [--out FILE] [--launches 40] [--steps 200]

1. Kernel time against batch size, 0.25 .. 4 M strings: CUDA events around the tokenize launch (the ones
   latok_b200_last_stats reads), median of `--launches` launches after warm-up.  The batches are slices of one 4 M-string
   pool (584 MB) taken in turn, so the footprint stays above the 126 MB of L2.  Least-squares slope (us per MB) and
   intercept (us per launch), and about how many tiles of each size each CTA of the grid runs (the last wave's sawtooth;
   estimated from the short geometry's range and tile size below and the mean batch size, not read from the plan).
2. The resident loop of bench.py (back-to-back submit_device of 1 M strings): ms per step against the kernel time, and a
   torch.profiler trace of the same loop, from which the gap between two tokenize kernels and what lies in it: the string
   index kernel, the result copy, the result memset.  The trace stands in for events around each item (it widens the gaps
   a little).  No per-CTA timeline is taken.
The card's name and power limit are read in the same run.  Prints one JSON document and writes it to --out.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(1, str(ROOT / "tests"))

SIZES = [250_000, 500_000, 1_000_000, 2_000_000, 4_000_000]
RANGE, NW = 3 * 1024 - 128, 11          # ShortGeometry of latok_tok5.cuh (tweets): bytes per range, ranges per tile


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def kernel_ms(lib, eng):
    ms, w = C.c_float(0), C.c_int64(0)
    lib.latok_b200_last_stats(eng._h, C.byref(ms), C.byref(w))
    return ms.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--launches", type=int, default=40)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()

    import bench
    pool_b, pool_o = bench.generate({"p": [("tweets", 1_000_000, 20240601 + k) for k in range(4)]})["p"]
    import torch
    from latok_b200 import _lib
    from latok_b200.engine import Engine, SPLITS, SPANS
    lib = _lib.load()
    what = SPLITS | SPANS
    d_buf = torch.from_numpy(pool_b).cuda()
    d_off = torch.from_numpy(pool_o).cuda()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    grid = 2 * n_sm
    out = {"card": card(), "sm": n_sm, "grid": grid}
    eng = Engine(0)

    def slices(n):
        """device batches of n strings cut from the pool, each a tensor of its own (aligned): (text, offsets, n_bytes)"""
        res = []
        for s0 in range(0, len(pool_o) - n, n):
            b0, b1 = int(pool_o[s0]), int(pool_o[s0 + n])
            res.append((d_buf[b0:b1].clone(), (d_off[s0:s0 + n + 1] - b0).contiguous(), b1 - b0))
        return res

    # ---- 1. kernel time against batch size
    rows = []
    for n in SIZES:
        bs = slices(n)
        if not bs:
            continue
        for i in range(6):
            p, o, nb = bs[i % len(bs)]
            eng.submit_device(p.data_ptr(), o.data_ptr(), n, nb, what); eng.sizes()
        t = []
        for i in range(args.launches):
            p, o, nb = bs[i % len(bs)]
            eng.submit_device(p.data_ptr(), o.data_ptr(), n, nb, what); eng.sizes()
            t.append(kernel_ms(lib, eng))
        mb = float(np.mean([b[2] for b in bs])) / 1e6
        nranges = int(mb * 1e6) // RANGE + 1
        full = -(-nranges // NW)
        rows.append({"strings": n, "mb": mb, "batches": len(bs), "kernel_ms_median": float(np.median(t)),
                     "kernel_ms_spread": [float(np.min(t)), float(np.max(t))], "ranges_approx": nranges,
                     "tiles_approx": full, "tiles_per_cta_approx": full / grid})
    x = np.array([r["mb"] for r in rows]); y = np.array([r["kernel_ms_median"] for r in rows]) * 1e3
    slope, icpt = np.polyfit(x, y, 1)
    out["kernel_vs_size"] = rows
    out["fit"] = {"slope_us_per_mb": float(slope), "intercept_us": float(icpt),
                  "residuals_us": [float(v) for v in (y - (slope * x + icpt))]}

    # ---- 2. the resident loop at 1 M strings (as bench.py: three batches in turn)
    bs = slices(1_000_000)[:3]

    def loop(k):
        for i in range(k):
            p, o, nb = bs[i % len(bs)]
            eng.submit_device(p.data_ptr(), o.data_ptr(), 1_000_000, nb, what)

    loop(10); eng.sizes()
    per_step = []
    for _ in range(3):
        eng.timer_begin(); loop(args.steps); per_step.append(eng.timer_end() / args.steps)
    out["resident"] = {"ms_per_step": per_step}

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loop(40); eng.sizes()
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "trace.json")
        prof.export_chrome_trace(f)
        ev = json.load(open(f))["traceEvents"]
    dev = [e for e in ev if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]

    def kind(e):
        n = e["name"]
        if "tokenize5_kernel" in n: return "tokenize"
        if "tile_index_kernel" in n: return "string_index"
        if e["cat"] == "gpu_memcpy": return "result_copy"
        if e["cat"] == "gpu_memset": return "result_memset"
        return n[:40]

    tok = sorted([e for e in dev if kind(e) == "tokenize"], key=lambda e: e["ts"])
    gaps = []
    for a, b in zip(tok[:-1], tok[1:]):
        g0, g1 = a["ts"] + a["dur"], b["ts"]
        inside = {}
        for e in dev:
            k = kind(e)
            if k == "tokenize": continue
            lo, hi = max(g0, e["ts"]), min(g1, e["ts"] + e["dur"])
            if hi > lo: inside[k] = inside.get(k, 0.0) + (hi - lo)
            if k == "string_index" and e["ts"] < g0 and e["ts"] + e["dur"] > a["ts"]:
                inside["string_index_under_previous_kernel"] = inside.get("string_index_under_previous_kernel", 0.0) + \
                    (min(g0, e["ts"] + e["dur"]) - max(a["ts"], e["ts"]))
        gaps.append({"gap": g1 - g0, **inside})
    keys = sorted({k for g in gaps for k in g})
    durs = {}
    for e in dev:
        durs.setdefault(kind(e), []).append(e["dur"])
    out["trace"] = {"tokenize_kernels": len(tok),
                    "gap_us_median": {k: float(np.median([g.get(k, 0.0) for g in gaps])) for k in keys},
                    "duration_us_median": {k: float(np.median(v)) for k, v in durs.items()}}
    eng.close()
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
