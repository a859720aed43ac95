#!/usr/bin/env python3
"""Cost of the irregular tiles of the long-document corpus (development aid; run under gpurun):
clean documents, then the same with k documents given a 32 KB space-free run / a 300-byte multi-mark stretch.
   LATOK_B200_PRINT_PROF=1 python tools/docs_probe.py
The [latok prof] line printed per launch holds the kernel's statistics counters (Result::stats): repeat_rounds,
ranges_repeated, repeats_hot_tail (ranges repeated because the guess about a hot tail was wrong), open_head / open_tail
(analyses of ranges that begin / end inside a chunk), backlog_out (ranges that leave a backlog), lookback_restarts, and the
look-ahead walks; a LATOK_PROFILE build adds the phase clocks (Result::clocks)."""
import sys; sys.path.insert(0, '.'); sys.path.insert(1, 'tests')
import numpy as np, ctypes as C
from latok_b200 import _lib
import synth
from latok_b200.engine import Engine

buf, off = synth.long_docs(3000, 65536)
keep = [i for i in range(3000) if (buf[off[i]:off[i + 1]] == 0x2C).mean() < 0.02]
parts = [buf[off[i]:off[i + 1]].copy() for i in keep]
no = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)


def variant(n_runs, n_marks, run_len=32768):
    ps = [p.copy() for p in parts]
    rng = np.random.default_rng(1)
    for d in rng.choice(len(ps), size=n_runs, replace=False):
        seg = ps[d][16384:16384 + run_len]
        seg[(seg == 0x20) | (seg == 0x0A)] = 0x2C
    for d in rng.choice(len(ps), size=n_marks, replace=False):
        a = int(rng.integers(0, len(ps[d]) - 400))
        seg = ps[d][a:a + 300]
        seg[(seg == 0x20) | (seg == 0x0A)] = 0x2C
    return np.concatenate(ps)


with Engine(0) as e:
    for name, nr, nm, rl in [("clean", 0, 0, 0), ("10 runs", 10, 0, 32768), ("40 runs", 40, 0, 32768), ("40 short runs (6 KB)", 40, 0, 6144),
                             ("40 runs of 12 KB", 40, 0, 12288), ("60 mark stretches", 0, 60, 0), ("600 mark stretches", 0, 600, 0)]:
        nb = variant(nr, nm, rl)
        for i in range(2):
            e.submit(nb, no, 3); c, t = e.sizes()
            ms = C.c_float(0); w = C.c_int64(0)
            _lib.check(_lib.load().latok_b200_last_stats(e._h, C.byref(ms), C.byref(w)))
        print(f"{name:24s} B={len(nb)} kernel={ms.value:.3f} ms in={len(nb)/ms.value/1e6:.1f} GB/s walks={w.value}", flush=True)
