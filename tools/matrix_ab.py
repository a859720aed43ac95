#!/usr/bin/env python3
"""A/B timing of the parse-matrix modes of two or more library builds (development aid).

    python tools/matrix_ab.py --out FILE.json [--rounds 3] [--reps 10] LIB.so [LIB.so ...]

Workloads: 1 M tweets and 1 M mixed-Unicode strings (tests/synth.py), each with what = 8, 1|2|8 and 15, submitted from
device memory.  The time of a submit is the device time from timer_begin before it to timer_end after sizes: every
kernel of the submit and the copy of its result record, not only the tokenize kernel that latok_b200_last_stats
reports.  Also the wall time of one gen_parse_matrix call on a tweet-length string, and its kernel launches.

Every library runs in a process of its own (LATOK_B200_LIB), the libraries in turn, --rounds times, so that the spread
between rounds shows next to the difference between builds.  The first round also records a SHA-256 of every output
(matrix, split mask, spans, offsets, token features), so that the builds can be compared byte for byte.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
WHATS = (8, 1 | 2 | 8, 15)


def worker(data_dir: Path, reps: int, digest: bool, calls: int) -> dict:
    sys.path.insert(0, str(ROOT))
    import numpy as np
    import torch
    from latok_b200 import _lib
    from latok_b200.engine import Engine
    out = {"lib": str(_lib.LIB_PATH), "submit_ms": {}, "sha256": {}}
    with Engine(0) as e:
        for wl in ("tweets", "mixed"):
            buf, off = np.load(data_dir / f"{wl}_buf.npy"), np.load(data_dir / f"{wl}_off.npy")
            d_buf, d_off = torch.from_numpy(buf).cuda(), torch.from_numpy(off).cuda()
            torch.cuda.synchronize()
            for what in WHATS:
                ts = []
                for i in range(reps + 1):               # the first submit sizes the buffers and loads the kernels
                    e.timer_begin()
                    e.submit_device(d_buf.data_ptr(), d_off.data_ptr(), len(off) - 1, len(buf), what)
                    e.sizes()
                    ms = e.timer_end()
                    if i:
                        ts.append(ms)
                key = f"{wl}/what={what}"
                out["submit_ms"][key] = {"best": min(ts), "median": statistics.median(ts), "max": max(ts)}
                r = e.fetch()
                if digest:
                    h = {}
                    for name in ("matrix", "splits", "spans", "char_offsets", "tok_offsets", "tok_feats"):
                        a = getattr(r, name)
                        if a is not None:
                            h[name] = hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
                    out["sha256"][key] = {"n_chars": int(r.n_chars), "n_tokens": int(r.n_tokens), **h}
                del r
            del d_buf, d_off
        tw_buf, tw_off = np.load(data_dir / "tweets_buf.npy", mmap_mode="r"), np.load(data_dir / "tweets_off.npy")
        text = bytes(tw_buf[tw_off[0]:tw_off[1]]).decode("utf-8")
        for _ in range(100):
            m = e.gen_parse_matrix(text)
        l0 = e.launch_count()
        e.gen_parse_matrix(text)
        launches = e.launch_count() - l0
        walls = []
        for _ in range(5):
            t0 = time.perf_counter()
            for _ in range(calls):
                m = e.gen_parse_matrix(text)
            walls.append((time.perf_counter() - t0) / calls * 1e6)
        out["gen_parse_matrix"] = {"chars": len(text), "launches_per_call": launches, "us_per_call_best": min(walls),
                                   "us_per_call_median": statistics.median(walls), "calls": calls * 5}
        if digest:
            out["sha256"]["gen_parse_matrix"] = hashlib.sha256(m.tobytes()).hexdigest()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*")
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--calls", type=int, default=2000)
    ap.add_argument("--worker", metavar="DATA_DIR")
    ap.add_argument("--digest", action="store_true")
    a = ap.parse_args()
    if a.worker:
        print(json.dumps(worker(Path(a.worker), a.reps, a.digest, a.calls)))
        return
    sys.path.insert(0, str(ROOT / "tests"))
    import numpy as np
    import synth
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "workloads": {}, "rounds": []}
    with tempfile.TemporaryDirectory() as tmp:
        for wl, gen in (("tweets", synth.tweets), ("mixed", synth.mixed_unicode)):
            buf, off = gen(1_000_000)
            np.save(Path(tmp) / f"{wl}_buf.npy", buf)
            np.save(Path(tmp) / f"{wl}_off.npy", off)
            res["workloads"][wl] = {"strings": len(off) - 1, "bytes": int(len(buf))}
        for k in range(a.rounds):
            rnd = {}
            for lib in a.libs:
                cmd = [sys.executable, __file__, "--worker", tmp, "--reps", str(a.reps), "--calls", str(a.calls)]
                if k == 0:
                    cmd.append("--digest")
                p = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, LATOK_B200_LIB=lib))
                if p.returncode:
                    sys.exit(f"{lib}: worker failed\n{p.stderr[-4000:]}")
                rnd[lib] = json.loads(p.stdout.strip().splitlines()[-1])
                print(f"round {k} {lib}: " + json.dumps(rnd[lib]["submit_ms"]) + " " + json.dumps(rnd[lib]["gen_parse_matrix"]), flush=True)
            res["rounds"].append(rnd)
    first = res["rounds"][0]
    digests = [json.dumps(first[lib]["sha256"], sort_keys=True) for lib in a.libs]
    res["outputs_identical"] = len(set(digests)) == 1
    print("outputs identical across builds:", res["outputs_identical"])
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
