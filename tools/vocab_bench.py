#!/usr/bin/env python3
"""Token vocabulary on the GPU (latok_b200.vocab) against the host baseline it replaces.

    python tools/vocab_bench.py --out DIR [--strings 250000] [--batches 4] [--reps 5] [--devices 0,1,...]

Workloads: config #2 tweets (tests/synth.py tweets, seeds 20240601 + i), config #4 mixed Unicode (seeds 20240603 + i)
and `one_key`, a batch whose tokens are all the same key: every count increment of the launch lands on one address,
which is the worst case of the same-address contention a Zipf token stream causes (compare its device time per token
with the tweets' known-key pass).  Every batch is tokenized once (submitted with SPANS); on that batch in flight:

  add_first   encode(add=1) into a fresh vocabulary sized from a warm-up pass: mostly new keys (batch 0 only)
  add_known   encode(add=1) of batches 1.. into the vocabulary that holds the batches before: mostly known keys
  lookup      encode(add=0) of every batch against the vocabulary of all batches
Device time is latok_b200_vocab_last_ms (token byte ranges, insert / lookup, commit and count kernels; not the id copy
to the host), after one warm-up of each shape.  Host baseline on the same strings: `Counter.update` over
`tokenize_batch` (the tokenize_batch time itself is reported apart) and a dict lookup per token.  The card name and
power limit are read in the same process and written beside the numbers to DIR/vocab_bench.json.

--devices adds a `sharded` section: one batch of --sharded-strings strings (config #2 tweets, seed 20240601, and config
#4 mixed Unicode, seed 20240603) through `encode_sharded` and `update_sharded` over those devices (a device may repeat),
and through `encode_packed` on the first device alone, in alternating runs, each into a fresh vocabulary sized for the
batch's keys, from the host packed buffer.  Per run: host wall ms; the largest per-shard device ms (scratch
vocabulary encode), the merges' device ms (sum of `last_ms`, copy-in included) and the id gathers' device ms.  One
check per workload that keys, counts and ids of the sharded and one-GPU runs are identical.
"""
from __future__ import annotations

import argparse
import collections
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def card():
    import torch
    rec = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        rec["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        rec["nvidia_smi"] = f"unavailable: {exc}"
    return rec


def batches_for(name, n, count):
    import synth
    if name == "tweets":
        return [synth.tweets(n, 20240601 + i) for i in range(count)]
    if name == "mixed":
        return [synth.mixed_unicode(n, 20240603 + i) for i in range(count)]
    text = ("the " * 40).strip().encode()                         # one_key: 40 tokens per string, all "the"
    buf = np.frombuffer(text * n, dtype=np.uint8)
    return [(buf, np.arange(n + 1, dtype=np.int64) * len(text))] * count


def timed(v, add, reps):
    """device ms and host wall ms of `reps` encodes of the batch in flight (after one warm-up)"""
    v.encode_oldest(add=add)
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        v.encode_oldest(add=add)
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(v.last_ms())
    return dev, wall


def run_workload(e, name, n, count, reps):
    import synth
    from latok_b200.core.default_tokenizer import tokenize_batch
    from latok_b200.engine import SPANS
    from latok_b200.vocab import Vocab
    data = batches_for(name, n, count)
    rec = {"strings_per_batch": n, "batches": count, "add_first": {}, "add_known": [], "lookup": [], "host": []}
    main = Vocab(e)
    for i, (buf, off) in enumerate(data):
        e.submit(buf, off, SPANS)
        T = e.sizes()[1]
        if i == 0:
            warm = Vocab(e)
            warm.encode_oldest()
            dev, wall = [], []
            for _ in range(reps):
                v = Vocab(e, capacity=len(warm))
                t0 = time.perf_counter()
                v.encode_oldest()
                wall.append((time.perf_counter() - t0) * 1e3)
                dev.append(v.last_ms())
            rec["add_first"] = {"tokens": T, "distinct_keys": len(warm), "table_slots": v.table_slots(),
                                "load": len(v) / v.table_slots(), "device_ms": dev, "wall_ms": wall,
                                "tokens_per_s_device": T / (np.median(dev) * 1e-3)}
            main.encode_oldest()
        else:
            before = len(main)
            main.encode_oldest()                                  # the batch's first pass: mostly known keys
            d0 = main.last_ms()
            dev, wall = timed(main, True, reps)
            rec["add_known"].append({"batch": i, "tokens": T, "new_keys": len(main) - before, "first_pass_ms": d0,
                                     "device_ms": dev, "wall_ms": wall,
                                     "tokens_per_s_device": T / (np.median([d0] + dev) * 1e-3)})
    for i, (buf, off) in enumerate(data):
        e.submit(buf, off, SPANS)
        T = e.sizes()[1]
        dev, wall = timed(main, False, reps)
        rec["lookup"].append({"batch": i, "tokens": T, "device_ms": dev, "wall_ms": wall,
                              "tokens_per_s_device": T / (np.median(dev) * 1e-3)})
    rec["distinct_keys"], rec["table_slots"] = len(main), main.table_slots()
    rec["load"] = len(main) / main.table_slots()
    # host baseline on the same strings
    cnt, d = collections.Counter(), {}
    for i, (buf, off) in enumerate(data[:2]):
        texts = synth.to_strings(buf, off, 0, len(off) - 1)
        t0 = time.perf_counter()
        toks = tokenize_batch(texts, engine=e)
        t1 = time.perf_counter()
        flat = [t for ts in toks for t in ts]
        t2 = time.perf_counter()
        cnt.update(flat)
        t3 = time.perf_counter()
        if i == 0:
            for t in flat:
                d.setdefault(t, len(d))
        t4 = time.perf_counter()
        ids = [d.get(t, -1) for t in flat]
        t5 = time.perf_counter()
        rec["host"].append({"batch": i, "tokens": len(flat), "tokenize_batch_s": t1 - t0, "flatten_s": t2 - t1,
                            "counter_update_s": t3 - t2, "dict_lookup_s": t5 - t4,
                            "counter_tokens_per_s": len(flat) / (t3 - t2), "lookup_tokens_per_s": len(flat) / (t5 - t4),
                            "tokenize_batch_plus_counter_tokens_per_s": len(flat) / ((t1 - t0) + (t3 - t1))})
        del ids
    return rec


def run_sharded(name, n, devices, reps):
    from latok_b200.sharding import device_engine, encode_sharded, update_sharded
    from latok_b200.vocab import Vocab
    (buf, off), = batches_for(name, n, 1)
    e = device_engine(devices[0])
    single = Vocab(e)
    ids1, off1 = single.encode_packed(buf, off)                  # warm-up of every shape, and the reference
    keys = len(single)
    sh, up = Vocab(e, capacity=keys), Vocab(e, capacity=keys)
    ids2, off2 = encode_sharded(sh, buf, off, devices)
    update_sharded(up, buf, off, devices)
    want = (single.tokens(), single.counts().tolist())
    rec = {"strings": n, "devices": devices, "tokens": int(off1[-1]), "distinct_keys": keys,
           "identical": {"ids": bool(np.array_equal(ids1, ids2)), "tok_offsets": bool(np.array_equal(off1, off2)),
                         "encode_sharded_keys_counts": (sh.tokens(), sh.counts().tolist()) == want,
                         "update_sharded_keys_counts": (up.tokens(), up.counts().tolist()) == want},
           "single": [], "encode_sharded": [], "update_sharded": []}
    del sh, up
    for _ in range(reps):
        v = Vocab(e, capacity=keys)
        t0 = time.perf_counter()
        v.encode_packed(buf, off)
        rec["single"].append({"wall_ms": (time.perf_counter() - t0) * 1e3, "device_ms": v.last_ms()})
        for kind, fn in (("encode_sharded", encode_sharded), ("update_sharded", update_sharded)):
            v, st = Vocab(e, capacity=keys), {}
            t0 = time.perf_counter()
            fn(v, buf, off, devices, stats=st)
            wall = (time.perf_counter() - t0) * 1e3
            rec[kind].append({"wall_ms": wall, "max_shard_device_ms": max(st["shard_ms"]),
                              "merge_device_ms": sum(st["merge_ms"]), "remap_device_ms": sum(st.get("remap_ms", [])),
                              "shard_ms": st["shard_ms"], "merge_ms": st["merge_ms"]})
        del v
    med = lambda k, f: float(np.median([x[f] for x in rec[k]]))   # noqa: E731
    rec["median"] = {k: {f: med(k, f) for f in rec[k][0] if f.endswith("_ms") and not isinstance(rec[k][0][f], list)}
                     for k in ("single", "encode_sharded", "update_sharded")}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for vocab_bench.json")
    ap.add_argument("--strings", type=int, default=250_000, help="strings per batch")
    ap.add_argument("--batches", type=int, default=4, help="distinct batches per workload")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="tweets,mixed,one_key", help="comma-separated; empty: none")
    ap.add_argument("--devices", default="", help="comma-separated device list for the sharded section, e.g. 0,1")
    ap.add_argument("--sharded-strings", type=int, default=1_000_000, help="strings of the sharded section's batch")
    args = ap.parse_args()
    import torch
    from latok_b200.engine import Engine
    out = {"card": card(), "gpus": torch.cuda.device_count(), "args": vars(args), "workloads": {}}
    with Engine(0) as e:
        for name in [w for w in args.workloads.split(",") if w]:
            out["workloads"][name] = run_workload(e, name, args.strings, args.batches, args.reps)
            print(name, "done", file=sys.stderr)
    if args.devices:
        from latok_b200.sharding import close_engines
        devices = [int(d) for d in args.devices.split(",")]
        out["sharded"] = {name: run_sharded(name, args.sharded_strings, devices, args.reps) for name in ("tweets", "mixed")}
        close_engines()
    d = Path(args.out)
    d.mkdir(parents=True, exist_ok=True)
    (d / "vocab_bench.json").write_text(json.dumps(out, indent=1))
    summary = {"card": out["card"], "gpus": out["gpus"]}
    for name, r in out["workloads"].items():
        summary[name] = {"add_first_Mtok_s": r["add_first"]["tokens_per_s_device"] / 1e6,
                         "add_known_Mtok_s": [x["tokens_per_s_device"] / 1e6 for x in r["add_known"]],
                         "lookup_Mtok_s": [x["tokens_per_s_device"] / 1e6 for x in r["lookup"]],
                         "distinct_keys": r["distinct_keys"], "load": r["load"],
                         "host_counter_Mtok_s": [x["counter_tokens_per_s"] / 1e6 for x in r["host"]],
                         "host_lookup_Mtok_s": [x["lookup_tokens_per_s"] / 1e6 for x in r["host"]]}
    for name, r in out.get("sharded", {}).items():
        summary["sharded_" + name] = {"devices": r["devices"], "tokens": r["tokens"], "distinct_keys": r["distinct_keys"],
                                      "identical": r["identical"], "median_ms": r["median"]}
    print(json.dumps(summary))
    return 0


if __name__ == "__main__":
    sys.exit(main())
