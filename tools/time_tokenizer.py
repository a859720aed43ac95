#!/usr/bin/env python3
"""Timing / ingest CLI over the GPU batch path -- the counterpart of the reference's
scripts/timing/time_tokenizer.py:25-123 (same input format, same flags, same --outfile TSV), SURVEY 8 f3.

    python tools/time_tokenizer.py <csv or csv.gz: one record per row, JSON-encoded text in column 1>
        [--split | --matrix | --features] [--outfile tokens.tsv] [--counts counts.tsv] [--batch 200000] [--device 0]

The reference calls the tokenizer once per line; here lines are packed into batches (flat UTF-8 + offsets) by a
reader thread while the GPU works on the previous batch, and `--outfile` is written from the token byte ranges
(latok_b200_fetch_token_bytes) with NumPy gathers -- no Python string is created per token.  `--counts` counts the
tokens of all rows in one vocabulary on the GPU (latok_b200.vocab) and writes `token<TAB>count` lines, most common first
(equal counts in order of first occurrence).
"""
from __future__ import annotations

import argparse
import csv
import gzip
import json
import queue
import sys
import threading
import time
from datetime import datetime
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def read_batches(path: str, batch: int):
    """Yield (uint8 buffer, int64 offsets) per `batch` rows; text = json.loads(row[1]).strip() (time_tokenizer.py:35)."""
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "rt", encoding="utf-8", newline="") as f:
        enc, n = [], 0
        for row in csv.reader(f):
            enc.append(json.loads(row[1]).strip().encode("utf-8", "surrogatepass"))
            n += 1
            if n == batch:
                yield pack(enc)
                enc, n = [], 0
        if enc:
            yield pack(enc)


def pack(enc):
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in enc], out=off[1:])
    return np.frombuffer(b"".join(enc), dtype=np.uint8), off


def tsv_bytes(buf: np.ndarray, byte_spans: np.ndarray, tok_offsets: np.ndarray) -> bytes:
    """'\\t'.join(tokens) + '\\n' per string (time_tokenizer.py:107) as one bytes object, by gathers."""
    S, T = len(tok_offsets) - 1, len(byte_spans)
    ln = (byte_spans[:, 1] - byte_spans[:, 0]) + 1                       # token + its separator
    off = np.zeros(T + 1, dtype=np.int64)
    np.cumsum(ln, out=off[1:])
    out = np.empty(int(off[-1]), dtype=np.uint8)
    if T:
        idx = np.repeat(byte_spans[:, 0] - off[:-1], ln) + np.arange(off[-1], dtype=np.int64)
        sep_pos = off[1:] - 1
        idx[sep_pos] = 0
        out[:] = buf[idx] if len(buf) else 0
        out[sep_pos] = 0x09
        last = tok_offsets[1:][tok_offsets[1:] > tok_offsets[:-1]] - 1   # last token of every string that has tokens
        out[sep_pos[last]] = 0x0A
    empty = np.nonzero(tok_offsets[1:] == tok_offsets[:-1])[0]           # strings without tokens: an empty line
    if len(empty):
        out = np.insert(out, off[tok_offsets[empty]], 0x0A)
    return out.tobytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("infile", help="csv / csv.gz with the JSON-encoded text in column 1")
    ap.add_argument("--split", action="store_true", help="only generate the split mask")
    ap.add_argument("--matrix", action="store_true", help="only generate the parse matrix")
    ap.add_argument("--features", action="store_true", help="featurize the tokens")
    ap.add_argument("--mincount", type=int, default=100000, help="rows between progress lines")
    ap.add_argument("--outfile", help="write the tokens of every row, tab-separated, one row per line")
    ap.add_argument("--counts", help="write `token\tcount` per distinct token of the file, most common first")
    ap.add_argument("--batch", type=int, default=200_000, help="rows per GPU batch")
    ap.add_argument("--batch-bytes", type=int, default=64 << 20, help="native reader: UTF-8 bytes per GPU batch at most")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--reader", choices=["native", "python"], default="native",
                    help="native: rows parsed, JSON-decoded, stripped and packed by liblatok_b200 (latok_reader.cpp) into "
                         "pinned buffers; python: csv + json modules")
    args = ap.parse_args()
    print(f"{datetime.now()}: {args}", file=sys.stderr)
    from latok_b200.engine import Engine, FEATS, MATRIX, SPANS, SPLITS
    split, matrix = (False, False) if args.outfile else (args.split, args.matrix)
    what = SPLITS if split else MATRIX if matrix else (SPANS | FEATS) if args.features else SPANS
    if args.counts:
        what |= SPANS

    q: "queue.Queue" = queue.Queue(maxsize=2)
    done = threading.Event()

    def reader():
        try:
            if args.reader == "native":
                from latok_b200.reader import CsvReader
                # 4 buffer sets: one in the GPU call, two queued, one being filled
                with CsvReader(args.infile, args.batch, args.batch_bytes, pinned=True, n_buffers=4) as rd:
                    for item in rd:
                        q.put(item)
                    q.put(None)
                    done.wait()              # the pinned buffers must outlive the last GPU call
                return
            for item in read_batches(args.infile, args.batch):
                q.put(item)
            q.put(None)
        except BaseException as exc:
            q.put(exc)

    threading.Thread(target=reader, daemon=True).start()
    out = open(args.outfile, "wb") if args.outfile else None
    rows = n_bytes = n_tokens = 0
    gpu_s = write_s = 0.0
    next_report = args.mincount
    t_start = time.perf_counter()
    print(f"{datetime.now()}: Beginning tokenization...")
    with Engine(args.device) as e:
        vocab = None
        if args.counts:
            from latok_b200.vocab import Vocab
            vocab = Vocab(e)
        while True:
            item = q.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            buf, off = item
            t0 = time.perf_counter()
            e.submit(buf, off, what)
            r = e.fetch()
            bs = e.token_bytes() if out is not None else None
            if vocab is not None:
                vocab.encode_oldest(add=True, want_ids=False)
            gpu_s += time.perf_counter() - t0
            if out is not None:
                t0 = time.perf_counter()
                out.write(tsv_bytes(buf, bs, r.tok_offsets))
                write_s += time.perf_counter() - t0
            rows += len(off) - 1
            n_bytes += len(buf)
            n_tokens += r.n_tokens
            if rows >= next_report:
                dt = time.perf_counter() - t_start
                print(f"{datetime.now()}: {rows} lines, {rows / dt:.0f} lines/s, {n_bytes / dt / 1e6:.1f} MB/s", file=sys.stderr)
                next_report += args.mincount
        if vocab is not None:
            with open(args.counts, "wb") as f:
                f.write("".join(f"{t}\t{c}\n" for t, c in vocab.most_common()).encode("utf-8", "surrogatepass"))
            n_distinct = len(vocab)
            vocab.close()
    done.set()
    if out is not None:
        out.close()
    dt = time.perf_counter() - t_start
    print(f"{datetime.now()}: ...tokenized {rows} lines")
    print(json.dumps({"lines": rows, "bytes": n_bytes, "tokens": n_tokens, "seconds": dt, "lines_per_s": rows / dt,
                      "MB_per_s": n_bytes / dt / 1e6, "gpu_call_seconds": gpu_s, "write_seconds": write_s,
                      "mode": "split" if split else "matrix" if matrix else "features" if args.features else "tokenize",
                      "reader": args.reader, "distinct_tokens": None if vocab is None else n_distinct}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
