#!/usr/bin/env python3
"""WordPiece on the GPU (Vocab.wordpiece_packed) against the host baselines it replaces.

    python tools/wordpiece_bench.py --out DIR [--strings 250000] [--reps 7] [--ref-strings 2000]

Workloads: config #2 tweets (tests/synth.py tweets, seed 20240601 + i) and config #4 mixed Unicode (seed 20240603 + i),
batch i = 0 timed, and `worst`: words of exactly max_chars characters whose only pieces are single characters, so that
every start of every word probes every candidate end the longest key allows.  It bounds what lanes that diverge on long
searches cost next to the one-probe whole-token hits.

Vocabulary (vocab_tokens, also used by tests/test_gpu_wordpiece.py): from the tokens of a separate batch of the same
generator (seed + 1), the 20 000 most common whole tokens, every character seen alone and as "##" + character, the
10 000 most common "##" + substrings of 2 to 4 characters at non-initial positions, and "[UNK]".  `worst` uses the
config #4 vocabulary.

Per workload: words, pieces per word, share of one-piece words and of unk words; device ms per call
(latok_b200_vocab_last_ms: token byte ranges, count, scan and write kernels; median of --reps after a warm-up) and
G words/s; HF tokenizers' Tokenizer(WordPiece) with a WhitespaceSplit pre-tokenizer and encode_batch over every
string's LaTok tokens joined by one space (the host core count is recorded); the Python reference
(tests/test_gpu_wordpiece.py wordpiece_ref) on the first --ref-strings strings; and whether the GPU and HF ids are
identical over the whole batch.  The card name and power limit are read in the same process and written beside the
numbers to DIR/wordpiece_bench.json.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

UNK = "[UNK]"


def vocab_tokens(token_counts, prefix: str = "##", n_whole: int = 20_000, n_sub: int = 10_000):
    """The benchmark's vocabulary from (token, count) pairs, most common first (Vocab.most_common()): the n_whole most
    common tokens, every character alone and as prefix + character, the n_sub most common prefix + substrings of 2-4
    characters that do not start a token, and "[UNK]"; each key once, in that order."""
    out = dict.fromkeys(t for t, _ in token_counts[:n_whole])
    chars = {}
    subs = collections.Counter()
    for t, c in token_counts:
        for ch in t:
            chars.setdefault(ch, None)
        for n in (2, 3, 4):
            for i in range(1, len(t) - n + 1):
                subs[t[i:i + n]] += c
    for ch in chars:
        out.setdefault(ch, None)
        out.setdefault(prefix + ch, None)
    for s, _ in subs.most_common(n_sub):
        out.setdefault(prefix + s, None)
    out.setdefault(UNK, None)
    return list(out)


def worst_words(vocab: set, max_chars: int, n: int, seed: int, prefix: str = "##"):
    """n words of exactly max_chars characters, each a lower-case letter of `vocab` alone and as prefix + character (so
    that LaTok keeps the word one token), such that no piece of two or more characters is a key: WordPiece splits them
    into max_chars single characters."""
    rng = np.random.default_rng(seed)
    chars = sorted(c for c in vocab if len(c) == 1 and c.isalpha() and c == c.lower() and prefix + c in vocab)
    longest = max(len(k) for k in vocab)
    words = []
    while len(words) < n:
        w = ""
        while len(w) < max_chars:
            cand = w + chars[rng.integers(len(chars))]
            if not any((prefix if j else "") + cand[j:] in vocab for j in range(max(0, len(cand) - longest), len(cand) - 1)):
                w = cand
        words.append(w)
    return words


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


def batch(name, n, i):
    import synth
    if name == "tweets":
        return synth.tweets(n, 20240601 + i)
    return synth.mixed_unicode(n, 20240603 + i)


def token_strings(engine, buf, off):
    """every string's LaTok tokens (trimmed, as Vocab keys them)"""
    from latok_b200.core.default_tokenizer import tokenize_packed
    pt = tokenize_packed(buf, off, engine=engine)
    return [pt.tokens(i) for i in range(len(off) - 1)]


def run_workload(engine, name, buf, off, toks, keys, args):
    from latok_b200.vocab import Vocab
    from test_gpu_wordpiece import wordpiece_ref
    from tokenizers import Tokenizer
    from tokenizers.models import WordPiece
    from tokenizers.pre_tokenizers import WhitespaceSplit

    v = Vocab.from_tokens(keys, engine=engine)
    unk = keys.index(UNK)
    v.wordpiece_packed(buf, off, unk, max_chars=args.max_chars)                    # warm-up
    ms = []
    for _ in range(args.reps):
        ids, offsets, word_off = v.wordpiece_packed(buf, off, unk, max_chars=args.max_chars)
        ms.append(v.last_ms())
    T = len(word_off) - 1
    n_pieces = np.diff(word_off)
    one = n_pieces == 1
    rec = {"strings": len(off) - 1, "bytes": int(off[-1]), "words": T, "pieces": len(ids),
           "pieces_per_word": len(ids) / max(T, 1),
           "one_piece_share": float(np.mean(one & (ids[word_off[:-1]] != unk))) if T else 0.0,
           "unk_share": float(np.mean(one & (ids[word_off[:-1]] == unk))) if T else 0.0,
           "device_ms": ms, "device_ms_median": float(np.median(ms)),
           "gwords_per_s": T / (float(np.median(ms)) * 1e-3) / 1e9}

    hf = Tokenizer(WordPiece({k: i for i, k in enumerate(keys)}, unk_token=UNK, max_input_chars_per_word=args.max_chars,
                             continuing_subword_prefix="##"))
    hf.pre_tokenizer = WhitespaceSplit()
    joined = [" ".join(t) for t in toks]
    t0 = time.perf_counter()
    enc = hf.encode_batch(joined, add_special_tokens=False)
    hf_s = time.perf_counter() - t0
    hf_ids = np.fromiter((i for e in enc for i in e.ids), dtype=np.int32)
    rec["hf"] = {"s": hf_s, "gwords_per_s": T / hf_s / 1e9, "host_cores": os.cpu_count()}
    rec["ids_equal_hf"] = bool(np.array_equal(hf_ids, ids))

    d = {k.encode("utf-8", "surrogatepass"): i for i, k in enumerate(keys)}
    words = [w.encode("utf-8", "surrogatepass") for t in toks[:args.ref_strings] for w in t]
    t0 = time.perf_counter()
    ref = [p for w in words for p in wordpiece_ref(w, d, unk, b"##", args.max_chars)]
    ref_s = time.perf_counter() - t0
    rec["python_ref"] = {"strings": min(args.ref_strings, len(toks)), "words": len(words), "s": ref_s,
                         "words_per_s": len(words) / ref_s if ref_s else None,
                         "ids_equal": ref == ids[:word_off[len(words)]].tolist()}
    print(name, json.dumps({k: v for k, v in rec.items() if k != "device_ms"}), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--strings", type=int, default=250_000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--ref-strings", type=int, default=2000)
    ap.add_argument("--max-chars", type=int, default=100)
    ap.add_argument("--worst-words", type=int, default=20_000)
    args = ap.parse_args()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)

    from latok_b200.engine import Engine, pack_strings
    from latok_b200.vocab import Vocab
    res = {"card": card(), "args": {k: v for k, v in vars(args).items() if k != "out"}, "workloads": {}}
    with Engine(0) as e:
        mixed_keys = None
        for name in ("tweets", "mixed"):
            vb, vo = batch(name, args.strings, 1)
            counter = Vocab(e)
            counter._run(vb, vo, True, -1, "none")
            keys = vocab_tokens(counter.most_common())
            counter.close()
            buf, off = batch(name, args.strings, 0)
            rec = run_workload(e, name, buf, off, token_strings(e, buf, off), keys, args)
            rec["vocab_size"] = len(keys)
            res["workloads"][name] = rec
            mixed_keys = keys
        words = worst_words(set(mixed_keys), args.max_chars, 2000, 20240607)
        rng = np.random.default_rng(20240608)
        pick = rng.integers(len(words), size=args.worst_words)
        texts = [" ".join(words[j] for j in pick[i:i + 4]) for i in range(0, len(pick), 4)]
        buf, off = pack_strings(texts)
        rec = run_workload(e, "worst", buf, off, token_strings(e, buf, off), mixed_keys, args)
        rec["vocab_size"] = len(mixed_keys)
        res["workloads"]["worst"] = rec
    (out / "wordpiece_bench.json").write_text(json.dumps(res, indent=1))
    print(json.dumps({k: {"gwords_per_s": r["gwords_per_s"], "device_ms": r["device_ms_median"],
                          "ids_equal_hf": r["ids_equal_hf"]} for k, r in res["workloads"].items()}))


if __name__ == "__main__":
    main()
