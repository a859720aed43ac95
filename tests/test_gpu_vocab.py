"""Token vocabulary on the GPU (latok_b200.vocab, csrc/latok_vocab.cu) against plain Python over the oracle's tokens:
counts = collections.Counter, ids = dict.setdefault(token, len(d)) in token order.  Needs a B200 (-m gpu)."""
import collections
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import corpus
from oracle import oracle

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def engine():
    from latok_b200.engine import Engine
    with Engine(0) as e:
        yield e


def otoks(t):
    return oracle.tokens(t) if t else []


def expected(batches):
    """per batch the expected ids (flat, token order), and the final Counter and key order"""
    d, cnt, ids = {}, collections.Counter(), []
    for texts in batches:
        toks = [tok for t in texts for tok in otoks(t)]
        ids.append(np.array([d.setdefault(tok, len(d)) for tok in toks], dtype=np.int32))
        cnt.update(toks)
    return ids, cnt, list(d)


def check_vocab(v, batches):
    want_ids, want_cnt, want_keys = expected(batches)
    for texts, want in zip(batches, want_ids):
        ids, tok_off = v.encode(texts)
        assert np.array_equal(ids, want)
        assert tok_off[-1] == len(want) and len(tok_off) == len(texts) + 1
    assert len(v) == len(want_keys)
    assert v.tokens() == want_keys
    assert v.counts().tolist() == [want_cnt[k] for k in want_keys]
    return want_keys


def golden_texts():
    recs = json.loads((Path(__file__).parent / "golden" / "reference_outputs.json").read_text())["records"]
    return [r["text"] for r in recs]


def hard_keys():
    """long tokens, every UTF-8 length, lone surrogates, prefixes of one another, keys differing only in the last byte"""
    rng = np.random.default_rng(7)
    long1 = "x" * 70000
    long2 = "x" * 69999 + "y"
    long3 = "".join(rng.choice(["é", "日", "😀", "a"], size=90000))
    pre = ["a" * n for n in range(1, 40)] + ["ab" * n for n in range(1, 20)]
    last = [("q" * n) + c for n in (7, 8, 15, 16, 31, 255, 256, 257, 1000) for c in "ABC"]
    utf = ["é", "日本", "😀😀", "é日\U0001F600", "\ud800x", "a\udfff", "\ud83d"]
    return [long1, long2, long1, long3, long3 + "z", " ".join(pre), " ".join(last), " ".join(utf),
            " ".join(reversed(pre)), " ".join(utf + last)]


def test_counts_and_ids_fixtures_golden_fuzz(engine):
    from latok_b200.vocab import Vocab
    fuzz = corpus.fuzz_strings(41, 3000, 200, "mixed") + corpus.fuzz_strings(42, 3000, 120, "ascii")
    batches = [corpus.FIXTURES, golden_texts(), ["", "", "   "], [], fuzz[:1000], ["", " \t "] + fuzz[1000:3500],
               fuzz[3500:], corpus.FIXTURES + fuzz[:200]]
    check_vocab(Vocab(engine), batches)


def test_lookup_known_and_unknown(engine):
    from latok_b200.vocab import Vocab
    v = Vocab(engine)
    known = corpus.fuzz_strings(51, 1500, 150, "mixed")
    v.update(known)
    d = {k: i for i, k in enumerate(v.tokens())}
    probe = known[:300] + corpus.fuzz_strings(52, 700, 150, "mixed")
    before = v.counts()
    ids, tok_off = v.encode(probe, add=False, unk=-7)
    want = [d.get(tok, -7) for t in probe for tok in otoks(t)]
    assert ids.tolist() == want and -7 in want
    assert np.array_equal(v.counts(), before) and len(v) == len(d)        # a lookup changes nothing


def test_hard_keys(engine):
    from latok_b200.vocab import Vocab
    keys = check_vocab(Vocab(engine), [hard_keys(), hard_keys()[::-1]])
    assert "x" * 70000 in keys and "\ud800x" in keys


def test_forced_collisions_three_hash_bits():
    """Every key hashes to one of 7 values: long probe chains, every comparison by bytes."""
    code = f"""
import sys
sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'tests')!r}]
import corpus
from test_gpu_vocab import check_vocab, hard_keys, golden_texts
from latok_b200.engine import Engine
from latok_b200.vocab import Vocab
with Engine(0) as e:
    fuzz = corpus.fuzz_strings(61, 400, 80, "mixed")
    check_vocab(Vocab(e, capacity=4), [corpus.FIXTURES, hard_keys(), fuzz[:200], golden_texts()[:40], fuzz[150:]])
    v = Vocab(e)
    v.update(fuzz)
    f = Vocab.from_tokens(v.tokens(), engine=e)
    ids, _ = f.encode(fuzz + ["unseen tokens"], add=False)
    ids2, _ = v.encode(fuzz + ["unseen tokens"], add=False)
    assert (ids == ids2).all() and ids[-1] == -1
print("ok")
"""
    env = dict(os.environ, LATOK_B200_VOCAB_HASH_BITS="3")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(ROOT))
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-3000:]


def test_growth_from_capacity_16(engine):
    from latok_b200.vocab import Vocab
    words = [f"w{i:x}" for i in range(100_000)]
    texts = [" ".join(words[i:i + 50]) for i in range(0, len(words), 50)]
    batches = [texts[:1000], texts[1000:] + texts[:10], texts[::7]]
    check_vocab(Vocab(engine, capacity=16), batches)


def test_pipeline_depth2_oldest_batch(engine):
    from latok_b200.engine import SPANS, pack_strings
    from latok_b200.vocab import Vocab
    batches = [corpus.fuzz_strings(s, 800, 150, "mixed") for s in (71, 72, 73)]
    want_ids, want_cnt, want_keys = expected(batches)
    v = Vocab(engine)
    engine.set_pipeline_depth(2)
    try:
        packed = [pack_strings(b) for b in batches]
        engine.submit(*packed[0], SPANS)
        got = []
        for i in range(len(batches)):
            if i + 1 < len(batches):
                engine.submit(*packed[i + 1], SPANS)
            got.append(v.encode_oldest())
            with pytest.raises(RuntimeError):
                v.encode(["a"])                     # compound calls refuse while batches are in flight
            engine.release()
    finally:
        engine.set_pipeline_depth(1)
    for g, w in zip(got, want_ids):
        assert np.array_equal(g, w)
    assert v.tokens() == want_keys and v.counts().tolist() == [want_cnt[k] for k in want_keys]


def test_device_output_equals_host(engine):
    import torch
    from latok_b200.engine import pack_strings
    from latok_b200.vocab import Vocab
    texts = corpus.fuzz_strings(81, 2000, 150, "mixed")
    a, b = Vocab(engine), Vocab(engine)
    ids_h, off_h = a.encode_packed(*pack_strings(texts))
    ids_d, off_d = b.encode_packed(*pack_strings(texts), device=True)
    assert ids_d.is_cuda and ids_d.dtype == torch.int32
    assert np.array_equal(ids_d.cpu().numpy(), ids_h) and np.array_equal(off_d.numpy(), off_h)
    look, _ = b.encode_packed(*pack_strings(texts[:100]), add=False, unk=-1, device=True)
    assert np.array_equal(look.cpu().numpy(), ids_h[:off_h[100]])


def test_import_export_round_trip(engine):
    from latok_b200.vocab import Vocab
    v = Vocab(engine)
    texts = corpus.fuzz_strings(91, 2000, 150, "mixed") + hard_keys()
    v.update(texts)
    toks, cnt = v.tokens(), v.counts()
    f = Vocab.from_tokens(toks, cnt, engine=engine)
    assert f.tokens() == toks and np.array_equal(f.counts(), cnt)
    assert np.array_equal(f.encode(texts, add=False)[0], v.encode(texts, add=False)[0])
    with pytest.raises(RuntimeError):
        f.update(texts)                             # frozen
    g = Vocab.from_tokens(toks[:5], engine=engine)
    assert g.counts().tolist() == [0] * 5
    pruned = Vocab.from_tokens([t for t, c in v.most_common() if c >= 3], engine=engine)
    assert len(pruned) == sum(1 for c in cnt if c >= 3)
    for bad in (["a", "b", "a"], ["a", "", "b"], [""]):
        with pytest.raises(ValueError):
            Vocab.from_tokens(bad, engine=engine)
    h = Vocab(engine)
    h.update(["one two"])
    ok = Vocab.from_tokens(["z"], engine=engine)
    assert ok.tokens() == ["z"]
    assert Vocab.from_tokens([], engine=engine).tokens() == []


def test_most_common_order(engine):
    from latok_b200.vocab import Vocab
    v = Vocab(engine)
    v.update(["b a c a b d", "d e"])
    assert v.most_common() == [("b", 2), ("a", 2), ("d", 2), ("c", 1), ("e", 1)]
    assert v.most_common(2) == [("b", 2), ("a", 2)]


def test_deterministic_ids(engine):
    from latok_b200.vocab import Vocab
    batches = [corpus.fuzz_strings(s, 3000, 150, "ascii") for s in (101, 102)]
    a, b = Vocab(engine), Vocab(engine)
    for t in batches:
        assert np.array_equal(a.encode(t)[0], b.encode(t)[0])
    assert a.tokens() == b.tokens()


def test_scale_200k_tweets_against_counter(engine):
    import synth
    from latok_b200.core.default_tokenizer import tokenize_batch
    from latok_b200.vocab import Vocab
    buf, off = synth.tweets(200_000, 20240601)
    v = Vocab(engine)
    ids, tok_off = v.encode_packed(buf, off)
    texts = synth.to_strings(buf, off, 0, len(off) - 1)
    toks = [t for ts in tokenize_batch(texts, engine=engine) for t in ts]
    d = {}
    assert ids.tolist() == [d.setdefault(t, len(d)) for t in toks]
    c = collections.Counter(toks)
    assert v.tokens() == list(d) and v.counts().tolist() == [c[k] for k in d]
    assert v.most_common(20) == sorted(c.items(), key=lambda kv: (-kv[1], d[kv[0]]))[:20]


def test_time_tokenizer_counts_cli(tmp_path):
    import csv
    import gzip
    texts = [t for t in corpus.FIXTURES + corpus.fuzz_strings(111, 600, 120) if "\x00" not in t]
    texts = [t for t in texts if not any(0xD800 <= ord(c) <= 0xDFFF for c in t)] + ["", "   "]
    src = tmp_path / "in.csv.gz"
    with gzip.open(src, "wt", encoding="utf-8", newline="") as f:
        w = csv.writer(f)
        for i, t in enumerate(texts):
            w.writerow([i, json.dumps(t)])
    toks = [tok for t in texts for tok in otoks(t.strip())]
    d = {}
    for t in toks:
        d.setdefault(t, len(d))
    c = collections.Counter(toks)
    want = "".join(f"{t}\t{n}\n" for t, n in sorted(c.items(), key=lambda kv: (-kv[1], d[kv[0]])))
    out = tmp_path / "counts.tsv"
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "time_tokenizer.py"), str(src), "--counts", str(out),
                        "--batch", "64", "--batch-bytes", "65536"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert out.read_text(encoding="utf-8") == want
    assert json.loads(r.stdout.strip().splitlines()[-1])["distinct_tokens"] == len(c)
