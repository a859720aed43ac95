"""WordPiece on the GPU (Vocab.wordpiece, csrc/latok_vocab.cu) against a plain-Python statement of the algorithm,
wordpiece_ref, over the oracle's tokens.  wordpiece_ref itself is checked against HF tokenizers' WordPiece without a
GPU; every other test needs a B200 (-m gpu)."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import corpus
from oracle import oracle
from test_gpu_vocab import golden_texts, hard_keys

ROOT = Path(__file__).resolve().parent.parent
_spec = importlib.util.spec_from_file_location("wordpiece_bench", ROOT / "tools" / "wordpiece_bench.py")
wordpiece_bench = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(wordpiece_bench)
PREFIX17 = "<cont-prefix-17b>"                  # 17 bytes: prefix + piece crosses 8-byte words at every offset


def wordpiece_ref(word: bytes, vocab: dict, unk: int, prefix: bytes = b"##", max_chars: int = 100):
    """BERT's WordpieceTokenizer.tokenize on UTF-8 bytes: greedy longest match first, candidate ends on character
    boundaries only, continuation keys = prefix + rest; too many characters or no match at some start: [unk]."""
    if len(word.decode("utf-8", "surrogatepass")) > max_chars:
        return [unk]
    ends = [i for i in range(1, len(word) + 1) if i == len(word) or word[i] & 0xC0 != 0x80]
    out, start = [], 0
    while start < len(word):
        for end in reversed([i for i in ends if i > start]):
            key = (prefix if start else b"") + word[start:end]
            if key in vocab:
                out.append(vocab[key])
                start = end
                break
        else:
            return [unk]
    return out


def words_of(t):
    return [w.encode("utf-8", "surrogatepass") for w in oracle.tokens(t)] if t else []


def expected(texts, keys, unk, prefix="##", max_chars=100):
    """(ids, offsets, word_offsets) of wordpiece_ref over the oracle's tokens of texts, memoised per distinct word"""
    d = {k if isinstance(k, bytes) else k.encode("utf-8", "surrogatepass"): i for i, k in enumerate(keys)}
    pre = prefix.encode("utf-8", "surrogatepass")
    memo, ids, offsets, word_off = {}, [], [0], [0]
    for t in texts:
        for w in words_of(t):
            if w not in memo:
                memo[w] = wordpiece_ref(w, d, unk, pre, max_chars)
            ids += memo[w]
            word_off.append(len(ids))
        offsets.append(len(ids))
    return np.array(ids, dtype=np.int32), np.array(offsets, dtype=np.int64), np.array(word_off, dtype=np.int64)


def recipe(texts, prefix="##"):
    """the benchmark's vocabulary recipe over the oracle's tokens of texts"""
    import collections
    c = collections.Counter(w for t in texts for w in (oracle.tokens(t) if t else []))
    return wordpiece_bench.vocab_tokens(c.most_common(), prefix)


def fuzz_texts():
    return corpus.fuzz_strings(301, 1500, 200, "mixed") + corpus.fuzz_strings(302, 1500, 120, "ascii")


def no_surrogates(texts):
    return [t for t in texts if not any(0xD800 <= ord(c) <= 0xDFFF for c in t)]


# ---- the reference against HF tokenizers (no GPU) ----------------------------------------------------------------------
@pytest.mark.parametrize("prefix", ["##", "", "▁"])
def test_reference_equals_hf_wordpiece(prefix):
    pytest.importorskip("tokenizers")
    from tokenizers.models import WordPiece
    texts = no_surrogates(corpus.FIXTURES + golden_texts() + fuzz_texts())
    keys = recipe(no_surrogates(corpus.fuzz_strings(303, 1500, 200, "mixed")), prefix)
    unk = keys.index("[UNK]")
    hf = WordPiece({k: i for i, k in enumerate(keys)}, unk_token="[UNK]", max_input_chars_per_word=100,
                   continuing_subword_prefix=prefix)
    d = {k.encode(): i for i, k in enumerate(keys)}
    words = {w for t in texts for w in (oracle.tokens(t) if t else [])}
    words |= {"é" * 100, "é" * 101, "x" * 101}
    n_multi = 0
    for w in sorted(words):
        want = [tok.id for tok in hf.tokenize(w)]
        assert wordpiece_ref(w.encode(), d, unk, prefix.encode()) == want, w
        n_multi += len(want) > 1
    assert n_multi > 100


# ---- the GPU against the reference -------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine():
    from latok_b200.engine import Engine
    from latok_b200.sharding import close_engines
    with Engine(0) as e:
        yield e
    close_engines()


def check(v, texts, keys, unk, prefix="##", max_chars=100):
    ids, offsets, word_off = v.wordpiece(texts, unk, prefix, max_chars)
    want = expected(texts, keys, unk, prefix, max_chars)
    assert ids.dtype == np.int32 and offsets.dtype == np.int64 and word_off.dtype == np.int64
    assert np.array_equal(word_off, want[2])
    assert np.array_equal(offsets, want[1])
    assert np.array_equal(ids, want[0])
    return ids, offsets, word_off


def vocabularies(prefix):
    """the benchmark's recipe, whole tokens only, and the recipe without a seeded 5 % of its single characters"""
    src = corpus.fuzz_strings(304, 2000, 200, "mixed") + corpus.fuzz_strings(305, 1000, 120, "ascii") + corpus.FIXTURES
    full = recipe(src, prefix)
    whole = list(dict.fromkeys(w for t in src for w in (oracle.tokens(t) if t else [])))[:20_000]
    chars = sorted({k for k in full if len(k) == 1})
    rng = np.random.default_rng(306)
    drop = set(rng.choice(chars, size=max(1, len(chars) // 20), replace=False).tolist())
    missing = [k for k in full if k not in drop and not (prefix and k.startswith(prefix) and k[len(prefix):] in drop)]
    return {"recipe": full, "whole": [k for k in whole if k != "[UNK]"] + ["[UNK]"], "missing": missing}


@pytest.mark.gpu
@pytest.mark.parametrize("prefix", ["##", "", "▁", PREFIX17])
def test_fixtures_golden_fuzz_hard_keys(engine, prefix):
    from latok_b200.vocab import Vocab
    texts = corpus.FIXTURES + golden_texts() + fuzz_texts() + hard_keys()
    for name, keys in vocabularies(prefix).items():
        v = Vocab.from_tokens(keys, engine=engine)
        unk = keys.index("[UNK]")
        ids, _, word_off = check(v, texts, keys, unk, prefix)
        assert (ids == unk).any(), name
        assert name == "whole" or (np.diff(word_off) > 1).any(), name


@pytest.mark.gpu
@pytest.mark.parametrize("max_chars", [1, 3, 100, 1024])
def test_max_chars_at_every_width(engine, max_chars):
    from latok_b200.vocab import Vocab
    chars = ["a", "\ud800", "é", "日", "\udfff", "😀"]          # no surrogate pair side by side
    words = [c * n for c in chars for n in (max_chars - 1, max_chars, max_chars + 1) if n]
    words += ["".join(chars[(i + j) % len(chars)] for j in range(n)) for i in range(3)
              for n in (max_chars - 1, max_chars, max_chars + 1) if n]
    keys = chars + ["##" + c for c in chars] + ["##" + c * 2 for c in chars] + ["[UNK]"]
    v = Vocab.from_tokens(keys, engine=engine)
    texts = [" ".join(words), words[0], " ".join(reversed(words))]
    check(v, texts, keys, keys.index("[UNK]"), "##", max_chars)
    for bad in (0, 1025):
        with pytest.raises(ValueError, match="max_chars"):
            v.wordpiece(texts, 0, max_chars=bad)


@pytest.mark.gpu
def test_long_pieces_and_words(engine):
    """keys and pieces longer than 256 bytes, with and without the prefix, through the candidate-length bound"""
    from latok_b200.vocab import Vocab
    keys = ["x" * 300, "##" + "y" * 280, "##" + "é" * 150, "日" * 100, "##z", "x", "##x", "##y", "[UNK]", "w" * 1000]
    v = Vocab.from_tokens(keys, engine=engine)
    words = ["x" * 300 + "y" * 280, "x" * 301, "x" * 300 + "é" * 150 + "z", "日" * 100, "日" * 99 + "z",
             "x" * 299 + "y" * 281, "x" * 300 + "y" * 279 + "z", "w" * 1000, "w" * 999]
    check(v, [" ".join(words), words[2]], keys, keys.index("[UNK]"), "##", 1024)


@pytest.mark.gpu
def test_raw_keys_inside_a_character_never_match(engine):
    """keys that end inside a multi-byte character (importable as raw bytes) are never a piece"""
    from latok_b200 import _lib
    from latok_b200.vocab import Vocab
    keys = [b"a\xc3", b"\xe6\x97", b"##\xc3", b"a", b"##\xc3\xa9", b"[UNK]", b"\xe6\x97\xa5\xe6", b"\xf0\x9f\x98",
            b"##\xe6\x97\xa5\xe6", b"b\xed\xa0", b"b"]
    v = Vocab(engine)
    buf = np.frombuffer(b"".join(keys), dtype=np.uint8)
    off = np.concatenate([[0], np.cumsum([len(k) for k in keys])]).astype(np.int64)
    _lib.check(v._L.latok_b200_vocab_import(engine._h, v._h, buf.ctypes.data, off.ctypes.data, len(keys), None))
    texts = ["aé 日 日日 😀 a日日 b\ud800 aéé", "ab é"]
    ids, _, _ = check(v, texts, keys, 5)
    assert ids.tolist()[:2] == [3, 4] and 0 not in ids and 1 not in ids and 6 not in ids


@pytest.mark.gpu
def test_empty_batch_and_strings(engine):
    from latok_b200.vocab import Vocab
    keys = ["a", "##b", "[UNK]"]
    v = Vocab.from_tokens(keys, engine=engine)
    ids, offsets, word_off = v.wordpiece([], 2)
    assert ids.tolist() == [] and offsets.tolist() == [0] and word_off.tolist() == [0]
    ids, offsets, word_off = v.wordpiece(["", "  ", "\t \n", ""], 2)
    assert ids.tolist() == [] and offsets.tolist() == [0] * 5 and word_off.tolist() == [0]
    check(v, ["", "ab  a abb", " ", "c ab"], keys, 2)


@pytest.mark.gpu
def test_device_output_and_unchanged_vocabulary(engine):
    import torch
    from latok_b200.engine import pack_strings
    from latok_b200.vocab import Vocab
    texts = fuzz_texts()
    v = Vocab(engine)                                                                  # not frozen, with counts
    v.update(corpus.fuzz_strings(307, 500, 200, "mixed"))
    v.merge(Vocab.from_tokens(recipe(corpus.fuzz_strings(308, 500, 200, "mixed")), engine=engine))
    keys, counts, slots = v.tokens(), v.counts(), v.table_slots()
    unk = -9
    ids_h, off_h, wo_h = check(v, texts, keys, unk)
    ids_d, off_d, wo_d = v.wordpiece_packed(*pack_strings(texts), unk, device=True)
    assert ids_d.is_cuda and ids_d.dtype == torch.int32 and wo_d.is_cuda and wo_d.dtype == torch.int64
    assert ids_d.device.index == engine.device
    assert np.array_equal(ids_d.cpu().numpy(), ids_h) and np.array_equal(wo_d.cpu().numpy(), wo_h)
    assert np.array_equal(np.asarray(off_d), off_h)
    assert v.tokens() == keys and np.array_equal(v.counts(), counts) and v.table_slots() == slots


@pytest.mark.gpu
def test_errors(engine):
    from latok_b200 import _lib
    from latok_b200.engine import SPANS, SPLITS, pack_strings
    from latok_b200.vocab import Vocab
    L = _lib.load()
    v = Vocab.from_tokens(["a", "##b", "[UNK]"], engine=engine)
    n = C.c_int64(-1)
    wo = np.zeros(16, dtype=np.int64)
    ids = np.zeros(16, dtype=np.int32)
    with engine._lock:
        engine.submit(*pack_strings(["ab a abb", "c"]), SPANS)
        assert L.latok_b200_vocab_wordpiece_fetch(engine._h, 16, ids.ctypes.data, 0) == _lib.ESTATE   # before a call
        args = (b"##", 2, 100, 2)
        assert L.latok_b200_vocab_wordpiece(engine._h, v._h, *args, 3, wo.ctypes.data, C.byref(n), 0) == _lib.EINVAL
        assert n.value == -1 and not wo.any()
        for plen, mc in ((-1, 100), (65, 100), (2, 0), (2, 1025)):
            assert L.latok_b200_vocab_wordpiece(engine._h, v._h, b"#" * 65, plen, mc, 2, 16, wo.ctypes.data, C.byref(n),
                                                0) == _lib.EINVAL
        assert L.latok_b200_vocab_wordpiece(engine._h, v._h, *args, 4, wo.ctypes.data, C.byref(n), 0) == _lib.OK
        assert n.value == 7 and wo[:5].tolist() == [0, 2, 3, 6, 7]
        assert L.latok_b200_vocab_wordpiece_fetch(engine._h, 6, ids.ctypes.data, 0) == _lib.EINVAL
        assert not ids.any()
        assert L.latok_b200_vocab_wordpiece_fetch(engine._h, 7, ids.ctypes.data, 0) == _lib.OK
        assert ids[:7].tolist() == [0, 1, 0, 0, 1, 1, 2]
        engine.submit(*pack_strings(["ab"]), SPLITS)
        assert L.latok_b200_vocab_wordpiece_fetch(engine._h, 16, ids.ctypes.data, 0) == _lib.ESTATE   # dropped
        assert L.latok_b200_vocab_wordpiece(engine._h, v._h, *args, 16, wo.ctypes.data, C.byref(n), 0) == _lib.ESTATE
    with pytest.raises(ValueError, match="prefix_len"):
        v.wordpiece(["a"], 2, prefix="#" * 65)
    import torch
    if torch.cuda.device_count() > 1:
        from latok_b200.engine import Engine
        with Engine(1) as e1:
            other = Vocab.from_tokens(["a"], engine=e1)
            with engine._lock:
                engine.submit(*pack_strings(["a"]), SPANS)
                assert L.latok_b200_vocab_wordpiece(engine._h, other._h, *args, 16, wo.ctypes.data, C.byref(n),
                                                    0) == _lib.EINVAL


@pytest.mark.gpu
def test_forced_collisions_three_hash_bits():
    """Every key hashes to one of 7 values: every probe of a candidate compares prefix + piece with the key by bytes."""
    code = f"""
import sys
sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'tests')!r}]
import corpus
from test_gpu_wordpiece import check, recipe, fuzz_texts, PREFIX17
from test_gpu_vocab import hard_keys
from latok_b200.engine import Engine
from latok_b200.vocab import Vocab
with Engine(0) as e:
    texts = corpus.FIXTURES + fuzz_texts()[:400] + hard_keys()[5:]
    for prefix in ("##", "", PREFIX17):
        keys = recipe(corpus.fuzz_strings(311, 80, 80, "mixed"), prefix)
        check(Vocab.from_tokens(keys, engine=e), texts, keys, keys.index("[UNK]"), prefix)
print("ok")
"""
    env = dict(os.environ, LATOK_B200_VOCAB_HASH_BITS="3")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(ROOT))
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-3000:]


def scale_check(engine, name, n):
    """the benchmark's workload: its recipe from batch 1 of the generator, batch 0 split, string by string"""
    import synth
    from latok_b200.core.default_tokenizer import tokenize_packed
    from latok_b200.vocab import Vocab
    gen = synth.tweets if name == "tweets" else synth.mixed_unicode
    seed = 20240601 if name == "tweets" else 20240603
    counter = Vocab(engine)
    counter.encode_packed(*gen(n, seed + 1))
    keys = wordpiece_bench.vocab_tokens(counter.most_common())
    v = Vocab.from_tokens(keys, engine=engine)
    unk = keys.index("[UNK]")
    buf, off = gen(n, seed)
    ids, offsets, word_off = v.wordpiece_packed(buf, off, unk)
    pt = tokenize_packed(buf, off, engine=engine)
    d = {k.encode("utf-8", "surrogatepass"): i for i, k in enumerate(keys)}
    memo, pos, k = {}, 0, 0
    for i in range(n):
        assert offsets[i] == pos, i
        for w in pt.tokens(i):
            if w not in memo:
                memo[w] = wordpiece_ref(w.encode("utf-8", "surrogatepass"), d, unk)
            want = memo[w]
            assert word_off[k] == pos and ids[pos:pos + len(want)].tolist() == want, (i, w)
            pos += len(want)
            k += 1
    assert pos == len(ids) == offsets[-1] and k == len(word_off) - 1
    assert (np.diff(word_off) > 1).mean() > 0.01


@pytest.mark.gpu
def test_scale_200k_tweets(engine):
    scale_check(engine, "tweets", 200_000)


@pytest.mark.gpu
def test_scale_100k_mixed_unicode(engine):
    scale_check(engine, "mixed", 100_000)


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0], [0, 0], [0] * 5, [0] * 7])
def test_sharded_one_device(engine, devices):
    from latok_b200.engine import pack_strings
    from latok_b200.sharding import wordpiece_sharded
    from latok_b200.vocab import Vocab
    keys = recipe(corpus.fuzz_strings(309, 400, 150, "mixed"))
    v = Vocab.from_tokens(keys, engine=engine)
    unk = keys.index("[UNK]")
    for texts in (["aé 日本 xyz", "", "hello wörld " * 30], fuzz_texts()[:300] + hard_keys()):
        buf, off = pack_strings(texts)
        want = v.wordpiece_packed(buf, off, unk, "##", 100)
        got = wordpiece_sharded(v, buf, off, devices, unk, "##", 100)
        for g, w in zip(got, want):
            assert g.dtype == w.dtype and np.array_equal(g, w)


@pytest.mark.gpu
def test_sharded_all_devices():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU: a replica on another device needs two")
    from latok_b200.engine import Engine, pack_strings
    from latok_b200.sharding import wordpiece_sharded
    from latok_b200.vocab import Vocab
    keys = recipe(corpus.fuzz_strings(310, 400, 150, "mixed"))
    with Engine(0) as e0:
        v = Vocab.from_tokens(keys, engine=e0)
        unk = keys.index("[UNK]")
        buf, off = pack_strings(fuzz_texts() + hard_keys())
        want = v.wordpiece_packed(buf, off, unk, PREFIX17, 50)
        for devices in (list(range(n)), list(range(n))[::-1] + [0, 0]):
            got = wordpiece_sharded(v, buf, off, devices, unk, PREFIX17, 50)
            for g, w in zip(got, want):
                assert np.array_equal(g, w)
        assert set(v._replicas) == set(range(1, n))
