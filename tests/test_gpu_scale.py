"""Full-size BASELINE configs on the GPU: size-independent invariants over the whole batch plus EXACT parity with the
oracle on every string of the batch (tests/fullcheck.py: the oracle's C batch path over a pool of processes).  -m gpu."""
import numpy as np
import pytest

import fullcheck
from oracle import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from latok_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def check_invariants(buf, off, r, feats=False):
    S = len(off) - 1
    lead = ((buf & 0xC0) != 0x80).astype(np.int64)
    cum = np.concatenate([[0], np.cumsum(lead)])
    assert np.array_equal(r.char_offsets, cum[off]), "per-string character counts != UTF-8 lead-byte counts"
    assert r.n_chars == int(cum[-1]) and len(r.splits) == r.n_chars
    assert r.tok_offsets[0] == 0 and r.tok_offsets[-1] == r.n_tokens and np.all(np.diff(r.tok_offsets) >= 0)
    L = np.diff(r.char_offsets)
    nonempty = L > 0
    assert np.all(r.splits[r.char_offsets[:-1][nonempty]] == 1), "first character of a string is always a boundary (=1)"
    assert r.splits.min() >= 0 and r.splits.max() <= 5
    # spans: inside their string, ordered, start on a split, end on a split or the string end, no split inside
    sid = np.repeat(np.arange(S), np.diff(r.tok_offsets))
    st, en = r.spans[:, 0].astype(np.int64), r.spans[:, 1].astype(np.int64)
    assert np.all((0 <= st) & (st < en) & (en <= L[sid]))
    same = sid[1:] == sid[:-1]
    assert np.all(en[:-1][same] <= st[1:][same]), "tokens of a string are disjoint and ordered"
    g0 = r.char_offsets[sid]
    assert np.all(r.splits[g0 + st] != 0)
    inner_end = en < L[sid]
    assert np.all(r.splits[(g0 + en)[inner_end]] != 0)
    nzc = np.concatenate([[0], np.cumsum(r.splits != 0)])
    assert np.all(nzc[g0 + en] - nzc[g0 + st + 1] == 0), "a token contains no split point besides its first character"
    if feats:
        assert r.tok_feats.shape == (r.n_tokens, 25)
        # ALPHA_NUM >= ALPHA, ALPHA_NUM >= NUM per token while nothing wraps (short tokens)
        short = (en - st) < 120
        assert np.all(r.tok_feats[short, 1] >= r.tok_feats[short, 0]) and np.all(r.tok_feats[short, 1] >= r.tok_feats[short, 2])


def check_sample(buf, off, r, idx, feats=False):
    import synth
    raw = buf.tobytes()
    for i in idx:
        t = raw[off[i]:off[i + 1]].decode("utf-8")
        m = oracle.parse_matrix(t)
        s = oracle.split_mask(m) if len(t) else np.zeros(0, np.int8)
        assert np.array_equal(r.string_splits(i), s), f"string {i}: split mask"
        sp, _ = oracle.spans(s, m)
        assert np.array_equal(r.string_spans(i), sp), f"string {i}: spans"
        if feats:
            assert np.array_equal(r.string_feats(i), oracle.token_feats(m, sp)), f"string {i}: token features"


def test_config2_one_million_tweets(engine):
    import synth
    buf, off = synth.tweets(1_000_000)
    r = engine.run_packed(buf, off, 1 | 2)
    check_invariants(buf, off, r)
    assert fullcheck.compare_all(buf, off, r) == 1_000_000          # every string: split mask, spans, CSR offsets
    check_sample(buf, off, r, range(0, 50))                         # (and a few through the per-string oracle calls)
    r2 = engine.run_packed(buf, off, 1 | 2)     # deterministic
    assert np.array_equal(r.splits, r2.splits) and np.array_equal(r.spans, r2.spans)
    # sharding property: two byte-balanced halves tokenized separately concatenate to the whole
    from latok_b200 import sharding
    halves = sharding.tokenize_sharded(buf, off, [0, 0])
    assert np.array_equal(halves.splits, r.splits) and np.array_equal(halves.spans, r.spans)
    assert np.array_equal(halves.tok_offsets, r.tok_offsets) and np.array_equal(halves.char_offsets, r.char_offsets)


def test_config4_mixed_unicode_with_classification(engine):
    import synth
    buf, off = synth.mixed_unicode(1_000_000)
    r = engine.run_packed(buf, off, 1 | 2 | 4)
    check_invariants(buf, off, r, feats=True)
    assert fullcheck.compare_all(buf, off, r, feats=True) == 1_000_000      # every string, token feature sums included
    check_sample(buf, off, r, range(0, 50), feats=True)
    r3 = engine.run_packed(buf, off, 1 | 2)                                   # the kernel instantiation without token features
    assert np.array_equal(r3.splits, r.splits) and np.array_equal(r3.spans, r.spans) and np.array_equal(r3.tok_offsets, r.tok_offsets)


def test_config3_long_documents(engine):
    import synth
    # 1.07 GB of unique text (8 blocks of 2 000 documents generated in parallel), incl. >= 32 KB space-free runs and
    # multi-mark (backlog) chunks: every document compared with the oracle
    import bench
    buf, off = bench.generate({"d": [("docs", 2000, 20240602 + 1000 * k) for k in range(8)]})["d"]
    assert len(buf) > 1_000_000_000
    r = engine.run_packed(buf, off, 1 | 2)
    check_invariants(buf, off, r)
    assert fullcheck.compare_all(buf, off, r, target_bytes=8 << 20) == 16_000
    assert r.lookahead_walks > 0                 # the corpus does exercise the look-ahead walk


def test_parse_matrix_past_2gb(engine):
    """More than 86 M characters: the matrix passes 2^31 bytes (64-bit row offsets in parse_matrix_kernel).  The strings
    whose rows lie past that byte, against the oracle."""
    import synth
    buf, off = synth.tweets(700_000)
    r = engine.run_packed(buf, off, 8)
    assert r.n_chars == int(((buf & 0xC0) != 0x80).sum()) and r.n_chars * 25 > 2 ** 31
    first = int(np.searchsorted(r.char_offsets, 2 ** 31 // 25, side="right")) - 1       # holds the row at byte 2^31
    raw = buf.tobytes()
    S = len(off) - 1
    for i in list(range(first, first + 2000)) + list(range(S - 2000, S)):
        t = raw[off[i]:off[i + 1]].decode("utf-8")
        assert np.array_equal(r.string_matrix(i), oracle.parse_matrix(t)), f"string {i}"
