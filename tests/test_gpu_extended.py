"""Alignment sweeps (-m gpu): strings a few bytes longer or shorter than every unit of work drift through all
alignments when they are laid end to end -- the kind of input that exposed the token-end bug fixed in round 1
(test_gpu_parity.py::test_token_covering_a_whole_range).  First run on a B200 in round 2 (12 passed); part of the
`gpu` suite since.  Also here: tokens that span two or more whole ranges / a tile boundary (spans only and with token
features), token-feature rows in the order of their ordinals (dense, sparse, > 512 per step), a pre-sized token buffer that is too small (the cap_tokens direct path + the re-run), the in-library
pipeline (depth 2), compact 16-bit spans, and the UCD-15 library check.
"""
import os

import numpy as np
import pytest

import corpus
from oracle import oracle
from test_gpu_parity import check_batch

pytestmark = pytest.mark.gpu

STEP = 1024
GEOMETRIES = {"long": (3968, 9 * 3968), "short": (2944, 11 * 2944)}       # (range, tile) bytes of the two kernel geometries


@pytest.fixture(scope="module", params=["long", "short"])
def engine(request):
    """Every test of this module runs with each geometry of the kernel forced (LATOK_B200_GEOMETRY is read at every
    submit); the sweeps use that geometry's range and tile sizes."""
    from latok_b200.engine import Engine
    old = os.environ.pop("LATOK_B200_GEOMETRY", None)
    os.environ["LATOK_B200_GEOMETRY"] = request.param
    e = Engine(0)
    e.geometry = GEOMETRIES[request.param]
    yield e
    e.close()
    os.environ.pop("LATOK_B200_GEOMETRY", None)
    if old is not None:
        os.environ["LATOK_B200_GEOMETRY"] = old


def _drift(ch, unit_chars, count, spread=12):
    """`count` strings of ch * n with n cycling through unit_chars - spread .. unit_chars + spread."""
    return [ch * (unit_chars - spread + (k % (2 * spread + 1))) for k in range(count)]


@pytest.mark.parametrize("ch,width", [("x", 1), ("é", 2), ("日", 3), ("\U00020000", 4), (",", 1), ("A", 1)])
def test_split_free_strings_around_a_range(engine, ch, width):
    RANGE, TILE5 = engine.geometry
    # no split point inside (or, for ',' and 'A', a symbol / upper-case run): one token per string, ends drift over the
    # closer search windows of consecutive ranges
    texts = _drift(ch, RANGE // width, 600) + _drift(ch, 2 * RANGE // width, 300) + _drift(ch, STEP // width, 400, 5)
    check_batch(engine, texts, 7, label=f"drift {ch!r}")


def test_split_free_strings_around_a_tile(engine):
    RANGE, TILE5 = engine.geometry
    texts = _drift("x", TILE5, 60, 20) + _drift("日", TILE5 // 3, 60, 20) + _drift("x", 7936, 120, 10)
    check_batch(engine, texts, 15, label="drift tile")


@pytest.mark.parametrize("sep", [" ", " a@b,c@d ", "　", " #tag "])
def test_one_separator_drifting_through_long_strings(engine, sep):
    RANGE, TILE5 = engine.geometry
    # a single closer / multi-mark chunk inside an otherwise split-free string of about two ranges
    texts = []
    for k in range(500):
        n = 2 * RANGE + (k % 37) - 18
        cut = (k * 131) % n
        texts.append("x" * cut + sep + "y" * (n - cut))
    check_batch(engine, texts, 7, label=f"one separator {sep!r}")


def test_token_bytes_around_words_and_groups(engine):
    # token byte ranges and the parse matrix: multi-byte strings around the 32-byte words and the 128 KB scan groups of
    # the character prefix (latok_tokbytes.cu)
    from latok_b200.core.default_tokenizer import tokenize_packed
    from latok_b200.engine import pack_strings
    rng = np.random.default_rng(9)
    alphabet = ["a", "é", "日", "\U0001F600", " ", ",", "B"]
    texts = ["".join(rng.choice(alphabet, size=n)) for n in list(range(1, 200, 3)) + [131072 // 2 + d for d in range(-3, 4)]]
    texts += ["é" * n + " z" for n in range(1, 70)] + ["日" * (43690 + d) + " q" for d in range(-2, 3)]
    texts = [t for t in texts if t]
    pt = tokenize_packed(*pack_strings(texts), engine=engine)
    for i, t in enumerate(texts):
        assert pt.tokens(i) == oracle.tokens(t), i
    # the parse matrix uses the same per-word character prefix (and one warp per 32-byte word)
    check_batch(engine, texts, 15, label="words and groups")


def test_tokens_spanning_whole_ranges_and_tiles(engine):
    RANGE, TILE5 = engine.geometry
    # one token that covers 2, 3 and 10 whole ranges (the last one crosses a tile boundary), started and ended at
    # drifting offsets; once with spans only and once with token features (the open-token sums chain, `osum`)
    texts = corpus.tokens_spanning_ranges(RANGE)
    check_batch(engine, texts, 3, label="long tokens, spans")
    check_batch(engine, texts, 7, label="long tokens, token features")


def test_token_feature_rows_in_ordinal_order(engine):
    """Token-feature rows are written in the order of the token ordinals, 32 per trip, staged at their byte phase
    (latok_tok5.cuh, token-feature mode): steps with few, many and more than 512 token ends (the per-lane fallback),
    the 25-byte rows at every phase of a 16-byte chunk, tokens longer than 255 characters (uint8 wrap-around of the
    sums, latok.c:342-354), tokens that begin several lane-words / steps / ranges before they end."""
    RANGE, _ = engine.geometry
    texts = corpus.token_feature_rows(RANGE)
    check_batch(engine, texts, 7, label="token-feature rows")
    # exactly around the list capacity: 505..520 token ends in the first step of a string, then sparse text
    check_batch(engine, corpus.token_feature_rows_at_capacity(), 7, label="token-feature rows around the list capacity")
    # one token / a handful of tokens per batch (the trip's first and last chunk are the same one)
    for t in corpus.TINY_BATCHES:
        check_batch(engine, t, 7, label=f"token-feature rows, tiny batch {t!r}")


def test_small_presized_token_buffer(engine):
    # an engine whose token buffers were sized for a tiny batch: the kernel's cap_tokens path (direct span writes are
    # bounds-checked, error bit 2), then the re-run with grown buffers
    from latok_b200.engine import Engine
    texts = ["a b c d e f g h i j k l m n o p q r s t u v w x y z " * 40 for _ in range(400)]
    with Engine(0, 4096, 8) as small:
        for what in (3, 7):
            r = small.run(["tiny"], what)
            assert r.n_tokens == 1
            check_batch(small, texts, what, label=f"regrow what={what}")


def test_pipeline_depth_two(engine):
    # the in-library double buffering: results of a pipelined pass equal those of one-at-a-time submits, in order
    from latok_b200.engine import Engine, pack_strings
    batches = [pack_strings(corpus.fuzz_strings(300 + i, 2000 + 900 * (i % 3), 80, "mixed")) for i in range(7)]
    with Engine(0) as e:
        got = list(e.stream(iter(batches), 1 | 2 | 4))
        assert len(got) == len(batches)
        for (buf, off), r in zip(batches, got):
            o = oracle.tokenize_batch_utf8(buf, off, feats=True)
            assert np.array_equal(r.splits, o["splits"]) and np.array_equal(r.spans, o["spans"])
            assert np.array_equal(r.tok_offsets, o["tok_offsets"]) and np.array_equal(r.tok_feats, o["tok_feats"])
        # depth-2 protocol errors: a third submit, fetch with too small capacities
        e.set_pipeline_depth(2)
        e.submit(*batches[0]); e.submit(*batches[1])
        with pytest.raises(RuntimeError):
            e.submit(*batches[2])
        r0 = e.fetch(); e.release()
        r1 = e.fetch(); e.release()
        assert r0.n_strings == len(batches[0][1]) - 1 and r1.n_strings == len(batches[1][1]) - 1
        with pytest.raises(RuntimeError):
            e.release()
        e.set_pipeline_depth(1)
        r = e.run_packed(*batches[3])
        assert np.array_equal(r.spans, got[3].spans)


def test_fetch_checks_capacities(engine):
    import ctypes as C
    from latok_b200 import _lib
    from latok_b200.engine import pack_strings
    buf, off = pack_strings(corpus.fuzz_strings(77, 500, 60, "mixed"))
    engine.submit(buf, off, 3)
    c, t = engine.sizes()
    L = _lib.load()
    sp = np.zeros((t, 2), np.int32)
    assert L.latok_b200_fetch(engine._h, c, t - 1, len(off) - 1, None, None, sp.ctypes.data, None, None, None) == _lib.EINVAL
    assert not sp.any()
    spl = np.zeros(c, np.int8)
    assert L.latok_b200_fetch(engine._h, c - 1, t, len(off) - 1, spl.ctypes.data, None, None, None, None, None) == _lib.EINVAL
    assert L.latok_b200_fetch(engine._h, c, t, len(off) - 1, spl.ctypes.data, None, sp.ctypes.data, None, None, None) == _lib.OK
    assert sp.any() and spl.any()


def test_compact_spans16(engine):
    from latok_b200.engine import SPANS16, pack_strings
    texts = corpus.FIXTURES + corpus.fuzz_strings(5, 3000, 200, "mixed") + ["w " * 30000]
    buf, off = pack_strings(texts)
    r32 = engine.run_packed(buf, off, 2)
    r16 = engine.run_packed(buf, off, SPANS16)
    assert r16.spans.dtype == np.uint16 and np.array_equal(r16.spans.astype(np.int32), r32.spans)
    assert np.array_equal(r16.tok_offsets, r32.tok_offsets)
    # a string of 65 536+ characters cannot be expressed: the fetch fails, nothing silently wraps
    with pytest.raises(ValueError):
        engine.run_packed(*pack_strings(["x " * 40000]), SPANS16)
    assert engine.run_packed(*pack_strings(["x " * 40000]), 2).n_tokens == 40000


def test_ucd15_library():
    """SURVEY 8 f4: a library built over the class ranges of a newer UCD (tools/build_ucd_variant.py, run by
    __graft_entry__.build()) against an oracle built over the same ranges: every code point in three arrangements +
    fuzz, all outputs bit-exact (tools/ucd_check.py)."""
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    lib, orc = root / "latok_b200" / "_variants" / "liblatok_ucd.so", root / "latok_b200" / "_variants" / "liblatok_oracle_ucd.so"
    if not (lib.exists() and orc.exists()):
        pytest.skip("latok_b200/_variants/ not built (python tools/build_ucd_variant.py)")
    p = subprocess.run([sys.executable, str(root / "tools" / "ucd_check.py")], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, LATOK_B200_LIB=str(lib), LATOK_ORACLE_LIB=str(orc)))
    assert p.returncode == 0 and "ucd check ok" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]
