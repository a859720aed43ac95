"""Parity of the CUDA path (through the C ABI) against the CPU oracle: bit-exact split masks, token
spans, CSR offsets, per-token feature sums and feature matrices.  Needs a B200 (-m gpu)."""
import json
import zlib

import numpy as np
import pytest

import corpus
from oracle import oracle

pytestmark = pytest.mark.gpu

ALL = 1 | 2 | 4 | 8
# units of work of the two kernel geometries (corpus.py)
RANGES = corpus.RANGES
UNITS = corpus.UNITS
TILE = 7936


@pytest.fixture(scope="module", params=["auto", "long", "short"])
def engine(request):
    """Every test of this module runs three times: with the geometry the library picks for the batch (by average string
    length), and with each of the two forced (LATOK_B200_GEOMETRY is read at every submit)."""
    import os
    from latok_b200.engine import Engine
    old = os.environ.pop("LATOK_B200_GEOMETRY", None)
    if request.param != "auto":
        os.environ["LATOK_B200_GEOMETRY"] = request.param
    e = Engine(0)
    yield e
    e.close()
    os.environ.pop("LATOK_B200_GEOMETRY", None)
    if old is not None:
        os.environ["LATOK_B200_GEOMETRY"] = old


def check_batch(engine, texts, what=ALL, rules=None, label=""):
    if (what & 12) and (what & 3):
        # the tokenize kernel has an instantiation with token features and one without: check both
        check_batch(engine, texts, what & 3, rules, label + " [splits+spans only]")
    r = engine.run(texts, what)
    o = oracle.tokenize_batch(texts, rules=rules or oracle.DEFAULT_RULES, matrix=bool(what & 8), feats=bool(what & 4))
    assert r.n_chars == o["n_chars"], label
    assert np.array_equal(r.char_offsets, o["char_offsets"]), label
    if what & 1:
        bad = np.nonzero(r.splits != o["splits"])[0]
        assert bad.size == 0, f"{label}: split mask differs at chars {bad[:10]} (of {bad.size})"
    if what & 8:
        bad = np.nonzero((r.matrix != o["matrix"]).any(axis=1))[0]
        assert bad.size == 0, f"{label}: matrix differs at chars {bad[:10]} (of {bad.size})"
    if what & (2 | 4):
        assert r.n_tokens == o["n_tokens"], f"{label}: {r.n_tokens} tokens vs {o['n_tokens']}"
        assert np.array_equal(r.tok_offsets, o["tok_offsets"]), label
    if what & 2:
        bad = np.nonzero((r.spans != o["spans"]).any(axis=1))[0]
        assert bad.size == 0, f"{label}: spans differ at tokens {bad[:10]}: {r.spans[bad[:5]]} vs {o['spans'][bad[:5]]}"
    if what & 4:
        bad = np.nonzero((r.tok_feats != o["tok_feats"]).any(axis=1))[0]
        assert bad.size == 0, f"{label}: token feats differ at tokens {bad[:10]}"
    return r


def test_fixture_strings(engine):
    check_batch(engine, corpus.FIXTURES, label="fixtures")
    # one at a time (every string is also its own batch, tile 0 with the terminator in the window)
    for t in corpus.FIXTURES:
        check_batch(engine, [t], label=repr(t[:30]))


def test_golden_reference_outputs(engine, golden_dir):
    """GPU results against the committed outputs of the reference itself (not via the oracle)."""
    recs = json.load(open(golden_dir / "reference_outputs.json"))["records"]
    texts = [r["text"] for r in recs]
    res = engine.run(texts, ALL)
    for i, r in enumerate(recs):
        w = np.asarray(r["matrix_words"], dtype=np.int64)[:, None]
        assert np.array_equal(res.string_matrix(i), ((w >> np.arange(25)) & 1).astype(np.int8)), r["text"]
        assert res.string_splits(i).tolist() == r["splits"], r["text"]
        sp = res.string_spans(i)
        assert [r["text"][a:b].strip() for a, b in sp] == r["tokens"], r["text"]
        if "feats" in r:
            assert sp.tolist() == r["feat_spans"], r["text"]
            assert res.string_feats(i).tolist() == r["feats"], r["text"]


def test_notebook_cell(engine, golden_dir):
    cell = json.load(open(golden_dir / "notebook_cell.json"))
    res = engine.run([cell["text"]], 1 | 8)
    assert res.matrix.tolist() == cell["matrix"]
    assert res.splits.tolist() == cell["splits"]


def test_empty_inputs(engine):
    check_batch(engine, [], label="no strings")
    check_batch(engine, [""], label="one empty")
    check_batch(engine, ["", "", ""], label="three empty")
    check_batch(engine, ["", "a", "", "", "b c", ""], label="ragged")
    check_batch(engine, [""] * 3000 + ["x"] + [""] * 3000, label="many empty")


@pytest.mark.parametrize("seed,count,max_len,profile", [
    (1, 6000, 60, "mixed"), (2, 6000, 140, "ascii"), (3, 6000, 100, "marks"), (4, 400, 3000, "mixed"),
    (5, 20000, 12, "mixed"), (6, 3000, 300, "marks"),
])
def test_fuzz(engine, seed, count, max_len, profile):
    check_batch(engine, corpus.fuzz_strings(seed, count, max_len, profile), label=f"fuzz {profile} {seed}")


def test_every_code_point(engine, golden_dir):
    want = np.frombuffer(zlib.decompress((golden_dir / "codepoint_classes.bin").read_bytes()), dtype=np.uint16)
    step = 1 << 16
    texts = ["".join(chr(c) for c in range(b, b + step)) for b in range(0, 0x110000, step)]
    res = engine.run(texts, 8)
    got = (res.matrix[:, :12].astype(np.uint16) << np.arange(12, dtype=np.uint16)).sum(axis=1).astype(np.uint16)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [hex(int(b)) for b in bad[:10]]


_long_doc = corpus.long_doc


def test_long_documents_cross_tiles(engine):
    check_batch(engine, corpus.long_documents(), label="long docs")


def test_boundary_alignment_sweep(engine):
    """Slide interesting patterns across the tile boundary one byte at a time."""
    for unit in UNITS:
        texts = corpus.alignment_sweep(unit)
        check_batch(engine, texts, label=f"alignment sweep {unit} (one string per case)")
        # same but as one long string so the boundary falls inside a string at many different phases
        check_batch(engine, [" ".join(texts[:20])], label=f"alignment sweep {unit} (joined)")
    # the same patterns against the 1 KB steps inside a range and against the 116-byte closer search windows
    check_batch(engine, corpus.alignment_sweep_steps(), label="alignment sweep (steps / search windows)")


def test_multibyte_straddling_tiles(engine):
    for ch in corpus.STRADDLE_CHARS:
        n = len(ch.encode("utf-8"))
        check_batch(engine, corpus.multibyte_straddle(ch), label=f"straddle {ch!r} ({n} bytes)")


def test_long_space_free_runs_and_walk(engine):
    """Chunks longer than the right halo force the look-ahead walk; marks far ahead must blank
    characters in earlier tiles (latok.c:218-244 has unbounded reach)."""
    cases = corpus.space_free_runs()
    r = check_batch(engine, cases, label="space-free runs")
    assert r.lookahead_walks > 0
    # multibyte inside the long run
    check_batch(engine, corpus.cjk_runs(), label="cjk run")


def test_backlog_across_tiles(engine):
    """Q2: k marks in one whitespace chunk blank the following k-1 chunks too; make the backlog
    cross tile boundaries and string boundaries (it must reset at each string start)."""
    texts = corpus.backlog_across_tiles()
    check_batch(engine, texts, label="backlog")


def test_many_tiny_strings_and_long_mixed(engine):
    rng = np.random.default_rng(7)
    texts = []
    for _ in range(200):
        texts += corpus.fuzz_strings(int(rng.integers(1 << 30)), 50, 8)
        texts.append(_long_doc(rng, int(rng.integers(10, 40000)), "mixed"))
    check_batch(engine, texts, label="tiny+long mix")


def test_partial_outputs(engine):
    texts = corpus.fuzz_strings(99, 3000, 80)
    for what in (1, 2, 1 | 2, 2 | 4, 8, 1 | 8, 4):
        check_batch(engine, texts, what=what, label=f"what={what}")


def test_token_capacity_regrow(engine):
    """A symbol-only corpus has one token per character: the span buffers must grow and the batch rerun."""
    from latok_b200.engine import Engine
    with Engine(0) as e:
        check_batch(e, ["!?" * 40000, "a b " * 5000], label="regrow")


def test_custom_rules(engine):
    from latok_b200.core import offsets as oft
    from latok_b200.core.latok_utils import build_combo_matrix
    c_split = build_combo_matrix([[oft.SPACE_IDX], [oft.SYMBOL_IDX, oft.NEXT_ALPHA_IDX], [oft.NUM_IDX, oft.PREV_ALPHA_IDX]])
    c_mask = build_combo_matrix([[oft.CHAR_SLASH_IDX, oft.NEXT_ALPHA_NUM_IDX], [oft.TWITTER_IDX]])
    c_sym = build_combo_matrix([[oft.SYMBOL_IDX, oft.NEXT_SPACE_IDX], [oft.CHAR_PERIOD_IDX]])
    from latok_b200.engine import Engine
    with Engine(0) as e:
        e.set_rules(c_split, c_mask, c_sym)
        texts = corpus.FIXTURES + corpus.fuzz_strings(5, 3000, 80, "marks")
        check_batch(e, texts, rules=(c_split, c_mask, c_sym), label="custom rules")
        e.set_rules()  # back to defaults
        check_batch(e, texts, label="defaults restored")
        with pytest.raises(ValueError):
            e.set_rules(build_combo_matrix([[oft.SYMBOL_IDX]]), c_mask, c_sym)   # no [SPACE] row
        with pytest.raises(ValueError):
            e.set_rules(build_combo_matrix([[oft.SPACE_IDX], [99]]), c_mask, c_sym)


def test_bad_offsets_rejected(engine):
    buf = np.frombuffer(b"hello world", dtype=np.uint8)
    with pytest.raises(ValueError):
        engine.run_packed(buf, np.array([0, 7, 5, 11], dtype=np.int64))
    with pytest.raises(ValueError):
        engine.run_packed(buf, np.array([1, 11], dtype=np.int64))
    # engine still usable afterwards
    check_batch(engine, ["still fine"], label="after error")


def test_back_to_back_submits_alternate_index_sets(engine):
    """Several device-resident batches submitted without waiting in between (the string index of batch i+1 is built on
    an aux stream while batch i is tokenized; two index / result sets alternate): the results are those of the last one,
    whichever kernel instantiation (split mask + spans, or with token features and the matrix) each batch used."""
    torch = pytest.importorskip("torch")
    from latok_b200.engine import pack_strings
    batches = [corpus.fuzz_strings(100 + i, 3000 + 700 * i, 60 + 30 * i, "mixed") for i in range(5)]
    dev = []
    for texts in batches:
        b, o = pack_strings(texts)
        dev.append((torch.from_numpy(b.copy()).cuda(), torch.from_numpy(o.copy()).cuda(), len(texts)))
    torch.cuda.synchronize()
    for order, whats in (((0, 1, 2, 3, 4), (3, 3, 3, 3, 3)), ((4, 2, 0, 3, 1), (3, 7, 3, 15, 3)), ((1, 1, 3), (7, 3, 3))):
        for i, what in zip(order, whats):
            b, o, n = dev[i]
            engine.submit_device(b.data_ptr(), o.data_ptr(), n, b.numel(), what)
        last, what = order[-1], whats[-1]
        r = engine.fetch()
        ref = oracle.tokenize_batch(batches[last])
        assert r.n_chars == ref["n_chars"] and r.n_tokens == ref["n_tokens"]
        assert np.array_equal(r.splits, ref["splits"]) and np.array_equal(r.spans, ref["spans"])
        assert np.array_equal(r.char_offsets, ref["char_offsets"]) and np.array_equal(r.tok_offsets, ref["tok_offsets"])


def test_backlog_handoff_between_ranges(engine):
    """A chunk with several marks that ends right at a range end hands its backlog to the next range (the service warp's
    settle(): the next range repeats its ordinary analysis with the backlog entering): swept over the range end, with
    hand-offs in consecutive ranges (cascade), across a tile boundary, from a tile's last range into the next tile, and
    with backlogs larger than one."""
    texts = corpus.handoff_between_ranges()
    check_batch(engine, texts[:40], ALL, label="hand-off, all outputs")
    check_batch(engine, texts, 3, label="hand-off")
    # the same chunks with no space after them for a long while: the backlog is carried through several ranges
    check_batch(engine, corpus.handoff_long_tail(), 7, label="hand-off into a space-free run")


def test_token_covering_a_whole_range(engine):
    """A token (here: a whole string without a split point) that begins in one range, covers the next one completely
    and ends within the closer search window of the third: the middle range must write its end.  Strings of 4-byte
    characters a few bytes longer than a range drift through every alignment (found by tools/ucd_check.py)."""
    texts = corpus.token_over_whole_range()
    check_batch(engine, texts, 3, label="token over a whole range")
    check_batch(engine, texts[:400], 7, label="token over a whole range, token features")
