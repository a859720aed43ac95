"""Custom tokenizer rules (-m gpu): `Engine.set_rules` runs the generic instantiation of the tokenize kernel (rule terms
summed into 4 count and 4 sym planes, 5 split-value planes, the parked state in its own buffer, its own occupancy).
Every result is compared bit for bit with the oracle under the same rules: named rule sets that each drive one part of
the generic path, the long-string scenarios of the default-rule sweeps (corpus.py), mask rows that fire on chunk
closers (a space, the last character of a string), a seeded rule fuzz, the consumers of the spans, the rules a
pipelined batch was submitted with, and the rejected rule sets.  Both kernel geometries are forced in turn."""
import os
from collections import Counter

import numpy as np
import pytest

import corpus
from oracle import oracle
from oracle.oracle import (ALPHA, ALPHA_NUM, NUM, LOWER, UPPER, SPACE, SYMBOL, TWITTER, CHAR_AT, CHAR_COLON,
                           CHAR_SLASH, CHAR_PERIOD, PREV_ALPHA, NEXT_ALPHA, PREV_ALPHA_NUM, NEXT_ALPHA_NUM, PREV_LOWER,
                           NEXT_LOWER, PREV_SPACE, NEXT_SPACE, PREV_SYMBOL, NEXT_AT, NEXT_SLASH, AFTER_NEXT_ALPHA,
                           AFTER_NEXT_SLASH, combo)
from test_gpu_parity import check_batch

pytestmark = pytest.mark.gpu

GEOMETRIES = {"long": (3968, 9 * 3968), "short": (2944, 11 * 2944)}       # (range, tile) bytes of the two kernel geometries
MAX_ROWS = 15                                                              # MAX_RULE_ROWS (latok_internal.h)
NONE = np.zeros((0, 1), np.int8)                                           # a rule matrix without rows
C_SPLIT, C_MASK, C_SYM = oracle.DEFAULT_RULES


def _permuted(m, extra_cols=2):
    """The rows of `m` in reverse order, each row's columns reversed, padded with trailing -1 columns."""
    rows = [[int(v) for v in r if v >= 0][::-1] for r in m][::-1]
    out = np.full((len(rows), m.shape[1] + extra_cols), -1, np.int8)
    for i, r in enumerate(rows):
        out[i, :len(r)] = r
    return out


RULES = {
    # the set of test_gpu_parity.py::test_custom_rules
    "parity": (combo([[SPACE], [SYMBOL, NEXT_ALPHA], [NUM, PREV_ALPHA]]),
               combo([[CHAR_SLASH, NEXT_ALPHA_NUM], [TWITTER]]),
               combo([[SYMBOL, NEXT_SPACE], [CHAR_PERIOD]])),
    # mask rows that fire on closers: a space after a symbol, a trailing # @ $ ^, a symbol at the end of a string
    "closer_marks": (C_SPLIT, combo([[SPACE, PREV_SYMBOL], [TWITTER], [SYMBOL, NEXT_SPACE]]), C_SYM),
    # every letter is a mark: backlogs of thousands cross ranges and tiles
    "dense_marks": (C_SPLIT, combo([[ALPHA]]), C_SYM),
    # 15 + 15 rows that fire together: a split value of 30 at every space (the top of the 5 value planes)
    "max_counts": (combo([[SPACE]] * MAX_ROWS), C_MASK, combo([[SPACE]] * MAX_ROWS)),
    # no mask rows (the block mask is all ones) / no sym rows
    "no_mask": (C_SPLIT, NONE, C_SYM),
    "no_sym": (C_SPLIT, C_MASK, NONE),
    # every context column: their values at string starts and ends and across range edges decide the result
    "context": (combo([[SPACE], [NEXT_SPACE, ALPHA], [PREV_SPACE, ALPHA_NUM], [PREV_SYMBOL], [NEXT_AT],
                       [AFTER_NEXT_SLASH], [UPPER, PREV_LOWER], [LOWER, NEXT_LOWER, PREV_ALPHA_NUM]]),
                combo([[NEXT_SLASH, PREV_ALPHA], [AFTER_NEXT_ALPHA, PREV_SPACE, SYMBOL], [CHAR_AT, NEXT_ALPHA_NUM],
                       [CHAR_COLON, PREV_ALPHA_NUM], [CHAR_PERIOD, NEXT_ALPHA]]),
                combo([[NEXT_LOWER, PREV_LOWER, SYMBOL], [NEXT_ALPHA, SYMBOL], [NEXT_SPACE, PREV_SPACE],
                       [PREV_ALPHA, NEXT_AT]])),
    # the default rows in another order and with padding: still the default instantiation, default outputs
    "default_permuted": (_permuted(C_SPLIT), _permuted(C_MASK), _permuted(C_SYM, 1)),
    # the default rows with [SYMBOL] twice: the generic instantiation, the row counts twice
    "default_plus_one": (np.concatenate([C_SPLIT, combo([[SYMBOL, -1]])]), C_MASK, C_SYM),
}
# the mask rows of "closer_marks" one at a time: a mark on a closer with no other mark in its chunk (in the combined
# set the symbol in front of a marked space is a mark too)
CLOSER_ROWS = {
    "space_after_symbol": (C_SPLIT, combo([[SPACE, PREV_SYMBOL]]), C_SYM),
    "twitter": (C_SPLIT, combo([[TWITTER]]), C_SYM),
    "symbol_at_end": (C_SPLIT, combo([[SYMBOL, NEXT_SPACE]]), C_SYM),
    "closer_marks": RULES["closer_marks"],
}


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


def _check(engine, name, rules, texts, what, label):
    engine.set_rules(*rules)
    return check_batch(engine, texts, what, rules=rules, label=f"{name}: {label}")


# ---------------------------------------------------------------------------------------------- named rule sets
@pytest.mark.parametrize("name", list(RULES))
def test_fixtures(engine, name):
    rules = RULES[name]
    for what in (15, 3):
        _check(engine, name, rules, corpus.FIXTURES, what, f"fixtures what={what}")
        # one string per batch: one step without a chunk that holds two marks takes the block mask's fast path
        for t in corpus.FIXTURES:
            _check(engine, name, rules, [t], what, f"{t[:30]!r} what={what}")


@pytest.mark.parametrize("name", list(RULES))
def test_long_scenarios(engine, name):
    """The long-string scenarios of the default-rule sweeps (test_gpu_parity.py, test_gpu_extended.py) under every
    named set: documents across tiles, patterns slid over every unit, multi-byte characters straddling them, long
    space-free runs (the look-ahead walk), backlogs across tiles and handed from range to range, tokens over whole
    ranges, token-feature rows in the order of their ordinals."""
    rules = RULES[name]
    RANGE, _ = engine.geometry
    for what in (15, 3):
        _check(engine, name, rules, corpus.long_documents(), what, f"long docs what={what}")
        _check(engine, name, rules, corpus.alignment_sweep_steps(), what, f"alignment sweep (steps) what={what}")
        _check(engine, name, rules, corpus.backlog_across_tiles(), what, f"backlog what={what}")
    for unit in engine.geometry:             # this geometry's range and tile
        _check(engine, name, rules, corpus.alignment_sweep(unit), 7, f"alignment sweep {unit}")
    for ch in corpus.STRADDLE_CHARS:
        _check(engine, name, rules, corpus.multibyte_straddle(ch), 7, f"straddle {ch!r}")
    r = _check(engine, name, rules, corpus.space_free_runs(), 7, "space-free runs")
    # (with every letter a mark, a mark is pending wherever a chunk runs past a tile: no walk is needed)
    assert r.lookahead_walks > 0 or name == "dense_marks", name
    _check(engine, name, rules, corpus.cjk_runs(), 7, "cjk run")
    handoff = corpus.handoff_between_ranges()
    _check(engine, name, rules, handoff[:40], 15, "hand-off, all outputs")
    _check(engine, name, rules, handoff, 3, "hand-off")
    _check(engine, name, rules, corpus.handoff_long_tail(), 7, "hand-off into a space-free run")
    _check(engine, name, rules, corpus.token_over_whole_range(), 3, "token over a whole range")
    _check(engine, name, rules, corpus.tokens_spanning_ranges(RANGE), 7, "long tokens")
    _check(engine, name, rules, corpus.token_feature_rows(RANGE), 7, "token-feature rows")
    _check(engine, name, rules, corpus.token_feature_rows_at_capacity(), 7, "token-feature rows at the list capacity")


def test_dense_marks_backlog_over_many_tiles(engine):
    """~200 000 letters (200 000 marks in one chunk) followed by ~3 000 short words: the backlog blanks thousands of
    chunks over many ranges and tiles; then the same behind a string boundary, which resets it."""
    name, rules = "dense_marks", RULES["dense_marks"]
    words = " ".join(f"w{i}" for i in range(3000))
    texts = ["x" * 200000 + " " + words, "ab " * 50 + "y" * 199999 + " " + words + " " + "tail, end!"]
    _check(engine, name, rules, texts, 7, "200 000 marks")
    _check(engine, name, rules, ["z" * 200000, words], 7, "200 000 marks, then a new string")


@pytest.mark.parametrize("name", ["default_permuted", "default_plus_one"])
def test_default_rows_reordered_or_repeated(engine, name):
    """Rules equal to the defaults up to row order and padding give the default outputs; one duplicated row changes
    them.  (Equal outputs do not show which instantiation ran -- a correct generic one gives them too, and the API
    does not expose the choice; `latok_b200_set_rules` compares the rows as sets, and the default instantiation's
    code is checked by the default-rule tests.)"""
    rules = RULES[name]
    texts = corpus.FIXTURES + corpus.fuzz_strings(11, 2000, 120, "marks")
    engine.set_rules(*rules)
    r = check_batch(engine, texts, 15, rules=rules, label=name)
    engine.set_rules()
    d = engine.run(texts, 15)
    if name == "default_permuted":
        for a in ("splits", "spans", "tok_offsets", "tok_feats", "matrix"):
            assert np.array_equal(getattr(r, a), getattr(d, a)), a
    else:
        assert not np.array_equal(r.splits, d.splits)


# ------------------------------------------------------------------------------------------- marks on closers
def closer_mark_sweep(range_bytes, ends, count=160):
    """Strings laid end to end in one batch, each a space-free run of 120..540 characters that ends with a mark on
    a closer -- a trailing `#` or `!` (the last character of the string), or a space after a symbol -- at a byte
    position that drifts from 60 bytes in front of a range end to 300 behind it.  A range end is every `range_bytes`
    bytes, so every 9th / 11th one is a tile end; the run straddles it, or covers the next range's closer search
    window (then the next range begins inside the chunk, and the mark on that chunk's closer -- counted in the next
    range's summary of marks in front of its first closer -- decides whether the open tail of this one is blanked).
    The run is ",ab" repeated: every comma is a split point unless the block mask blanks it, so a tail that is
    wrongly kept or blanked changes the splits in the range that owns it."""
    filler = "lorem ipsum dolor sit amet consectetur "
    texts, g = [], 0
    for j in range(count):
        end = ends[j % len(ends)]
        run = 120 + (j * 41) % 421
        d = (j * 23) % 361 - 60
        target = ((g + run + 200) // range_bytes + 1) * range_bytes + d     # batch byte of the closer that is a mark
        head = target - g - run - (len(end) - 1)
        body = (filler * (head // len(filler) + 1))[:head - 1] + " " + (",ab" * run)[:run] + end
        tail = " a b" if end.endswith(" ") else ""
        texts.append(body + tail)
        g += len(body) + len(tail)
    return texts


@pytest.mark.parametrize("name", list(CLOSER_ROWS))
def test_closer_marks(engine, name):
    rules = CLOSER_ROWS[name]
    RANGE, _ = engine.geometry
    # the examples of the analysis (one string, one step: the fast path)
    for t in ("x a,b#", "a,b! c,d e", "#", "a#", "x!", "a, b", "q@", "ab ,c d!", "!" * 40, "w " * 40 + "k!"):
        _check(engine, name, rules, [t], 7, repr(t))
    for ends in (("#",), ("!",), (", ",), ("#", "!", "; ")):
        _check(engine, name, rules, closer_mark_sweep(RANGE, ends), 7, f"sweep {ends}")
    _check(engine, name, rules, closer_mark_sweep(RANGE, ("#", "!", ", "), 40), 15, "sweep, all outputs")


# ------------------------------------------------------------------------------------------------ rule fuzz
def random_rules(seed):
    """1..15 split rows (one of them [SPACE]), 0..15 mask and 0..15 sym rows of 1..4 columns over all 25 (repeats
    allowed), -1 only as trailing padding (build_combo_matrix layout)."""
    rng = np.random.default_rng(seed)

    def rows(n):
        return [[int(c) for c in rng.integers(0, oracle.NFEAT, size=int(rng.integers(1, 5)))] for _ in range(n)]

    def matrix(rs):
        if not rs:
            return NONE
        m = combo(rs)
        return np.concatenate([m, np.full((len(rs), int(rng.integers(0, 3))), -1, np.int8)], axis=1)

    split = rows(int(rng.integers(0, MAX_ROWS)))
    split.insert(int(rng.integers(0, len(split) + 1)), [SPACE])
    return (matrix(split), matrix(rows(int(rng.integers(0, MAX_ROWS + 1)))),
            matrix(rows(int(rng.integers(0, MAX_ROWS + 1)))))


FUZZ_SEEDS = range(1000, 1060)


def _fuzz_texts(seed):
    rng = np.random.default_rng(seed)
    texts = corpus.fuzz_strings(seed, 1500, 100, "mixed") + corpus.fuzz_strings(seed + 1, 500, 100, "marks")
    texts += [corpus.long_doc(rng, int(n), p) for n, p in ((9000, "ascii"), (20000, "marks"), (40000, "mixed"))]
    texts += ["x" * 9000 + "#", "a, " * 3000 + "b!"]
    return texts


@pytest.mark.parametrize("seed", FUZZ_SEEDS)
def test_rule_fuzz(engine, seed):
    rules = random_rules(seed)
    about = f"rule seed {seed}: split {rules[0].tolist()} mask {rules[1].tolist()} sym {rules[2].tolist()}"
    _check(engine, "fuzz", rules, _fuzz_texts(seed), 15, about)
    for t in corpus.fuzz_strings(seed + 2, 50, 80, "marks"):
        _check(engine, "fuzz", rules, [t], 7, f"{about}, one string {t!r}")


# ----------------------------------------------------------------------------------------------- consumers
def test_token_texts_and_vocabulary(engine):
    from latok_b200.core.default_tokenizer import tokenize_packed
    from latok_b200.engine import pack_strings
    from latok_b200.vocab import Vocab
    texts = corpus.FIXTURES + corpus.fuzz_strings(21, 3000, 120, "marks") + corpus.long_documents()[:6] + ["x a,b#", ""]
    for name in ("parity", "closer_marks", "max_counts"):
        rules = RULES[name]
        engine.set_rules(*rules)
        want = [oracle.tokens(t, rules) if t else [] for t in texts]
        pt = tokenize_packed(*pack_strings(texts), engine=engine)
        for i, t in enumerate(texts):
            assert pt.tokens(i) == want[i], f"{name}: string {i} {t[:40]!r}"
        v = Vocab(engine=engine)
        v.update(texts)
        want_counts = Counter(tok for toks in want for tok in toks)
        assert dict(zip(v.tokens(), v.counts().tolist())) == dict(want_counts), name
        v.close()
    engine.set_rules()


# ----------------------------------------------------------------------------------- rules in force at submit
def test_rules_in_force_at_submit(engine):
    """A batch is tokenized with the rules that were set when it was submitted, also when set_rules comes between
    its submit and its fetch, and when the fetch has to run it again with larger token buffers."""
    from latok_b200.engine import Engine, pack_strings
    A = corpus.FIXTURES + corpus.fuzz_strings(31, 2000, 100, "marks")
    C = corpus.fuzz_strings(32, 2000, 100, "mixed") + ["x a,b#"]
    R1, R2 = RULES["parity"], RULES["closer_marks"]
    # symbols only: one token per character under the default rules, more tokens than the buffers are sized for
    # at submit (the re-run at fetch); one token under `only_space`
    only_space = (combo([[SPACE]]), NONE, NONE)
    big = ["!?" * 40000, "a b " * 500]
    cases = [(engine, A, R1, C, R2), (engine, C, R2, A, None)]
    with Engine(0) as fresh:
        cases.append((fresh, big, None, C, only_space))
        for e, first, r_first, second, r_second in cases:
            e.set_pipeline_depth(2)
            e.set_rules(*(r_first or ()))
            e.submit(*pack_strings(first), 7)
            e.set_rules(*(r_second or ()))
            e.submit(*pack_strings(second), 7)
            for texts, rules in ((first, r_first), (second, r_second)):
                r = e.fetch()
                e.release()
                o = oracle.tokenize_batch(texts, rules=rules or oracle.DEFAULT_RULES)
                assert r.n_tokens == o["n_tokens"], (r.n_tokens, o["n_tokens"])
                for a in ("splits", "spans", "tok_offsets", "tok_feats"):
                    assert np.array_equal(getattr(r, a), o[a]), a
            e.set_pipeline_depth(1)
            e.set_rules()


# ----------------------------------------------------------------------------------------------- rejection
def test_rejected_rules_leave_the_engine_usable(engine):
    rules = RULES["parity"]
    engine.set_rules(*rules)
    bad = [
        (combo([[SPACE]] * (MAX_ROWS + 1)), C_MASK, C_SYM),           # 16 split rows
        (C_SPLIT, combo([[TWITTER]] * (MAX_ROWS + 1)), C_SYM),        # 16 mask rows
        (C_SPLIT, C_MASK, combo([[SYMBOL]] * (MAX_ROWS + 1))),        # 16 sym rows
        (C_SPLIT, combo([[TWITTER], [-1]]), C_SYM),                   # a row of only -1
        (combo([[SPACE], [-1, -1]]), C_MASK, C_SYM),
        (C_SPLIT, C_MASK, combo([[SYMBOL, 25]])),                     # column 25
        (combo([[SPACE], [oracle.NFEAT]]), C_MASK, C_SYM),
        (combo([[SYMBOL], [SPACE, NEXT_SPACE]]), C_MASK, C_SYM),      # no [SPACE] split row
    ]
    for b in bad:
        with pytest.raises(ValueError):
            engine.set_rules(*b)
        # the rules set before are still in force
        check_batch(engine, corpus.FIXTURES, 7, rules=rules, label=f"after rejecting {[m.tolist() for m in b]}")
    engine.set_rules()
    check_batch(engine, corpus.FIXTURES, 7, label="defaults after rejections")
