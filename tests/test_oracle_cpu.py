"""Pins the CPU oracle (oracle/latok_oracle.c) to the reference:
  * the reference's one stored golden vector (executed notebook cell),
  * committed outputs of the compiled reference on the fixture corpus (tests/golden),
  * sha256 digests of the compiled reference over 12 300 fuzz strings,
  * and every code point's class as read off the compiled reference.
No GPU needed."""
import hashlib
import json
import zlib

import numpy as np

import corpus
from oracle import oracle


def words_to_matrix(words):
    w = np.asarray(words, dtype=np.int64)[:, None]
    return ((w >> np.arange(25)) & 1).astype(np.int8)


def test_notebook_cell(golden_dir):
    cell = json.load(open(golden_dir / "notebook_cell.json"))
    m = oracle.parse_matrix(cell["text"])
    assert m.tolist() == cell["matrix"]
    assert oracle.split_mask(m).tolist() == cell["splits"]
    # SURVEY.md section 4 quotes the same vector
    assert cell["splits"] == [1, 0, 0, 0, 1, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0, 1, 2, 1, 0, 0, 0, 0, 0, 0, 2, 2, 1,
                              0, 0, 0, 0, 0, 0, 2, 2, 0, 1, 0, 1, 0]


def test_fixture_outputs(golden_dir):
    recs = json.load(open(golden_dir / "reference_outputs.json"))["records"]
    assert [r["text"] for r in recs] == corpus.FIXTURES
    for r in recs:
        t = r["text"]
        m = oracle.parse_matrix(t)
        assert np.array_equal(m, words_to_matrix(r["matrix_words"])), t
        s = oracle.split_mask(m)
        assert s.tolist() == r["splits"], t
        assert oracle.tokens(t) == r["tokens"], t
        if "feats" in r:
            sp, tr = oracle.spans(s, m)
            assert sp.tolist() == r["feat_spans"], t
            assert [t[a:b] for a, b in tr] == r["feat_texts"], t
            assert oracle.token_feats(m, sp).tolist() == r["feats"], t


def test_fuzz_digests(golden_dir):
    sets = json.load(open(golden_dir / "fuzz_digest.json"))["sets"]
    for d in sets:
        strings = corpus.fuzz_strings(d["seed"], d["count"], d["max_len"], d["profile"])
        h_m, h_s, h_t, n_tok = hashlib.sha256(), hashlib.sha256(), hashlib.sha256(), 0
        for t in strings:
            if not t:
                continue
            m = oracle.parse_matrix(t)
            s = oracle.split_mask(m)
            toks = oracle.tokens(t)
            h_m.update(m.tobytes())
            h_s.update(s.tobytes())
            h_t.update(("\x00".join(toks) + "\x01").encode("utf-8", "surrogatepass"))
            n_tok += len(toks)
        assert (h_m.hexdigest(), h_s.hexdigest(), h_t.hexdigest(), n_tok) == \
               (d["matrix"], d["splits"], d["tokens"], d["n_tokens"]), d["profile"]


def test_every_codepoint_class(golden_dir):
    want = np.frombuffer(zlib.decompress((golden_dir / "codepoint_classes.bin").read_bytes()), dtype=np.uint16)
    assert len(want) == 0x110000
    got = np.fromiter((oracle.base_features(cp) for cp in range(0x110000)), dtype=np.uint16, count=0x110000)
    assert np.array_equal(got, want)
    assert oracle.base_features(0x110000) == 0 and oracle.base_features(0xFFFFFFFF) == 0


def test_space_class_is_python_isspace():
    # A5 relies on text[s:e].strip() == trimming SPACE-class characters (SURVEY.md Q9)
    space = [cp for cp in range(0x110000) if oracle.base_features(cp) & (1 << oracle.SPACE)]
    assert space == [cp for cp in range(0x110000) if chr(cp).isspace()]
    assert len(space) == 29


def test_batch_driver_matches_per_string():
    texts = corpus.FIXTURES + ["", "", "tail"] + corpus.fuzz_strings(7, 200, 80)
    out = oracle.tokenize_batch(texts, matrix=True, feats=True)
    c = t = 0
    for i, s in enumerate(texts):
        assert out["char_offsets"][i] == c and out["tok_offsets"][i] == t
        if s:
            m = oracle.parse_matrix(s)
            sm = oracle.split_mask(m)
            sp, _ = oracle.spans(sm, m)
            n = len(m)
            assert np.array_equal(out["matrix"][c:c + n], m)
            assert np.array_equal(out["splits"][c:c + n], sm)
            assert np.array_equal(out["spans"][t:t + len(sp)], sp)
            assert np.array_equal(out["tok_feats"][t:t + len(sp)], oracle.token_feats(m, sp))
            c += n
            t += len(sp)
    assert out["n_chars"] == c and out["n_tokens"] == t


def test_utf8_front_end():
    texts = corpus.FIXTURES + corpus.fuzz_strings(11, 300, 50)
    enc = [s.encode("utf-8", "surrogatepass") for s in texts]
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(e) for e in enc])
    buf = np.frombuffer(b"".join(enc), dtype=np.uint8)
    cps, char_off = oracle.decode_utf8(buf, off)
    want = np.concatenate([oracle.codepoints(s) for s in texts])
    assert np.array_equal(cps, want)
    assert char_off[-1] == len(want)


def test_block_mask_scan_form():
    """The closed form the CUDA kernel uses (backlog x: +1 per mark, max(x-1,0) per space) agrees with
    the sequential merge of latok.c:218-244, including the no-space / no-mark cases."""
    rng = np.random.default_rng(5)
    for _ in range(3000):
        n = int(rng.integers(1, 40))
        a1 = (rng.random(n) < rng.choice([0.05, 0.2, 0.5])).astype(np.int8)
        a2 = (rng.random(n) < rng.choice([0.0, 0.1, 0.3])).astype(np.int8)
        want = oracle.block_mask(a1, a2)
        got = np.ones(n, dtype=np.int8)
        if a1.any() and not a2.any():
            got[:] = 0
        else:
            x, start = 0, 1
            for i in range(n + 1):
                if i < n and a1[i]:
                    x += 1
                if i == n or a2[i]:
                    if x >= 1 and (i < n or True):
                        got[start:i] = 0
                    x = max(x - 1, 0)
                    start = i + 1
        assert np.array_equal(got, want), (a1, a2, got, want)

