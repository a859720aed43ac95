"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol include/*.h
declares, argument validation works without a GPU (no compute calls), string packing, byte-balanced
sharding, and the world_size-2 token-count exchange over gloo."""
import ctypes as C
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

import corpus
from oracle import oracle

ROOT = Path(__file__).resolve().parent.parent


def header_functions():
    text = (ROOT / "include" / "latok_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"LATOK_B200_API\s+[\w\s\*]+?\b(latok_b200_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from latok_b200 import _lib
    L = _lib.load()
    names = header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/latok_b200.h but not exported"
    assert L.latok_b200_abi_version() == 2


def test_header_cites_the_reference_interface():
    text = (ROOT / "include" / "latok_b200.h").read_text()
    for cite in ("latok.c:373-378", "latok.c:31-138", "latok.c:140-258", "latok.c:275-370", "default_tokenizer.py:113-134"):
        assert cite in text


def test_no_gpu_means_loud_failure_not_fallback():
    from latok_b200 import _lib
    if _lib.device_count() > 0:
        pytest.skip("a GPU is present")
    from latok_b200.engine import Engine
    with pytest.raises(_lib.LatokCudaError, match="no CPU fallback"):
        Engine(0)
    from latok_b200.core.default_tokenizer import tokenize
    with pytest.raises(_lib.LatokCudaError):
        list(tokenize("no gpu here"))


def test_argument_validation_without_gpu():
    from latok_b200 import _lib
    L = _lib.load()
    h = C.c_void_p()
    assert L.latok_b200_create(0, 0, -1, C.byref(h)) == _lib.EINVAL
    assert L.latok_b200_submit(None, None, None, 0, 3) == _lib.EINVAL
    assert b"engine is NULL" in L.latok_b200_last_error()
    assert L.latok_b200_fetch(None, 0, 0, 0, None, None, None, None, None, None) == _lib.EINVAL
    assert L.latok_b200_set_pipeline_depth(None, 2) == _lib.EINVAL and L.latok_b200_release(None) == _lib.EINVAL
    assert L.latok_b200_destroy(None) == _lib.OK


def test_product_never_imports_the_oracle():
    for path in (ROOT / "latok_b200").rglob("*"):
        if path.suffix in (".py", ".cu", ".h", ".cuh") and "_gen" not in path.parts:
            assert not re.search(r"import\s+oracle|from\s+oracle|from\s+\.+oracle|liblatok_oracle|oracle[/.](oracle|ref_driver|_ref|_build)",
                                 path.read_text()), f"{path} reaches into oracle/"


def test_pack_strings_roundtrip():
    from latok_b200.engine import pack_strings
    texts = corpus.FIXTURES + ["", "x", ""] + corpus.fuzz_strings(3, 200, 40)
    buf, off = pack_strings(texts)
    assert off[0] == 0 and off[-1] == len(buf) and np.all(np.diff(off) >= 0)
    raw = buf.tobytes()
    assert [raw[off[i]:off[i + 1]].decode("utf-8", "surrogatepass") for i in range(len(texts))] == texts


def test_c_packer_matches_python_encode():
    """pack_strings runs in C (csrc/latok_pypack.c): same bytes and offsets as str.encode('utf-8', 'surrogatepass')
    for every PEP-393 kind (ASCII, Latin-1, UCS-2, UCS-4), lone surrogates, empty strings, tuples and generators,
    into a caller's buffer, and with a buffer that is too small."""
    from latok_b200.engine import pack_strings, pack_strings_python
    texts = corpus.FIXTURES + ["", "\xe9\xff latin1", "\u20ac ucs2 \ud800", "\U0001F600 ucs4 \udfff", "\x00nul\x7f", ""] \
        + corpus.fuzz_strings(8, 3000, 120, "mixed") + ["".join(map(chr, range(0x7F0, 0x810))), "".join(map(chr, range(0xFFF0, 0x10010)))]
    want = pack_strings_python(texts)
    for form in (texts, tuple(texts), (t for t in texts)):
        got = pack_strings(form)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[1].dtype == np.int64
    big = np.zeros(len(want[0]) + 100, dtype=np.uint8)
    got = pack_strings(texts, big)
    assert got[0].base is big and np.array_equal(got[0], want[0])
    small = np.zeros(10, dtype=np.uint8)
    got = pack_strings(texts, small)                               # does not fit: a fresh buffer of the exact size
    assert np.array_equal(got[0], want[0]) and not small.any() or np.array_equal(got[0], want[0])
    assert pack_strings([])[1].tolist() == [0] and len(pack_strings([])[0]) == 0
    with pytest.raises(TypeError):
        pack_strings(["ok", b"bytes are not str"])


def test_c_token_slicing_matches_the_reference_loop():
    """_pack.slice_tokens (the C loop behind tokenize_batch) = the reference's `text[s:e].strip()`, dropped when empty
    (default_tokenizer.py:151-158), on the oracle's spans, for int32 and uint16 span arrays."""
    from latok_b200 import _pack
    from oracle import oracle
    texts = [t for t in corpus.FIXTURES + corpus.fuzz_strings(2, 1500, 100, "mixed") if t]
    o = oracle.tokenize_batch(texts, feats=False)
    want = [[tok for tok in (t[s:e].strip() for s, e in o["spans"][o["tok_offsets"][i]:o["tok_offsets"][i + 1]]) if tok]
            for i, t in enumerate(texts)]
    assert want == [oracle.tokens(t) for t in texts]
    assert _pack.slice_tokens(texts, o["spans"], o["tok_offsets"]) == want
    assert _pack.slice_tokens(texts, o["spans"].astype(np.uint16), o["tok_offsets"]) == want
    bad = o["spans"].copy(); bad[0, 1] = 10 ** 6
    with pytest.raises(ValueError):
        _pack.slice_tokens(texts, bad, o["tok_offsets"])


def test_mirror_modules_match_reference_constants():
    from latok_b200.core import offsets as oft
    from latok_b200.core.latok_utils import FEATURE_NAMES, NUM_FEATURES, build_combo_matrix
    assert oft.FEATURE_COUNT == NUM_FEATURES == 25 and oft.SPACE_IDX == 5 and oft.AFTER_NEXT_SLASH_IDX == 24
    assert oft.CHAR_PERIOD_MASK == 0x80000 and oft.SPECIALS_MASK == 0x8000
    assert FEATURE_NAMES[0] == "Alpha" and FEATURE_NAMES[24] == "After_Next_/" and FEATURE_NAMES[8] == "@"
    m = build_combo_matrix([[1], [2, 3, 4], [5, 6]])
    assert m.dtype == np.int8 and m.tolist() == [[1, -1, -1], [2, 3, 4], [5, 6, -1]]
    assert np.array_equal(m, oracle.combo([[1], [2, 3, 4], [5, 6]]))


def test_synthetic_corpora_are_valid_and_seeded():
    import synth
    for fn, kw in ((synth.tweets, dict(n_strings=3000)), (synth.mixed_unicode, dict(n_strings=2000)),
                   (synth.long_docs, dict(n_docs=6, doc_bytes=20000))):
        b1, o1 = fn(**kw)
        b2, o2 = fn(**kw)
        assert np.array_equal(b1, b2) and np.array_equal(o1, o2)
        assert o1[0] == 0 and o1[-1] == len(b1) and np.all(np.diff(o1) > 0)
        b1.tobytes().decode("utf-8")   # well-formed
    b, o = synth.tweets(3000)
    lens = [len(s) for s in synth.to_strings(b, o)]
    assert 100 < np.mean(lens) < 190


def oracle_run(device, buf, offsets, what):
    """Stand-in for an Engine on a box without GPUs: the oracle packaged as a BatchResult (test only)."""
    from latok_b200.engine import BatchResult
    o = oracle.tokenize_batch_utf8(buf, offsets, feats=bool(what & 4), matrix=bool(what & 8))
    r = BatchResult(len(offsets) - 1, o["n_chars"], o["n_tokens"], splits=o["splits"], char_offsets=o["char_offsets"],
                    spans=o["spans"], tok_offsets=o["tok_offsets"], tok_feats=o.get("tok_feats"), matrix=o.get("matrix"))
    return r


def test_shard_ranges_and_merge():
    from latok_b200 import sharding
    import synth
    buf, off = synth.tweets(5000, seed=7)
    for g in (1, 2, 3, 4, 8):
        rng = sharding.shard_ranges(off, g)
        assert rng[0][0] == 0 and rng[-1][1] == len(off) - 1
        assert all(a[1] == b[0] for a, b in zip(rng, rng[1:]))
        sizes = [int(off[b] - off[a]) for a, b in rng]
        assert max(sizes) - min(sizes) <= 2 * int(np.diff(off).max())      # byte balanced to within a string
        merged = sharding.tokenize_sharded(buf, off, list(range(g)), what=1 | 2 | 4, run_fn=oracle_run)
        whole = oracle_run(0, buf, off, 1 | 2 | 4)
        for name in ("splits", "char_offsets", "spans", "tok_offsets", "tok_feats"):
            assert np.array_equal(getattr(merged, name), getattr(whole, name)), (g, name)
    # more shards than strings, empty strings, empty batch
    tiny_b, tiny_o = np.frombuffer(b"ab cd", dtype=np.uint8), np.array([0, 2, 2, 5], dtype=np.int64)
    m = sharding.tokenize_sharded(tiny_b, tiny_o, [0, 1, 2, 3, 4], run_fn=oracle_run)
    w = oracle_run(0, tiny_b, tiny_o, 3)
    assert np.array_equal(m.spans, w.spans) and np.array_equal(m.tok_offsets, w.tok_offsets)
    assert sharding.shard_ranges(np.array([0], dtype=np.int64), 4) == [(0, 0)] * 4


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
    from latok_b200 import sharding
    import synth
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    buf, off = synth.tweets(2000, seed=11)
    s0, s1 = sharding.shard_ranges(off, world)[rank]
    b, o = sharding.slice_shard(buf, off, s0, s1)
    r = oracle_run(rank, np.ascontiguousarray(b), np.ascontiguousarray(o), 3)
    counts, cbase, tbase = sharding.allgather_counts(r.n_chars, r.n_tokens)
    r = sharding.rebase_for_rank(r, cbase, tbase)
    q.put((rank, s0, s1, counts.tolist(), r.char_offsets.tolist(), r.tok_offsets.tolist(), r.spans.tolist()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_count_exchange_over_gloo():
    import torch.multiprocessing as mp
    import synth
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    buf, off = synth.tweets(2000, seed=11)
    whole = oracle_run(0, buf, off, 3)
    (r0, a0, b0, counts0, co0, to0, sp0), (r1, a1, b1, counts1, co1, to1, sp1) = got
    assert counts0 == counts1 and a0 == 0 and b0 == a1 and b1 == 2000
    assert co0[:-1] + co1 == whole.char_offsets.tolist()
    assert to0[:-1] + to1 == whole.tok_offsets.tolist()
    assert sp0 + sp1 == whole.spans.tolist()


def test_bit_plane_primitives_selftest(tmp_path):
    """latok_bits.h (byte->plane transpose, bit-sliced ASCII classifier, squeeze, carry-add block mask, flood) is
    host-compilable: tools/bits_selftest.cpp checks it against the generated class table and scalar loops."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    root = Path(__file__).resolve().parent.parent
    exe = tmp_path / "bits_selftest"
    subprocess.run([gxx, "-O1", "-std=c++17", "-w", "-I", str(root / "latok_b200" / "csrc"),
                    str(root / "tools" / "bits_selftest.cpp"), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "bits selftest ok" in out.stdout


def test_timing_cli_tsv_assembly():
    """tools/time_tokenizer.py builds the --outfile rows ('\\t'.join(tokens) per input row,
    scripts/timing/time_tokenizer.py:105-107) from token byte ranges with NumPy gathers only."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
    from time_tokenizer import pack, tsv_bytes
    rows = [["ab", "cd"], [], [], ["e"], ["日本", "x"], []]
    texts = [" ".join(r) for r in rows]
    buf, off = pack([t.encode() for t in texts])
    spans, toff = [], [0]
    for t, o in zip(texts, off[:-1]):
        b = t.encode()
        p = 0
        for tok in t.split():
            p = b.index(tok.encode(), p)
            spans.append((o + p, o + p + len(tok.encode())))
            p += len(tok.encode())
        toff.append(len(spans))
    got = tsv_bytes(buf, np.array(spans, dtype=np.int64).reshape(-1, 2), np.array(toff, dtype=np.int64))
    assert got == "".join("\t".join(r) + "\n" for r in rows).encode()
    assert tsv_bytes(buf[:0], np.zeros((0, 2), np.int64), np.array([0, 0, 0], np.int64)) == b"\n\n"


def test_table_regeneration_rules_reproduce_ucd11():
    """tools/regen_classes.py applies the reference's flag rules (makeunicodedata.py:158-200,249-258) to the UCD of
    the running Python.  Wherever UCD 11 gave a code point features, the rules must give the same ones (a handful of
    code points changed properties in later UCD versions); the rest of the difference is newly assigned code points.
    The ranges file it writes reads back to the same classes."""
    import subprocess
    import sys
    import tempfile
    root = Path(__file__).resolve().parent.parent
    sys.path.insert(0, str(root / "tools"))
    import regen_classes as rc
    old = rc.read_ranges(rc.UCD11)
    feat = [rc.base_features(cp) for cp in range(0x110000)]
    assert feat[:128] == old[:128]
    redefined = [cp for cp in range(0x110000) if old[cp] != 0 and feat[cp] != old[cp]]
    assert len(redefined) <= 8, [hex(c) for c in redefined[:20]]
    assert len(set(feat)) <= 17
    spaces = [cp for cp in range(0x110000) if feat[cp] & 0x20]
    assert spaces == [cp for cp in range(0x110000) if chr(cp).isspace()]          # SURVEY Q9
    with tempfile.TemporaryDirectory() as d:
        out = Path(d) / "ucd_new.txt"
        subprocess.run([sys.executable, str(root / "tools" / "regen_classes.py"), "--out", str(out)], check=True)
        assert rc.read_ranges(out) == feat


def load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_config5_batch_shards_cover_the_batch():
    """bench.py --workload chars1b: every rank builds the same batch and keeps its byte-balanced range of whole
    strings; the ranges tile the batch and are balanced to within one string."""
    bench = load_bench()
    from latok_b200.sharding import shard_ranges, slice_shard
    buf, off = bench.make_batch("chars1b", 6000, 0)
    buf2, off2 = bench.make_batch("chars1b", 6000, 0)
    assert np.array_equal(buf, buf2) and np.array_equal(off, off2)            # same on every rank
    assert off[0] == 0 and off[-1] == len(buf) and np.all(np.diff(off) > 0) and len(off) == 6001
    for world in (1, 2, 4, 8):
        ranges = shard_ranges(off, world)
        assert ranges[0][0] == 0 and ranges[-1][1] == 6000
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        parts = [slice_shard(buf, off, s0, s1) for s0, s1 in ranges]
        assert np.array_equal(np.concatenate([p[0] for p in parts]), buf)
        sizes = [len(p[0]) for p in parts]
        assert max(sizes) - min(sizes) <= 2 * int(np.diff(off).max())


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: every array of the result as float32 / float64 .npy with exact values, the ones over
    the per-array budget as the same seeded, ordered sample of rows on every call, under 64 MB in all."""
    bench = load_bench()
    from latok_b200.engine import BatchResult
    S, C_, T = 1000, 4_000_000, 1_000_000
    rng = np.random.default_rng(1)
    r = BatchResult(S, C_, T, splits=rng.integers(0, 3, C_).astype(np.int8),
                    char_offsets=np.linspace(0, C_, S + 1).astype(np.int64) + (1 << 40),
                    spans=np.stack([np.arange(T), 3 * np.arange(T)], axis=1).astype(np.int32),
                    tok_offsets=np.linspace(0, T, S + 1).astype(np.int64),
                    tok_feats=rng.integers(-128, 128, (T, 25)).astype(np.int8))
    for d in ("a", "b"):
        bench.dump_outputs(r, tmp_path / d)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(f"{n}.npy" for n in bench.DUMP_ARRAYS)
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) < 64 << 20
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert got["splits"].dtype == got["tok_feats"].dtype == np.float32
    assert got["spans"].dtype == got["char_offsets"].dtype == got["tok_offsets"].dtype == np.float64
    assert np.array_equal(got["char_offsets"], r.char_offsets) and np.array_equal(got["tok_offsets"], r.tok_offsets)
    rows = got["spans"][:, 0].astype(np.int64)                 # spans row i is (i, 3 i): the sample's row numbers
    assert 0 < len(rows) < T and np.all(np.diff(rows) > 0) and np.array_equal(got["spans"][:, 1], 3 * rows)
    assert 0 < len(got["splits"]) < C_ and set(np.unique(got["splits"])) <= {0.0, 1.0, 2.0}
    n = len(got["tok_feats"])
    assert 0 < n < T and got["tok_feats"].shape[1] == 25
    pick = np.sort(np.random.default_rng(0).choice(T, n, replace=False))
    assert np.array_equal(got["tok_feats"], r.tok_feats[pick])


def test_native_csv_reader_matches_python_csv_json(tmp_path):
    """latok_b200_reader_* (host code, no GPU): the packed batches equal `json.loads(row[1]).strip()` per csv row
    (scripts/timing/time_tokenizer.py:25-40) -- quoting, escapes, surrogate pairs, every whitespace character at both
    ends, gzip, rows that do not fit the buffer, and the reference's failure cases."""
    import csv
    import gzip
    import json
    from latok_b200.reader import CsvReader
    spaces = "".join(chr(c) for c in range(0x110000) if chr(c).isspace())
    texts = list(corpus.FIXTURES) + corpus.fuzz_strings(41, 400, 150, "mixed")
    texts += [spaces + "x" + spaces, spaces, "", 'a "quoted", value', "comma,inside", "tab\tinside and \\ backslash",
              "\U0001F600 astral \ud83d lone", "line\nbreak\r\nin text", "\x00nul\x1f"]
    for name, ensure_ascii, opener in (("a.csv", True, open), ("b.csv.gz", False, gzip.open)):
        path = tmp_path / name
        with opener(path, "wt", encoding="utf-8", errors="surrogatepass", newline="") as f:
            w = csv.writer(f)
            for i, t in enumerate(texts):
                w.writerow([i, json.dumps(t, ensure_ascii=ensure_ascii), "third, column"])
        # (json.loads, not the original text: it joins an escaped high + low surrogate pair into one code point)
        want = [json.loads(json.dumps(t, ensure_ascii=ensure_ascii)).strip().encode("utf-8", "surrogatepass") for t in texts]
        for rows, nbytes in ((1000, 1 << 20), (7, 1 << 20), (1000, 700)):
            got = []
            with CsvReader(str(path), batch_rows=rows, batch_bytes=nbytes) as r:
                for buf, off in r:
                    assert off[0] == 0 and off[-1] == len(buf)
                    got += [bytes(buf[off[i]:off[i + 1]]) for i in range(len(off) - 1)]
            assert got == want, (name, rows, nbytes)
    # failure cases of the reference's loop: no column 1 (IndexError there), not a JSON string (AttributeError there)
    for content in ("0\n", '0,"123"\n', '0,"{""a"": 1}"\n', '0,"""unterminated"\n'):
        bad = tmp_path / "bad.csv"
        bad.write_text(content)
        with pytest.raises(ValueError):
            with CsvReader(str(bad)) as r:
                list(r)
    with pytest.raises(ValueError):
        CsvReader(str(tmp_path / "missing.csv"))


def _packed_table_lookup(header_text):
    """Emulates the kernels' class look-up (latok_device.cuh: class_of_cp / mb_features) on the arrays of a generated
    latok_tables.h; returns a function code point -> 12-bit feature word."""
    def arr(name):
        body = re.search(r"%s\[\d+\] = \{(.*?)\};" % name, header_text, re.S).group(1)
        return [int(x, 0) for x in body.replace("\n", " ").split(",") if x.strip()]
    low_limit = int(re.search(r"#define LATOK_TBL_LOW_LIMIT (0x[0-9A-Fa-f]+)u", header_text).group(1), 16)
    ascii_feat, stage1, stage2, class_feat = arr("LATOK_ASCII_FEAT"), arr("LATOK_STAGE1"), arr("LATOK_STAGE2"), arr("LATOK_CLASS_FEAT")
    high = [tuple(int(v, 16) for v in m) for m in re.findall(r"\{0x([0-9A-F]+)u, 0x([0-9A-F]+)u, 0x([0-9A-F]+)u\}", header_text)]
    assert len(high) == 1

    def look(cp):
        if cp < 0x80:
            return ascii_feat[cp]
        if cp < low_limit:
            b = stage2[stage1[cp >> 7] * 64 + ((cp & 127) >> 1)]
            return class_feat[(b >> 4) if cp & 1 else (b & 15)]
        return high[0][2] if high[0][0] <= cp <= high[0][1] else 0
    return look, max(stage1)


def test_packed_class_tables_cover_every_code_point():
    """The packed two-stage table the kernels read (tools/gen_tables.py) against the class ranges it was built from,
    for every code point: the UCD-11 table of the build, and a table generated for the UCD of the running Python
    (tools/regen_classes.py; needs 16-bit stage-1 entries, which the kernels take from latok_table_types.h)."""
    import subprocess
    import sys
    import tempfile
    root = Path(__file__).resolve().parent.parent
    sys.path.insert(0, str(root / "tools"))
    import regen_classes as rc
    gen = root / "latok_b200" / "csrc" / "_gen"
    look, top = _packed_table_lookup((gen / "latok_tables.h").read_text())
    want = rc.read_ranges(rc.UCD11)
    assert all(look(cp) == want[cp] for cp in range(0x110000))
    assert top < 256 and "typedef uint8_t latok_stage1_t" in (gen / "latok_table_types.h").read_text()
    with tempfile.TemporaryDirectory() as d:
        out = Path(d) / "ucd_new.txt"
        subprocess.run([sys.executable, str(root / "tools" / "regen_classes.py"), "--out", str(out)], check=True)
        env = dict(os.environ, LATOK_CLASSES=str(out), LATOK_LOW_LIMIT="0x32400")
        subprocess.run([sys.executable, str(root / "tools" / "gen_tables.py"), d], check=True, env=env, stdout=subprocess.DEVNULL)
        look, top = _packed_table_lookup((Path(d) / "latok_tables.h").read_text())
        want = rc.read_ranges(out)
        assert all(look(cp) == want[cp] for cp in range(0x110000))
        assert ("typedef uint16_t latok_stage1_t" in (Path(d) / "latok_table_types.h").read_text()) == (top >= 256)
