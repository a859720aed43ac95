"""Merging token vocabularies and counting / encoding one batch sharded over several devices (Vocab.merge,
latok_b200.sharding.encode_sharded / update_sharded) against plain Python over the oracle's tokens and against one
vocabulary fed the whole batch on one GPU.  A device may appear more than once in `devices`, so one GPU runs the same
merge path as eight; the cross-device copies need two GPUs.  Needs a B200 (-m gpu)."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import corpus
from test_gpu_vocab import expected, golden_texts, hard_keys

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def engine():
    from latok_b200.engine import Engine
    from latok_b200.sharding import close_engines
    with Engine(0) as e:
        yield e
    close_engines()


def state(v):
    return v.tokens(), v.counts().tolist()


def check_merge(engine_a, engine_b, a_batches, b_batches):
    """a.merge(b) for a fed a_batches and b fed b_batches: the vocabulary of a_batches + b_batches on one GPU, and the
    map gives every key of b its position in the result; the device map equals the host map."""
    from latok_b200.vocab import Vocab
    a, a2, b = Vocab(engine_a), Vocab(engine_a), Vocab(engine_b)
    for t in a_batches:
        a.update(t)
        a2.update(t)
    for t in b_batches:
        b.update(t)
    before_b = state(b)
    m = a.merge(b)
    md = a2.merge(b, device=True)
    _, want_cnt, want_keys = expected(list(a_batches) + list(b_batches))
    assert a.tokens() == want_keys
    assert a.counts().tolist() == [want_cnt[k] for k in want_keys]
    pos = {k: i for i, k in enumerate(want_keys)}
    assert m.dtype == np.int32 and m.tolist() == [pos[k] for k in before_b[0]]
    assert md.is_cuda and md.device.index == engine_a.device and np.array_equal(md.cpu().numpy(), m)
    assert state(a2) == state(a)
    assert state(b) == before_b                                     # the source is unchanged


def test_merge_fixtures_golden_fuzz_hard_keys(engine):
    fuzz = corpus.fuzz_strings(141, 3000, 200, "mixed") + corpus.fuzz_strings(142, 2000, 120, "ascii")
    cases = [
        ([corpus.FIXTURES], [golden_texts()]),
        ([golden_texts(), fuzz[:800]], [fuzz[500:2000], corpus.FIXTURES]),
        ([fuzz[:2500]], [fuzz[2500:]]),
        ([fuzz[:1000]], [fuzz[:1000]]),                             # every key known: counts only
        ([hard_keys()[:5]], [hard_keys(), hard_keys()[::-1]]),
        ([fuzz[:300]], [hard_keys()]),
        ([], [fuzz[:700]]),                                          # empty destination
        ([fuzz[:700]], []),                                          # empty source
        ([], []),
        ([["", "   "]], [[" \t "]]),
    ]
    for a_batches, b_batches in cases:
        check_merge(engine, engine, a_batches, b_batches)


def test_merge_grows_from_capacity_16(engine):
    from latok_b200.vocab import Vocab
    words = [f"w{i:x}" for i in range(100_000)]
    src_texts = [" ".join(words[i:i + 50]) for i in range(0, len(words), 50)]
    dst_texts = ["w5 zz w3 yy", "w1869f w5"]
    dst = Vocab(engine, capacity=16)
    dst.update(dst_texts)
    slots = dst.table_slots()
    src = Vocab(engine)
    src.update(src_texts)
    src.update(src_texts[::3])
    m = dst.merge(src)
    _, cnt, keys = expected([dst_texts, src_texts, src_texts[::3]])
    assert len(dst) == len(keys) == 100_002 and dst.table_slots() > slots
    assert dst.tokens() == keys and dst.counts().tolist() == [cnt[k] for k in keys]
    pos = {k: i for i, k in enumerate(keys)}
    assert m.tolist() == [pos[k] for k in src.tokens()]


def test_merge_errors_and_clear(engine):
    from latok_b200.engine import pack_strings
    from latok_b200.sharding import encode_sharded
    from latok_b200.vocab import Vocab
    v = Vocab(engine)
    v.update(["a b c", "b"])
    f = Vocab.from_tokens(["x", "y"], engine=engine)
    with pytest.raises(RuntimeError, match="frozen"):
        f.merge(v)
    with pytest.raises(ValueError, match="itself"):
        v.merge(v)
    with pytest.raises(RuntimeError, match="frozen"):
        f.clear()
    with pytest.raises(RuntimeError, match="frozen"):
        encode_sharded(f, *pack_strings(["x y"]), [0])
    assert state(v) == (["a", "b", "c"], [1, 2, 1]) and state(f) == (["x", "y"], [0, 0])
    # a cleared vocabulary behaves like a fresh one, also when it had more keys than the new batches bring
    v.update(corpus.fuzz_strings(151, 2000, 150, "mixed"))
    v.clear()
    assert len(v) == 0 and v.tokens() == [] and v.counts().tolist() == []
    batches = [corpus.fuzz_strings(152, 500, 150, "mixed"), corpus.FIXTURES]
    fresh = Vocab(engine)
    for t in batches:
        assert np.array_equal(v.encode(t)[0], fresh.encode(t)[0])
    assert state(v) == state(fresh)
    v.clear()
    v.merge(fresh)
    assert state(v) == state(fresh)


def batch_list():
    fuzz = corpus.fuzz_strings(161, 2400, 180, "mixed")
    return [fuzz[:900], corpus.FIXTURES + golden_texts(), [], hard_keys() + fuzz[900:1200], ["", "  "], fuzz[1200:]]


def check_sharded(engine, devices, batches, prefix):
    """encode_sharded / update_sharded over `devices`, batch after batch into a vocabulary that already holds the keys
    of `prefix`, against encode_packed / update of the same batches on one GPU; then add=False with an unk, against a
    frozen vocabulary and against a non-frozen one that changes between calls (its replicas are rebuilt)."""
    from latok_b200.engine import pack_strings
    from latok_b200.sharding import encode_sharded, update_sharded
    from latok_b200.vocab import Vocab
    ref, v = Vocab(engine), Vocab(engine)
    ref.update(prefix)
    v.update(prefix)
    for i, texts in enumerate(batches):
        buf, off = pack_strings(texts)
        if i % 3 == 2:
            ref.update(texts)
            assert update_sharded(v, buf, off, devices) is None
        else:
            want_ids, want_off = ref.encode_packed(buf, off)
            ids, tok_off = encode_sharded(v, buf, off, devices)
            assert ids.dtype == np.int32 and tok_off.dtype == np.int64
            assert np.array_equal(ids, want_ids) and np.array_equal(tok_off, want_off)
        assert state(v) == state(ref)
    keys = ref.tokens()
    frozen = Vocab.from_tokens(keys[::2], engine=engine)
    probe = [t for b in batches for t in b][::2] + ["tokens none of the batches had", ""]
    buf, off = pack_strings(probe)
    want_ids, want_off = frozen.encode_packed(buf, off, add=False, unk=-5)
    assert (want_ids == -5).any()
    ids, tok_off = encode_sharded(frozen, buf, off, devices, add=False, unk=-5)
    assert np.array_equal(ids, want_ids) and np.array_equal(tok_off, want_off)
    for extra in (None, ["tokens none of the batches had"], probe[:50]):
        if extra is not None:
            v.update(extra)
        want_ids, _ = v.encode_packed(buf, off, add=False, unk=-3)
        ids, tok_off = encode_sharded(v, buf, off, devices, add=False, unk=-3)
        assert np.array_equal(ids, want_ids) and np.array_equal(tok_off, want_off)
    assert (ids[tok_off[-3]:tok_off[-2]] >= 0).all()     # the keys added by the update are found
    return v


@pytest.mark.parametrize("devices", [[0], [0, 0], [0, 0, 0, 0, 0]])
def test_sharded_one_device(engine, devices):
    check_sharded(engine, devices, batch_list(), corpus.fuzz_strings(171, 300, 120, "mixed"))


def test_sharded_more_shards_than_strings(engine):
    check_sharded(engine, [0] * 7, [["one two", "two three four"], ["x"], [], ["a b", "b c", "c d"]], ["two b"])


def test_sharded_config2_200k_tweets(engine):
    import synth
    from latok_b200.sharding import encode_sharded
    from latok_b200.vocab import Vocab
    buf, off = synth.tweets(200_000, 20240601)
    ref, v = Vocab(engine), Vocab(engine)
    want_ids, want_off = ref.encode_packed(buf, off)
    ids, tok_off = encode_sharded(v, buf, off, [0, 0, 0, 0])
    assert np.array_equal(ids, want_ids) and np.array_equal(tok_off, want_off)
    assert state(v) == state(ref)


def test_sharded_all_devices():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU: the cross-device copies of a merge need two")
    from latok_b200.engine import Engine
    with Engine(0) as e0, Engine(n - 1) as e1:
        check_merge(e0, e1, [corpus.FIXTURES], [golden_texts(), hard_keys()])
        check_merge(e1, e0, [golden_texts()], [corpus.fuzz_strings(181, 1000, 150, "mixed"), hard_keys()])
        devices = list(range(n))
        v = check_sharded(e0, devices, batch_list(), corpus.fuzz_strings(182, 300, 120, "mixed"))
        assert set(v._replicas) == set(devices[1:])
        assert all(ver == v.version for ver, _ in v._replicas.values())
        check_sharded(e1, devices[::-1] + [0, 0], batch_list()[:4], [])


def test_forced_collisions_three_hash_bits():
    """Every key hashes to one of 7 values: merges and sharded encodes stay exact."""
    code = f"""
import sys
sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'tests')!r}]
import corpus
from test_gpu_vocab import hard_keys, golden_texts
from test_gpu_vocab_shard import check_merge, check_sharded
from latok_b200.engine import Engine
from latok_b200.sharding import close_engines
with Engine(0) as e:
    fuzz = corpus.fuzz_strings(191, 400, 80, "mixed")
    check_merge(e, e, [fuzz[:200], corpus.FIXTURES], [hard_keys(), fuzz[100:], golden_texts()[:40]])
    check_sharded(e, [0, 0, 0], [fuzz[:150], hard_keys(), fuzz[150:], golden_texts()[:40]], corpus.FIXTURES)
    close_engines()
print("ok")
"""
    env = dict(os.environ, LATOK_B200_VOCAB_HASH_BITS="3")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(ROOT))
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-3000:]
