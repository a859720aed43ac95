"""Multi-GPU sharding of a packed batch (SURVEY.md section 8e).

Every string is an independent unit (context fills at latok.c:69-73,114-134; the block mask restarts
per call), so a batch is cut into G contiguous ranges of whole strings, balanced by bytes, and every
GPU runs the identical single-GPU pipeline on its range.  There is no data-path collective.  The only
cross-GPU datum is each shard's token (and character) count, needed to rebase the per-shard CSR
offsets into global ones: one all-gather of two int64 per rank (NCCL when the ranks are processes on
GPUs, gloo on CPU), or a host-side prefix sum when one process drives all devices.

Token vocabularies (encode_sharded / update_sharded) add one step: every shard counts its tokens into a scratch
vocabulary on its own device, and the caller's vocabulary merges the scratch vocabularies in shard order, which gives
the keys, ids and counts one GPU gets from the whole batch.
"""
from __future__ import annotations

import threading
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from .engine import SPANS, SPLITS, BatchResult


def shard_ranges(offsets: np.ndarray, n_shards: int) -> List[Tuple[int, int]]:
    """Cut [0, S) into n_shards contiguous string ranges whose boundaries are the string boundaries
    nearest to k * B / n_shards (B = total bytes).  Ranges may be empty when S < n_shards."""
    offsets = np.asarray(offsets, dtype=np.int64)
    S = len(offsets) - 1
    if n_shards < 1:
        raise ValueError("n_shards must be >= 1")
    total = int(offsets[-1])
    cuts = [0]
    for k in range(1, n_shards):
        target = total * k / n_shards
        j = int(np.searchsorted(offsets, target, side="left"))
        j = min(max(j, 0), S)
        if j > 0 and abs(int(offsets[j - 1]) - target) <= abs(int(offsets[j]) - target):
            j -= 1
        cuts.append(max(j, cuts[-1]))
    cuts.append(S)
    return [(cuts[i], cuts[i + 1]) for i in range(n_shards)]


def slice_shard(buf: np.ndarray, offsets: np.ndarray, s0: int, s1: int):
    """Byte range + rebased offsets of strings [s0, s1) (views, no copy of the bytes)."""
    b0, b1 = int(offsets[s0]), int(offsets[s1])
    return buf[b0:b1], (offsets[s0:s1 + 1] - b0)


def concat_offsets(arrs: Sequence[np.ndarray], counts: Sequence[int]) -> np.ndarray:
    """CSR offsets of consecutive shards (shard i has counts[i] items) as one CSR over their concatenation."""
    base = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    pieces = [a[:-1] + b for a, b in zip(arrs, base)]
    return np.concatenate(pieces + [np.array([int(np.sum(counts))], dtype=np.int64)])


def merge_results(parts: Sequence[BatchResult]) -> BatchResult:
    """Concatenate per-shard results of consecutive string ranges into one batch result, rebasing the
    CSR offsets by the running character / token counts (the host-side form of the count exchange)."""
    out = BatchResult(sum(p.n_strings for p in parts), sum(p.n_chars for p in parts), sum(p.n_tokens for p in parts))

    def cat(name):
        arrs = [getattr(p, name) for p in parts]
        return None if any(a is None for a in arrs) else np.concatenate(arrs)

    def cat_offsets(name, counts):
        arrs = [getattr(p, name) for p in parts]
        return None if any(a is None for a in arrs) else concat_offsets(arrs, counts)

    out.splits, out.spans, out.tok_feats, out.matrix = cat("splits"), cat("spans"), cat("tok_feats"), cat("matrix")
    out.char_offsets = cat_offsets("char_offsets", [p.n_chars for p in parts])
    out.tok_offsets = cat_offsets("tok_offsets", [p.n_tokens for p in parts])
    out.kernel_ms = max((p.kernel_ms for p in parts), default=0.0)
    out.lookahead_walks = sum(p.lookahead_walks for p in parts)
    return out


_engines = {}
_scratch = {}            # (device, shard position) -> scratch Vocab of encode_sharded / update_sharded
_engines_lock = threading.Lock()


def device_engine(device: int):
    """The process-wide engine of a device (created on first use; an Engine serialises its callers itself)."""
    from .engine import Engine
    with _engines_lock:
        e = _engines.get(device)
        if e is None:
            e = _engines[device] = Engine(device)
        return e


def close_engines():
    with _engines_lock:
        for v in _scratch.values():
            v.close()
        _scratch.clear()
        for e in _engines.values():
            e.close()
        _engines.clear()


def _run_shards(buf, offsets, devices, fn):
    """fn(i, shard buf, shard offsets) on one host thread per shard of the byte-balanced string ranges; the results in
    shard order, the first error re-raised on the caller's thread."""
    ranges = shard_ranges(offsets, len(devices))
    results: List = [None] * len(devices)
    errors: List[Optional[BaseException]] = [None] * len(devices)

    def work(i):
        try:
            b, o = slice_shard(buf, offsets, *ranges[i])
            results[i] = fn(i, np.ascontiguousarray(b), np.ascontiguousarray(o))
        except BaseException as exc:  # re-raised on the caller's thread
            errors[i] = exc

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(devices))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for exc in errors:
        if exc is not None:
            raise exc
    return results


def tokenize_sharded(buf: np.ndarray, offsets: np.ndarray, devices: Sequence[int], what: int = SPLITS | SPANS,
                     run_fn: Optional[Callable[[int, np.ndarray, np.ndarray, int], BatchResult]] = None) -> BatchResult:
    """One process, several GPUs: one host thread per shard and one long-lived Engine per device, each shard on its
    byte-balanced string range; results are concatenated on the host.  `run_fn(device, buf, offsets, what)` can be
    injected (tests use it to exercise the host logic without a GPU)."""
    def default_run(dev, b, o, w):
        return device_engine(dev).run_packed(b, o, w)      # one engine per device, kept alive between calls

    fn = run_fn or default_run
    return merge_results(_run_shards(buf, offsets, devices, lambda i, b, o: fn(devices[i], b, o, what)))


def _scratch_vocab(device: int, position: int):
    from .vocab import Vocab
    engine = device_engine(device)
    with _engines_lock:
        v = _scratch.get((device, position))
        if v is None:
            v = _scratch[(device, position)] = Vocab(engine)
        return v


def _replica(vocab, device: int):
    """A lookup copy of `vocab` on `device` (an empty vocabulary + merge), kept on `vocab` and rebuilt when `vocab`
    has changed since."""
    from .vocab import Vocab
    engine = device_engine(device)
    ver, r = vocab._replicas.get(device, (None, None))
    if r is None or r.engine is not engine:
        r = Vocab(engine, capacity=len(vocab))
    elif ver == vocab.version:
        return r
    else:
        r.clear()
    r._merge(vocab, "none")
    vocab._replicas[device] = (vocab.version, r)
    return r


def encode_sharded(vocab, buf: np.ndarray, offsets: np.ndarray, devices: Sequence[int], add: bool = True,
                   unk: int = -1, stats: Optional[dict] = None) -> Tuple[np.ndarray, np.ndarray]:
    """`vocab.encode_packed(buf, offsets, add, unk)` with the batch sharded over `devices` (one host thread per shard,
    one engine per device; a device may appear more than once): the same (ids int32[T], tok_offsets int64[S+1]), and
    `vocab` ends in the same state.

    add=True: every shard encodes into a scratch vocabulary on its device, the caller's thread merges the scratch
    vocabularies into `vocab` in shard order, and each shard's local ids are mapped to `vocab`'s ids on its device.
    add=False: every shard looks its tokens up in `vocab` itself on `vocab`'s device and in a replica of `vocab` (kept
    until `vocab` changes) on any other device.
    stats (add=True): filled with the device ms of every shard's encode ("shard_ms"), of every merge ("merge_ms",
    copy-in included) and of every shard's id gather ("remap_ms")."""
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    if not add:
        targets = [vocab if d == vocab.engine.device else _replica(vocab, d) for d in devices]
        parts = _run_shards(buf, offsets, devices, lambda i, b, o: targets[i].encode_packed(b, o, False, unk))
        ids = np.concatenate([p[0] for p in parts])
        return ids, concat_offsets([p[1] for p in parts], [len(p[0]) for p in parts])
    import torch
    parts = _add_sharded(vocab, buf, offsets, devices, "device", stats)
    out, events = [], []
    for sv, (local, tok_off) in parts:
        m = vocab._merge(sv, "device").to(local.device)
        if stats is not None:
            stats["merge_ms"].append(vocab.last_ms())
            with torch.cuda.device(local.device):
                events.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
                events[-1][0].record()
        out.append((torch.index_select(m, 0, local), tok_off.numpy()))     # plumbing: map_k[local_ids_k], one gather
        if stats is not None:
            with torch.cuda.device(local.device):
                events[-1][1].record()
    ids = torch.cat([o[0].cpu() for o in out]).numpy()
    if stats is not None:
        stats["remap_ms"] = [a.elapsed_time(b) for a, b in events]
    return ids, concat_offsets([o[1] for o in out], [len(o[0]) for o in out])


def update_sharded(vocab, buf: np.ndarray, offsets: np.ndarray, devices: Sequence[int],
                   stats: Optional[dict] = None) -> None:
    """`vocab.update` of a packed batch sharded over `devices`: `encode_sharded(add=True)` without the ids."""
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    for sv, _ in _add_sharded(vocab, buf, offsets, devices, "none", stats):
        vocab._merge(sv, "none")
        if stats is not None:
            stats["merge_ms"].append(vocab.last_ms())


def _add_sharded(vocab, buf, offsets, devices, out, stats):
    """every shard counted into its cleared scratch vocabulary: [(scratch vocab, its encode result)] in shard order"""
    if vocab.frozen:
        raise RuntimeError("this vocabulary is frozen (Vocab.from_tokens): use add=False")
    scratch = [_scratch_vocab(d, i) for i, d in enumerate(devices)]

    def shard(i, b, o):
        scratch[i].clear()
        return scratch[i], scratch[i]._run(b, o, True, -1, out)

    parts = _run_shards(buf, offsets, devices, shard)
    if stats is not None:
        stats.update(shard_ms=[sv.last_ms() for sv in scratch], merge_ms=[])
    return parts


def allgather_counts(n_chars: int, n_tokens: int, group=None):
    """One rank per GPU (torchrun): exchange (characters, tokens) of every rank's shard -- the path's only
    collective, 16 bytes per rank -- and return (all_counts [world, 2], char_base, token_base) for this rank."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    backend = dist.get_backend(group)
    device = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    mine = torch.tensor([n_chars, n_tokens], dtype=torch.int64, device=device)
    out = torch.zeros(world * 2, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, mine, group=group)
    counts = out.view(world, 2).cpu().numpy()
    base = counts[:rank].sum(axis=0) if rank else np.zeros(2, dtype=np.int64)
    return counts, int(base[0]), int(base[1])


def rebase_for_rank(result: BatchResult, char_base: int, token_base: int) -> BatchResult:
    """Turn a rank's shard-local CSR offsets into offsets into the global (all ranks) arrays."""
    if result.char_offsets is not None:
        result.char_offsets = result.char_offsets + char_base
    if result.tok_offsets is not None:
        result.tok_offsets = result.tok_offsets + token_base
    return result
