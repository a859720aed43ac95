"""Token vocabulary on the GPU: corpus token counts and integer token ids (kernels: csrc/latok_vocab.cu).

    v = Vocab()                          # on the default engine's device
    v.update(texts)                      # Counter().update over the tokens of tokenize_batch(texts)
    ids, tok_offsets = v.encode(texts)   # int32 id per token (new tokens get the next ids), CSR per string
    v.most_common(10)                    # [(token, count), ...]
    frozen = Vocab.from_tokens([t for t, c in v.most_common() if c >= 5])
    ids, _ = frozen.encode(texts, add=False, unk=-1)
    m = v.merge(w)                       # Counter.update(w); m[i] = v's id of w's key i (w may be on another GPU)
    ids, offsets, word_offsets = frozen.wordpiece(texts, unk=0)    # WordPiece pieces of every token ("##" + rest)

Keys are the exact token texts (``text[s:e].strip()`` of the tokenizer, no normalisation); ids are dense and follow the
order of first occurrence, so two vocabularies fed the same batches agree id for id.  A vocabulary lives on one GPU;
merging vocabularies built from consecutive shards of a batch, in shard order, gives the vocabulary one GPU builds
from the whole batch (latok_b200.sharding.encode_sharded / update_sharded count and encode a batch over several GPUs).
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .engine import SPANS, default_engine, pack_strings


class Vocab:
    """Device-resident vocabulary bound to an engine (default: the process-wide engine of device 0).  `capacity`:
    keys expected (the table grows past it).  A vocabulary made by `from_tokens` is frozen: it only looks tokens up."""

    def __init__(self, engine=None, capacity: int = 0):
        self.engine = engine or default_engine()
        self._L = self.engine._L
        self.frozen = False
        self.version = 0             # +1 for every change of keys or counts (replicas of latok_b200.sharding)
        self._replicas = {}          # device -> (version, Vocab): lookup copies for sharded encodes
        h = C.c_void_p()
        with self.engine._lock:
            _lib.check(self._L.latok_b200_vocab_create(self.engine._h, int(capacity), C.byref(h)))
        self._h = h

    def close(self):
        for _, r in getattr(self, "_replicas", {}).values():
            r.close()
        if getattr(self, "_h", None):
            self._L.latok_b200_vocab_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- batches ---------------------------------------------------------------------------------
    def _encode_oldest(self, add: bool, unk: int, ids) -> None:
        if add and self.frozen:
            raise RuntimeError("this vocabulary is frozen (Vocab.from_tokens): use add=False")
        e = self.engine
        _, n_tokens = e.sizes()
        ptr, on_device = None, 0
        if ids is not None:
            if isinstance(ids, np.ndarray):
                ptr = ids.ctypes.data if n_tokens else None
            else:
                ptr, on_device = ids.data_ptr(), 1
        _lib.check(self._L.latok_b200_vocab_encode(e._h, self._h, 1 if add else 0, int(unk), n_tokens, ptr, on_device))
        if add:
            self.version += 1

    def encode_oldest(self, add: bool = True, unk: int = -1, want_ids: bool = True) -> Optional[np.ndarray]:
        """int32 ids of the tokens of the engine's oldest batch in flight (submitted with SPANS), or None without
        `want_ids` (counting only).  This is the pipelined form: at depth 2 the caller submits batch i+1, encodes batch
        i and releases it, so that the next batch's copy-in and kernels overlap this one."""
        with self.engine._lock:
            ids = None
            if want_ids:
                ids = np.empty(self.engine.sizes()[1], dtype=np.int32)
            self._encode_oldest(add, unk, ids)
            return ids

    def _run(self, buf, offsets, add: bool, unk: int, out: str):
        e = self.engine
        with e._lock:
            if e._depth == 2 and e._flight:
                raise RuntimeError("batches are in flight")
            e.submit(buf, offsets, SPANS)
            try:
                if out == "none":
                    self._encode_oldest(add, unk, None)
                    return None
                _, n_tokens = e.sizes()
                tok_off = np.empty(len(offsets), dtype=np.int64)
                _lib.check(self._L.latok_b200_fetch(e._h, 0, 0, len(offsets) - 1, None, None, None, tok_off.ctypes.data,
                                                    None, None))
                if out == "device":
                    import torch
                    ids = torch.empty(n_tokens, dtype=torch.int32, device=f"cuda:{e.device}")
                    self._encode_oldest(add, unk, ids)
                    return ids, torch.from_numpy(tok_off)
                ids = np.empty(n_tokens, dtype=np.int32)
                self._encode_oldest(add, unk, ids)
                return ids, tok_off
            finally:
                if e._depth == 2:
                    e.release()

    def update(self, texts: Sequence[str]) -> None:
        """Count the tokens of `texts` (new tokens get the next ids); no ids are copied out."""
        self._run(*pack_strings(texts), True, -1, "none")

    def encode(self, texts: Sequence[str], add: bool = True, unk: int = -1) -> Tuple[np.ndarray, np.ndarray]:
        """(ids int32[T], tok_offsets int64[S+1]): the id of every token in token order; string i has the ids
        ids[tok_offsets[i]:tok_offsets[i+1]].  add=True counts the tokens and adds new ones; add=False looks them up
        and gives `unk` to unknown ones."""
        return self._run(*pack_strings(texts), add, unk, "host")

    def encode_packed(self, buf, offsets, add: bool = True, unk: int = -1, device: bool = False):
        """`encode` for packed UTF-8 (uint8 buffer + int64 offsets[S+1]).  device=True: the ids are written straight
        into a CUDA int32 tensor on the engine's device and (ids, tok_offsets) come back as torch tensors."""
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        return self._run(buf, offsets, add, unk, "device" if device else "host")

    def wordpiece(self, texts: Sequence[str], unk: int, prefix: str = "##", max_chars: int = 100):
        """WordPiece pieces of the tokens of `texts`: every token is split greedily into the longest prefix that is a
        key, then the longest continuations that are keys as `prefix` + rest (BERT's WordpieceTokenizer, HF
        tokenizers' WordPiece); a token of more than `max_chars` characters, or one that cannot be split, is the single
        piece `unk`.  Returns (ids int32[P], offsets int64[S+1], word_offsets int64[T+1]): string i has the pieces
        ids[offsets[i]:offsets[i+1]], token k the pieces ids[word_offsets[k]:word_offsets[k+1]].  Only reads the
        vocabulary."""
        return self._wordpiece(*pack_strings(texts), unk, prefix, max_chars, False)

    def wordpiece_packed(self, buf, offsets, unk: int, prefix: str = "##", max_chars: int = 100, device: bool = False):
        """`wordpiece` for packed UTF-8 (uint8 buffer + int64 offsets[S+1]).  device=True: ids and word_offsets are
        CUDA tensors on the engine's device (offsets a CPU tensor)."""
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        return self._wordpiece(buf, offsets, unk, prefix, max_chars, device)

    def _wordpiece(self, buf, offsets, unk: int, prefix, max_chars: int, device: bool):
        pre = prefix.encode("utf-8", "surrogatepass") if isinstance(prefix, str) else bytes(prefix)
        pre_buf = C.create_string_buffer(pre, max(len(pre), 1))
        e = self.engine
        with e._lock:
            if e._depth == 2 and e._flight:
                raise RuntimeError("batches are in flight")
            e.submit(buf, offsets, SPANS)
            try:
                _, n_tokens = e.sizes()
                tok_off = np.empty(len(offsets), dtype=np.int64)
                _lib.check(self._L.latok_b200_fetch(e._h, 0, 0, len(offsets) - 1, None, None, None, tok_off.ctypes.data,
                                                    None, None))
                if device:
                    import torch
                    word_off = torch.empty(n_tokens + 1, dtype=torch.int64, device=f"cuda:{e.device}")
                    ptr = word_off.data_ptr()
                else:
                    word_off = np.empty(n_tokens + 1, dtype=np.int64)
                    ptr = word_off.ctypes.data
                n = C.c_int64(0)
                _lib.check(self._L.latok_b200_vocab_wordpiece(e._h, self._h, pre_buf, len(pre), int(max_chars), int(unk),
                                                              n_tokens, ptr, C.byref(n), 1 if device else 0))
                if device:
                    ids = torch.empty(n.value, dtype=torch.int32, device=word_off.device)
                    _lib.check(self._L.latok_b200_vocab_wordpiece_fetch(e._h, n.value, ids.data_ptr(), 1))
                    offs = word_off[torch.from_numpy(tok_off).to(word_off.device)].cpu()    # plumbing: S+1 gathers
                    return ids, offs, word_off
                ids = np.empty(n.value, dtype=np.int32)
                _lib.check(self._L.latok_b200_vocab_wordpiece_fetch(e._h, n.value, ids.ctypes.data if n.value else None, 0))
                return ids, word_off[tok_off], word_off
            finally:
                if e._depth == 2:
                    e.release()

    def merge(self, other: "Vocab", device: bool = False):
        """Counter.update(other) on the device: every key of `other` is added with its count, keys new to `self` get
        the next ids in `other`'s id order.  Returns the map from `other`'s ids to `self`'s: int32 NumPy array of
        len(other), or (device=True) a CUDA int32 tensor on `self`'s device.  `other` may live on another GPU."""
        return self._merge(other, "device" if device else "host")

    def _merge(self, other: "Vocab", out: str):
        if self.frozen:
            raise RuntimeError("this vocabulary is frozen (Vocab.from_tokens): it cannot take a merge")
        if other is self:
            raise ValueError("a vocabulary cannot be merged into itself")
        # both engines' locks, in one order for every caller: two threads merging in opposite directions cannot deadlock
        engines = {id(e): e for e in (self.engine, other.engine)}.values()
        with contextlib.ExitStack() as held:
            for e in sorted(engines, key=lambda e: (e.device, id(e))):
                held.enter_context(e._lock)
            n = len(other)
            m, ptr, on_device = None, None, 0
            if out == "device":
                import torch
                m = torch.empty(n, dtype=torch.int32, device=f"cuda:{self.engine.device}")
                ptr, on_device = m.data_ptr(), 1
            elif out == "host":
                m = np.empty(n, dtype=np.int32)
                ptr = m.ctypes.data if n else None
            _lib.check(self._L.latok_b200_vocab_merge(self.engine._h, self._h, other._h, ptr, on_device))
            self.version += 1
            return m

    def clear(self) -> None:
        """Drop every key and count (the device allocations stay for the next batches)."""
        if self.frozen:
            raise RuntimeError("this vocabulary is frozen (Vocab.from_tokens): it cannot be cleared")
        with self.engine._lock:
            _lib.check(self._L.latok_b200_vocab_clear(self._h))
            self.version += 1

    # ---- contents --------------------------------------------------------------------------------
    def _size(self):
        n, b = C.c_int64(0), C.c_int64(0)
        _lib.check(self._L.latok_b200_vocab_size(self._h, C.byref(n), C.byref(b), None))
        return n.value, b.value

    def table_slots(self) -> int:
        """Slots of the device hash table (the load is len(self) / table_slots())."""
        n = C.c_int64(0)
        _lib.check(self._L.latok_b200_vocab_size(self._h, None, None, C.byref(n)))
        return n.value

    def __len__(self):
        return self._size()[0]

    def _export(self, keys: bool, counts: bool):
        with self.engine._lock:
            n, nb = self._size()
            buf = np.empty(nb, dtype=np.uint8) if keys else None
            off = np.empty(n + 1, dtype=np.int64) if keys else None
            cnt = np.empty(n, dtype=np.int64) if counts else None
            _lib.check(self._L.latok_b200_vocab_export(
                self._h, n, nb, buf.ctypes.data if keys and nb else None, off.ctypes.data if keys else None,
                cnt.ctypes.data if counts and n else None))
            return buf, off, cnt

    def tokens(self) -> List[str]:
        """The keys in id order."""
        buf, off, _ = self._export(True, False)
        b = buf.tobytes()
        return [b[off[i]:off[i + 1]].decode("utf-8", "surrogatepass") for i in range(len(off) - 1)]

    def counts(self) -> np.ndarray:
        """int64 count per id."""
        return self._export(False, True)[2]

    def most_common(self, n: Optional[int] = None) -> List[Tuple[str, int]]:
        """(token, count) by count, highest first; equal counts in id order (first occurrence first)."""
        cnt = self.counts()
        order = np.argsort(-cnt, kind="stable")[:n]
        toks = self.tokens()
        return [(toks[i], int(cnt[i])) for i in order]

    @classmethod
    def from_tokens(cls, tokens: Sequence[str], counts=None, engine=None) -> "Vocab":
        """A frozen vocabulary with id = position in `tokens` (and the given counts, default 0).  An empty or repeated
        token raises ValueError."""
        v = cls(engine, capacity=len(tokens))
        enc = [t.encode("utf-8", "surrogatepass") for t in tokens]
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        if enc:
            np.cumsum([len(b) for b in enc], out=off[1:])
        buf = np.frombuffer(b"".join(enc), dtype=np.uint8)
        cnt = None if counts is None else np.ascontiguousarray(counts, dtype=np.int64)
        if cnt is not None and cnt.shape != (len(tokens),):
            raise ValueError("counts must have one entry per token")
        with v.engine._lock:
            _lib.check(v._L.latok_b200_vocab_import(v.engine._h, v._h, buf.ctypes.data if len(buf) else None,
                                                    off.ctypes.data, len(tokens),
                                                    None if cnt is None else cnt.ctypes.data))
        v.frozen = True
        v.version += 1
        return v

    def last_ms(self) -> float:
        """Device time of the last encode / update / import / merge / wordpiece (token byte ranges and a merge's copy-in
        included)."""
        ms = C.c_float(0)
        _lib.check(self._L.latok_b200_vocab_last_ms(self._h, C.byref(ms)))
        return ms.value
