// latok_vocab.cu -- token vocabulary on the device: corpus token counts and integer token ids.
//
// A vocabulary is an open-addressing hash table (linear probing, power-of-two capacity) keyed by the exact trimmed token
// bytes, i.e. utf8[b:e] of the byte ranges of latok_tokbytes.cu.  Two keys are equal only when their bytes are equal; a
// hash match alone never merges them.  A slot is 16 bytes {hash, ref}, claimed by one 128-bit atomicCAS:
//   hash  64-bit hash of the key (0 = empty slot)
//   ref   k + 1 for a key first claimed by token k of the current launch, VOCAB_COMMITTED | id for a committed key
// Committed key bytes live in the key arena: arena[key_off[id], key_off[id + 1]).
//
// One batch (host side: latok_capi.cu, latok_b200_vocab_encode / _import):
//   vocab_insert_kernel  every token probes its slot; an empty slot is claimed, a slot with the token's hash is compared
//                        byte for byte against the claiming token's text or the arena right away, so no thread waits on
//                        another.  Probe loops are bounded; a grid-wide count of new claims enforces the load limit and
//                        sets the overflow flag (the host then grows the table, rehashes the committed keys and runs the
//                        batch again: the batch commits all at once or not at all).  first_occ[slot] = min token index.
//   vocab_flag_kernel    rank[k] = 1 for the first occurrence of a key new in this batch; counts of new keys and bytes
//   (exclusive scan)     rank[k] = new id - n_keys, in token order: ids do not depend on which thread won a CAS
//   vocab_lens_kernel    lengths of the new keys at key_off[n_keys + rank]
//   (exclusive scan)     arena offsets of the new keys
//   vocab_commit_kernel  copies the new keys into the arena and rewrites their slots' ref to VOCAB_COMMITTED | id
//   vocab_count_kernel   ids per token; counts += 1 per token, aggregated within a warp first (__match_any_sync: a Zipf
//                        stream puts most increments on a handful of slots), or += weight[k] per key (merge)
// Lookup (frozen use) is vocab_insert_kernel without claims: id of the key, or the caller's unk id.
// Merge (latok_b200_vocab_merge) is one batch whose tokens are the source's keys in id order, weighted by their counts:
// vocab_ranges_kernel turns the source's key offsets into the batch's ranges on the device, and the count kernel's ids
// are the map source id -> destination id.
// WordPiece (latok_b200_vocab_wordpiece) only reads the table: vocab_max_key_kernel finds the longest key,
// vocab_wp_count_kernel splits every token greedily, longest piece first (one lane per token; a candidate piece is a Key
// "prefix + text range", hashed as a running sum while its end moves), a scan of the piece counts gives the word
// offsets, and vocab_wp_write_kernel writes the ids, searching again only for tokens of several pieces.
// Keys of up to VOCAB_LONG bytes take one lane each; longer keys (documents reach 64 KB per string) a whole warp each.
// Integer / memory-bound kernels; no tensor cores.
#include "latok_internal.h"

#include <type_traits>
#include <cub/device/device_scan.cuh>
#include <cuda/std/functional>

namespace latok {

constexpr int VOCAB_LONG = 256;

__device__ __forceinline__ unsigned long long fmix64(unsigned long long k)
{
    k ^= k >> 33; k *= 0xFF51AFD7ED558CCDULL;
    k ^= k >> 33; k *= 0xC4CEB9FE1A85EC53ULL;
    k ^= k >> 33;
    return k;
}

// bytes [p, p + 8) of a byte range that ends at e, little endian, zero at and beyond e (p < e).  Reads only the aligned
// 8-byte words that hold a byte of the range, so a range at the very end of an allocation is read in bounds.
__device__ __forceinline__ unsigned long long range_word(const uint8_t *base, long long p, long long e)
{
    const long long a = p & ~7LL;
    const int sh = (int)(p & 7);
    unsigned long long w = __ldg(reinterpret_cast<const unsigned long long *>(base + a)) >> (8 * sh);
    if (sh && a + 8 < e) w |= __ldg(reinterpret_cast<const unsigned long long *>(base + a + 8)) << (64 - 8 * sh);
    const long long n = e - p;
    if (n < 8) w &= (1ULL << (8 * n)) - 1ULL;
    return w;
}

// A key: the bytes pre[0, plen) followed by base[b, e).  A token, a claimed key and an arena key have plen = 0; a
// WordPiece candidate is the continuation prefix followed by a piece of a token (plen = 0 for a word's first piece).
struct Key {
    const uint8_t *pre;
    long long plen;
    const uint8_t *base;
    long long b, e;
    __device__ long long len() const { return plen + e - b; }
};
__device__ __forceinline__ Key plain_key(const uint8_t *base, long long b, long long e) { return Key{nullptr, 0, base, b, e}; }

// bytes [q, q + 8) of key k, little endian, zero at and beyond its end (0 <= q < k.len())
__device__ __forceinline__ unsigned long long key_word(const Key &k, long long q)
{
    if (q >= k.plen) return range_word(k.base, k.b + q - k.plen, k.e);
    unsigned long long w = range_word(k.pre, q, k.plen);
    const long long room = k.plen - q;
    if (room < 8 && k.b < k.e) w |= range_word(k.base, k.b, k.e) << (8 * room);
    return w;
}

// The hash of a key is the sum over its 8-byte words of a mix keyed by the word index (word_term), finalised with the
// length (hash_final): a warp adds its lanes' partial sums in any order and gets the value one lane computes, and a
// WordPiece search keeps the sum of a candidate's whole words while the candidate shrinks.  hmask truncates it
// (LATOK_B200_VOCAB_HASH_BITS).
__device__ __forceinline__ unsigned long long word_term(unsigned long long w, long long i)
{
    return fmix64(w ^ (0x9E3779B97F4A7C15ULL * (unsigned long long)(i + 1)));
}
__device__ __forceinline__ unsigned long long hash_final(unsigned long long s, long long len, unsigned long long hmask)
{
    const unsigned long long h = fmix64(s ^ (0xD6E8FEB86659FD93ULL * (unsigned long long)len)) & hmask;
    return h ? h : 1ULL;
}

template <bool WARP>
__device__ __forceinline__ unsigned long long key_hash(const Key &k, unsigned long long hmask, int lane)
{
    unsigned long long s = 0;
    const long long nw = (k.len() + 7) >> 3;
    for (long long i = WARP ? lane : 0; i < nw; i += WARP ? 32 : 1) s += word_term(key_word(k, 8 * i), i);
    if (WARP)
        for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
    return hash_final(s, k.len(), hmask);
}

// a == b for two keys of length len
template <bool WARP>
__device__ __forceinline__ bool key_equal(const Key &a, const Key &b, long long len, int lane)
{
    bool eq = true;
    const long long nw = (len + 7) >> 3;
    for (long long i = WARP ? lane : 0; eq && i < nw; i += WARP ? 32 : 1) eq = key_word(a, 8 * i) == key_word(b, 8 * i);
    return WARP ? __all_sync(0xFFFFFFFFu, eq) : eq;
}

// One lane per key of a warp's 32, then every key longer than VOCAB_LONG bytes by the whole warp.  visit(warp, k, range,
// lane) with warp = std::true_type / std::false_type; all lanes of the warp take part in the warp visits.  Then
// after(k, live) with the warp converged.
template <class Range, class Visit, class After>
__device__ __forceinline__ void each_key(long long n, Range range, Visit visit, After after)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long base = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < n; base += warps * 32) {
        const long long k = base + lane;
        const bool live = k < n;
        const longlong2 r = live ? range(k) : make_longlong2(0, 0);
        const bool wide = live && r.y - r.x > VOCAB_LONG;
        if (live && !wide) visit(std::false_type{}, k, r, lane, lane);
        for (unsigned m = __ballot_sync(0xFFFFFFFFu, wide); m; m &= m - 1) {
            const int src = __ffs(m) - 1;
            visit(std::true_type{}, base + src, range(base + src), lane, src);
        }
        after(k, live);
    }
}

__device__ __forceinline__ void set_overflow(VocabStatus *st) { atomicExch(&st->overflow, 1u); }

// the slot of `key` (hash h = key_hash(key)), token k of the launch: claimed if absent (add), -1 if absent (lookup) or
// no slot could be had (overflow flag set).  *committed_id: the key's id when it was committed before this launch, else -1.
template <bool WARP>
__device__ long long probe(const VocabParams &p, long long k, const Key &key, unsigned long long h, bool add, int lane,
                           long long *committed_id)
{
    const long long len = key.len();
    unsigned long long s = h & p.mask;
    for (unsigned long long i = 0; i <= p.mask; ++i, s = (s + 1) & p.mask) {
        VocabSlot v = p.table[s];
        if (WARP) { v.hash = __shfl_sync(0xFFFFFFFFu, v.hash, 0); v.ref = __shfl_sync(0xFFFFFFFFu, v.ref, 0); }
        if (add && (v.hash == 0 || v.ref == 0)) {
            // empty, or a claim of this launch not yet wholly visible to the plain load: the CAS claims the slot or
            // returns its value atomically
            VocabSlot old;
            if (!WARP || lane == 0) {
                VocabSlot mine; mine.hash = h; mine.ref = (unsigned long long)k + 1;
                VocabSlot none; none.hash = 0; none.ref = 0;
                old = atomicCAS(&p.table[s], none, mine);
                if (old.hash == 0 && atomicAdd(&p.st->claims, 1ULL) + 1 > p.limit) set_overflow(p.st);
            }
            if (WARP) { old.hash = __shfl_sync(0xFFFFFFFFu, old.hash, 0); old.ref = __shfl_sync(0xFFFFFFFFu, old.ref, 0); }
            if (old.hash == 0) { *committed_id = -1; return (long long)s; }
            v = old;
        } else if (v.hash == 0) {
            return -1;
        }
        if (v.hash != h) continue;
        bool eq;
        if (v.ref & VOCAB_COMMITTED) {
            const long long id = (long long)(v.ref & ~VOCAB_COMMITTED), kb = p.key_off[id];
            eq = p.key_off[id + 1] - kb == len && key_equal<WARP>(key, plain_key(p.arena, kb, kb + len), len, lane);
            if (eq) { *committed_id = id; return (long long)s; }
        } else {
            const longlong2 o = p.rng[v.ref - 1];
            eq = o.y - o.x == len && key_equal<WARP>(key, plain_key(p.text, o.x, o.y), len, lane);
            if (eq) { *committed_id = -1; return (long long)s; }
        }
    }
    if (add && (!WARP || lane == 0)) set_overflow(p.st);
    return -1;
}

// the slot of token k = text[r.x, r.y), as probe
template <bool WARP>
__device__ __forceinline__ long long probe_token(const VocabParams &p, long long k, longlong2 r, bool add, int lane,
                                                 long long *committed_id)
{
    const Key key = plain_key(p.text, r.x, r.y);
    return probe<WARP>(p, k, key, key_hash<WARP>(key, p.hmask, lane), add, lane, committed_id);
}

// first_occ[slot] = min token index over the keys of slots claimed in this launch: one atomicMin per group of lanes
// with the same slot (the lowest lane holds the group's smallest index), and none when a smaller index is already
// visible (a Zipf stream sends most tokens of a batch to a few slots)
__global__ void __launch_bounds__(256) vocab_insert_kernel(const VocabParams p)
{
    long long my_s = -1;
    each_key(p.n, [&](long long k) { return p.rng[k]; },
             [&](auto warp, long long k, longlong2 r, int lane, int owner) {
        long long id = -1;
        const long long s = probe_token<decltype(warp)::value>(p, k, r, true, lane, &id);
        if (lane == owner) my_s = s >= 0 && id < 0 ? s : -1;
        if (lane == 0 || !decltype(warp)::value) p.slot[k] = s < 0 ? 0u : (uint32_t)s;
    }, [&](long long k, bool live) {
        const int lane = threadIdx.x & 31;
        const bool claim = live && my_s >= 0;
        const unsigned same = __match_any_sync(0xFFFFFFFFu, claim ? my_s : -1 - lane);
        if (claim && lane == __ffs(same) - 1 && __ldcg(&p.first_occ[my_s]) > (unsigned long long)k)
            atomicMin(&p.first_occ[my_s], (unsigned long long)k);
        my_s = -1;
    });
}

__global__ void __launch_bounds__(256) vocab_lookup_kernel(const VocabParams p)
{
    each_key(p.n, [&](long long k) { return p.rng[k]; }, [&](auto warp, long long k, longlong2 r, int lane, int) {
        long long id = -1;
        const long long s = probe_token<decltype(warp)::value>(p, k, r, false, lane, &id);
        if (lane == 0 || !decltype(warp)::value) p.ids[k] = s >= 0 && id >= 0 ? (int32_t)id : p.unk;
    }, [](long long, bool) {});
}

// rank[k] = 1 for the first occurrence of a key claimed in this batch; rank[n] = 0 (the scan's total lands there)
__global__ void __launch_bounds__(256) vocab_flag_kernel(const VocabParams p)
{
    if (*(volatile unsigned *)&p.st->overflow) return;
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < p.n; base += stride) {
        const long long k = base + lane;
        bool f = false;
        long long len = 0;
        if (k < p.n) {
            const uint32_t s = p.slot[k];
            f = !(p.table[s].ref & VOCAB_COMMITTED) && p.first_occ[s] == (unsigned long long)k;
            if (f) { const longlong2 r = p.rng[k]; len = r.y - r.x; }
            p.rank[k] = f;
        }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, f);
        for (int d = 16; d; d >>= 1) len += __shfl_xor_sync(0xFFFFFFFFu, len, d);
        if (lane == 0 && m) {
            atomicAdd(&p.st->n_new, (unsigned long long)__popc(m));
            atomicAdd(&p.st->new_bytes, (unsigned long long)len);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) p.rank[p.n] = 0;
}

// after the scan of rank: key k is new iff rank[k + 1] != rank[k]
__global__ void __launch_bounds__(256) vocab_lens_kernel(const VocabParams p, long long n_new)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < p.n; k += (long long)gridDim.x * blockDim.x)
        if (p.rank[k + 1] != p.rank[k]) { const longlong2 r = p.rng[k]; p.key_off[p.n_keys + p.rank[k]] = r.y - r.x; }
    if (blockIdx.x == 0 && threadIdx.x == 0) p.key_off[p.n_keys + n_new] = 0;
}

// a warp per 32 keys: the new ones are copied into the arena by the whole warp, one after the other
__global__ void __launch_bounds__(256) vocab_commit_kernel(const VocabParams p)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long base = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < p.n; base += warps * 32) {
        const long long k = base + lane;
        const bool f = k < p.n && p.rank[k + 1] != p.rank[k];
        for (unsigned m = __ballot_sync(0xFFFFFFFFu, f); m; m &= m - 1) {
            const long long kk = base + __ffs(m) - 1;
            const long long id = p.n_keys + p.rank[kk];
            const longlong2 r = p.rng[kk];
            uint8_t *dst = p.arena + p.key_off[id];
            for (long long j = lane; j < r.y - r.x; j += 32) dst[j] = p.text[r.x + j];
            if (lane == 0) p.table[p.slot[kk]].ref = VOCAB_COMMITTED | (unsigned long long)id;
        }
    }
}

// ids per token (ids may be NULL) and counts += 1 per token (counts may be NULL), or counts += weight[k] per token with
// weights (a merge: its tokens are distinct keys, so there is nothing to aggregate)
__global__ void __launch_bounds__(256) vocab_count_kernel(const VocabParams p)
{
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < p.n; base += stride) {
        const long long k = base + lane;
        long long id = -1 - lane;                        // dead lanes: a group of their own
        if (k < p.n) {
            id = (long long)(p.table[p.slot[k]].ref & ~VOCAB_COMMITTED);
            if (p.ids) p.ids[k] = (int32_t)id;
        }
        if (p.weight) {
            if (k < p.n && p.counts) atomicAdd(&p.counts[id], (unsigned long long)p.weight[k]);
        } else if (p.counts) {
            const unsigned same = __match_any_sync(0xFFFFFFFFu, id);
            if (k < p.n && lane == __ffs(same) - 1) atomicAdd(&p.counts[id], (unsigned long long)__popc(same));
        }
    }
}

// committed keys 0..n_keys-1 into an empty table (keys are distinct: no comparison)
__global__ void __launch_bounds__(256) vocab_rehash_kernel(const VocabParams p)
{
    each_key(p.n_keys, [&](long long id) { return make_longlong2(p.key_off[id], p.key_off[id + 1]); },
             [&](auto warp, long long id, longlong2 r, int lane, int) {
        const unsigned long long h = key_hash<decltype(warp)::value>(plain_key(p.arena, r.x, r.y), p.hmask, lane);
        if (decltype(warp)::value && lane != 0) return;
        unsigned long long s = h & p.mask;
        VocabSlot mine; mine.hash = h; mine.ref = VOCAB_COMMITTED | (unsigned long long)id;
        VocabSlot none; none.hash = 0; none.ref = 0;
        for (unsigned long long i = 0; i <= p.mask; ++i, s = (s + 1) & p.mask)
            if (atomicCAS(&p.table[s], none, mine).hash == 0) return;
        set_overflow(p.st);
    }, [](long long, bool) {});
}

// rng[k] = (key_off[k], key_off[k + 1]): the ranges of a merge's source keys in its arena
__global__ void __launch_bounds__(256) vocab_ranges_kernel(const long long *key_off, long long n, longlong2 *rng)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x)
        rng[k] = make_longlong2(key_off[k], key_off[k + 1]);
}

// ---- WordPiece: the pieces of every token (latok_b200_vocab_wordpiece) ---------------------------------------------
// st->max_key = the longest key of the vocabulary (no candidate longer than it can match)
__global__ void __launch_bounds__(256) vocab_max_key_kernel(const VocabParams p)
{
    long long m = 0;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < p.n_keys; k += (long long)gridDim.x * blockDim.x)
        m = max(m, p.key_off[k + 1] - p.key_off[k]);
    for (int d = 16; d; d >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(&p.st->max_key, (unsigned long long)m);
}

// more than max_chars characters in text[b, e)?  Counts only as far as max_chars + 1 characters.
__device__ __forceinline__ bool wp_too_long(const uint8_t *text, long long b, long long e, long long max_chars)
{
    long long chars = 0;
    for (long long q = b; q < e && chars <= max_chars; q += 8) {
        const unsigned long long w = range_word(text, q, e);          // zero bytes past e: not continuation bytes
        chars += min(8LL, e - q) - __popcll(w & ~(w << 1) & 0x8080808080808080ULL);
    }
    return chars > max_chars;
}

// Greedy longest-match-first split of the word text[b, e): emit(id) for every piece in order; the number of pieces, or
// 0 when some start has no piece (the word is then unk).  At every start the candidate ends go down from the longest
// key the vocabulary holds and stop at the first character boundary whose key (the prefix after the first piece, then
// text[start, end)) is a key.  The hash of a candidate is the sum of the terms of its whole 8-byte words, kept while
// `end` moves (a word's term leaves the sum when the word stops being whole), plus the term of its partial last word.
template <class Emit>
__device__ __forceinline__ long long wp_search(const VocabParams &p, long long b, long long e, long long max_key, Emit emit)
{
    long long n = 0;
    for (long long start = b; start < e;) {
        Key key{p.pre, start > b ? (long long)p.plen : 0, p.text, start, min(e, start + max_key - (start > b ? p.plen : 0))};
        if (key.e <= start) return 0;
        unsigned long long whole = 0;
        for (long long i = 0; i < key.len() >> 3; ++i) whole += word_term(key_word(key, 8 * i), i);
        long long id = -1;
        for (; key.e > start; --key.e) {
            const long long len = key.len();
            if (key.e == e || (__ldg(p.text + key.e) & 0xC0) != 0x80) {
                const unsigned long long part = len & 7 ? word_term(key_word(key, len & ~7LL), len >> 3) : 0ULL;
                if (probe<false>(p, 0, key, hash_final(whole + part, len, p.hmask), false, 0, &id) < 0) id = -1;
                if (id >= 0) break;
            }
            if (!(len & 7)) whole -= word_term(key_word(key, len - 8), (len >> 3) - 1);
        }
        if (id < 0) return 0;
        emit(n++, (int32_t)id);
        start = key.e;
    }
    return n;
}

// wp_off[k] = pieces of token k (1 for an unk word), wp_first[k] = the id of a one-piece word; wp_off[n] = 0 (the
// scan's total lands there)
__global__ void __launch_bounds__(256, 2) vocab_wp_count_kernel(const VocabParams p)
{
    const long long max_key = (long long)*(volatile unsigned long long *)&p.st->max_key;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < p.n; k += (long long)gridDim.x * blockDim.x) {
        const longlong2 r = p.rng[k];
        int32_t first = p.unk;
        long long n = 0;
        if (!wp_too_long(p.text, r.x, r.y, p.max_chars))
            n = wp_search(p, r.x, r.y, max_key, [&](long long j, int32_t id) { if (j == 0) first = id; });
        p.wp_off[k] = n ? n : 1;
        p.wp_first[k] = n == 1 ? first : p.unk;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) p.wp_off[p.n] = 0;
}

// after the scan of wp_off: the ids of token k's pieces at ids[wp_off[k]]; only words of several pieces search again
__global__ void __launch_bounds__(256) vocab_wp_write_kernel(const VocabParams p)
{
    const long long max_key = (long long)*(volatile unsigned long long *)&p.st->max_key;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < p.n; k += (long long)gridDim.x * blockDim.x) {
        const long long o = p.wp_off[k];
        if (p.wp_off[k + 1] - o == 1) { p.ids[o] = p.wp_first[k]; continue; }
        const longlong2 r = p.rng[k];
        wp_search(p, r.x, r.y, max_key, [&](long long j, int32_t id) { p.ids[o + j] = id; });
    }
}

static unsigned grid_for(long long n, int per_block, int n_sm)
{
    const long long want = (n + per_block - 1) / per_block, cap = (long long)n_sm * 8;
    return (unsigned)(want < 1 ? 1 : want < cap ? want : cap);
}

cudaError_t launch_vocab(VocabPhase phase, const VocabParams &p, long long n_new, int n_sm, cudaStream_t s)
{
    switch (phase) {
    case VOCAB_INSERT: vocab_insert_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_LOOKUP: vocab_lookup_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_FLAG: vocab_flag_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_LENS: vocab_lens_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p, n_new); break;
    case VOCAB_COMMIT: vocab_commit_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_COUNT: vocab_count_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_REHASH: if (p.n_keys) vocab_rehash_kernel<<<grid_for(p.n_keys, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_MAX_KEY: if (p.n_keys) vocab_max_key_kernel<<<grid_for(p.n_keys, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_WP_COUNT: vocab_wp_count_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    case VOCAB_WP_WRITE: if (p.n) vocab_wp_write_kernel<<<grid_for(p.n, 256, n_sm), 256, 0, s>>>(p); break;
    }
    return cudaGetLastError();
}

cudaError_t launch_vocab_ranges(const long long *key_off, long long n, longlong2 *rng, int n_sm, cudaStream_t s)
{
    if (n) vocab_ranges_kernel<<<grid_for(n, 256, n_sm), 256, 0, s>>>(key_off, n, rng);
    return cudaGetLastError();
}

// which = 0: rank[0..n] (exclusive, in place); 1: key_off[n_keys .. n_keys + n_new] (exclusive, in place, from
// key_bytes); 2: wp_off[0..n] (exclusive, in place).  tmp == nullptr: *tmp_bytes = the temporary storage the scan needs.
cudaError_t vocab_scan(int which, void *tmp, size_t *tmp_bytes, const VocabParams &p, long long n_new, long long key_bytes,
                       cudaStream_t s)
{
    if (which == 0) return cub::DeviceScan::ExclusiveSum(tmp, *tmp_bytes, p.rank, p.rank, p.n + 1, s);
    if (which == 2) return cub::DeviceScan::ExclusiveSum(tmp, *tmp_bytes, p.wp_off, p.wp_off, p.n + 1, s);
    return cub::DeviceScan::ExclusiveScan(tmp, *tmp_bytes, p.key_off + p.n_keys, p.key_off + p.n_keys, cuda::std::plus<long long>(), key_bytes,
                                          n_new + 1, s);
}

}  // namespace latok
