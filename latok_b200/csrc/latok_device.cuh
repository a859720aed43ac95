// latok_device.cuh -- device helpers shared by the kernels (latok_tok5.cuh: tokenize; latok_kernels.cu: parse matrix;
// latok_tokbytes.cu: token byte ranges): PTX wrappers, Unicode class look-up, the context features, the scalar rule
// evaluation used on rare paths, the look-ahead walk and the decoupled look-back.
#pragma once
#include "latok_internal.h"
#include "latok_bits.h"

namespace latok {

constexpr int NEG = -(1 << 28);           // "-infinity" of the (max,+) backlog functions
constexpr unsigned SPIN_LIMIT = 1u << 23; // watchdog for look-back spins

// ---- small helpers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mask_lt(int k) { return __funnelshift_lc(0xFFFFFFFFu, 0u, (unsigned)max(k, 0)); }  // low k bits (k clamped to 0..32)
__device__ __forceinline__ uint32_t mask_lt_nn(int k) { return __funnelshift_lc(0xFFFFFFFFu, 0u, (unsigned)k); }       // same, k known to be >= 0
// bits of a thread's 32-character word that fall inside the character range [lo, hi)
__device__ __forceinline__ uint32_t range_mask(int base, int lo, int hi)
{
    return mask_lt(hi - base) & ~mask_lt(lo - base);
}

struct Fn { int u, v; };  // x -> max(x + u, v)
__device__ __forceinline__ Fn fn_id() { return Fn{0, NEG}; }
__device__ __forceinline__ Fn fn_compose(Fn f, Fn g)  // g after f
{
    return Fn{max(f.u + g.u, NEG), max(max(f.v + g.u, g.v), NEG)};
}
__device__ __forceinline__ int fn_apply(Fn f, int x) { return max(x + f.u, f.v); }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void *bar, uint32_t phase)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred P1;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, P1;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase) : "memory");
    return ok != 0u;
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, void *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ unsigned ld_volatile_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_volatile_u32(unsigned *p, unsigned v)
{
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- Unicode class lookup (replaces gettyperecord, latok.c:15-29, + the tests of latok.c:87-98) ----
struct Tables {
    const uint16_t *ascii_feat;
    const uint16_t *class_feat;
    const latok_stage1_t *stage1;
    const uint8_t *stage2;
    uint32_t low_limit, high_first, high_last, high_feat;
};

__device__ __forceinline__ uint32_t class_of_cp(uint32_t cp, const Tables &t)
{
    if (cp < 0x80u) return t.ascii_feat[cp];
    if (cp < t.low_limit) {
        uint32_t blk = t.stage1[cp >> 7];
        uint32_t b = t.stage2[blk * 64u + ((cp & 127u) >> 1)];
        return t.class_feat[(cp & 1u) ? (b >> 4) : (b & 15u)];
    }
    return (cp >= t.high_first && cp <= t.high_last) ? t.high_feat : 0u;
}

// p points at a character's first byte; up to 3 following bytes are read unconditionally
template <class BytePtr>
__device__ __forceinline__ uint32_t classify_at(BytePtr p, const Tables &t)
{
    uint32_t b0 = p[0];
    if (b0 < 0x80u) return t.ascii_feat[b0];
    if (b0 < 0xC0u || b0 >= 0xF8u) return 0u;  // stray continuation / invalid lead: no features
    uint32_t cp;
    if (b0 < 0xE0u) cp = ((b0 & 0x1Fu) << 6) | (p[1] & 0x3Fu);
    else if (b0 < 0xF0u) cp = ((b0 & 0x0Fu) << 12) | ((p[1] & 0x3Fu) << 6) | (p[2] & 0x3Fu);
    else cp = ((b0 & 0x07u) << 18) | ((p[1] & 0x3Fu) << 12) | ((p[2] & 0x3Fu) << 6) | (p[3] & 0x3Fu);
    return class_of_cp(cp, t);
}

// ---- context features (latok.c:68-73, 99-134) ------------------------------------------------------
// pw / nw / aw: words of the previous / next / after-next character (only base bits are used);
// F / L: this character starts / ends its string; L2: the next character ends the string.
__device__ __forceinline__ uint32_t make_word(uint32_t pw, uint32_t w, uint32_t nw, uint32_t aw, bool F, bool L, bool L2)
{
    pw = F ? 0x20u : pw;                 // start of string behaves as a space (latok.c:69-73,114-117)
    nw = L ? 0x20u : nw;                 // end of string behaves as a space   (latok.c:122-130)
    aw = (L || L2) ? 0u : aw;            // latok.c:131-134
    uint32_t x = w & 0xFFFu;
    x |= ((pw >> 0) & 1u) << 12;         // PREV_ALPHA
    x |= ((nw >> 0) & 1u) << 13;         // NEXT_ALPHA
    x |= ((pw >> 1) & 1u) << 14;         // PREV_ALPHA_NUM
    x |= ((nw >> 1) & 1u) << 15;         // NEXT_ALPHA_NUM
    x |= ((pw >> 3) & 1u) << 16;         // PREV_LOWER
    x |= ((nw >> 3) & 1u) << 17;         // NEXT_LOWER
    x |= ((pw >> 5) & 1u) << 18;         // PREV_SPACE
    x |= ((nw >> 5) & 1u) << 19;         // NEXT_SPACE
    x |= ((pw >> 6) & 1u) << 20;         // PREV_SYMBOL
    x |= ((nw >> 8) & 1u) << 21;         // NEXT_AT
    x |= ((nw >> 10) & 1u) << 22;        // NEXT_SLASH
    x |= ((aw >> 0) & 1u) << 23;         // AFTER_NEXT_ALPHA
    x |= ((aw >> 10) & 1u) << 24;        // AFTER_NEXT_SLASH
    return x;
}

// ---- rule evaluation (combine_matrix_rows 2-D, latok.c:318-341) -------------------------------------
__device__ __forceinline__ void eval_rules(const RuleSet &c_rules, uint32_t w, uint32_t &cnt, bool &mark, uint32_t &sym)
{
    if (c_rules.is_default) {
        // C_SPLIT: SPACE + SYMBOL + PREV_SYMBOL + UPPER*NEXT_LOWER + UPPER*PREV_LOWER (default_tokenizer.py:49-55)
        uint32_t upper = (w >> 4) & 1u;
        cnt = ((w >> 5) & 1u) + ((w >> 6) & 1u) + ((w >> 20) & 1u) + (upper & (w >> 17)) + (upper & (w >> 16));
        // C_MASK (default_tokenizer.py:80-91)
        const uint32_t M0 = (1u << 7) | (1u << 18) | (1u << 13);
        const uint32_t M1 = (1u << 11) | (1u << 18) | (1u << 21) | (1u << 23);
        const uint32_t M2 = (1u << 8) | (1u << 14) | (1u << 15);
        const uint32_t M3 = (1u << 9) | (1u << 22) | (1u << 24) | (1u << 12);
        mark = ((w & M0) == M0) | ((w & M1) == M1) | ((w & M2) == M2) | ((w & M3) == M3);
        // C_SYM: SYMBOL*NEXT_SPACE (default_tokenizer.py:100-102)
        sym = ((w >> 6) & (w >> 19)) & 1u;
    } else {
        cnt = 0; sym = 0; uint32_t mk = 0;
        for (int i = 0; i < c_rules.n_split; ++i) cnt += ((w & c_rules.split[i]) == c_rules.split[i]);
        for (int i = 0; i < c_rules.n_mask; ++i) mk += ((w & c_rules.mask[i]) == c_rules.mask[i]);
        for (int i = 0; i < c_rules.n_sym; ++i) sym += ((w & c_rules.sym[i]) == c_rules.sym[i]);
        mark = mk != 0;
    }
}

// 4 feature bits -> 4 byte counters (bit k -> byte k)
__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

// ---- look-ahead walk (rare): the whitespace chunk open at the end of a tile did not close inside
// the right halo.  Warp 0 scans forward from global byte `pos0` until the chunk closes (a SPACE
// character or the end of the string) and reports whether a mark occurs up to and including the
// closing character.  Exact but slow; it exists so that arbitrarily long space-free runs stay
// bit-exact (latok.c:218-244 has unbounded reach).
static __device__ bool walk_ahead(const Params &p, const Tables &t, long long pos0, int lane)
{
    const uint8_t *in = p.in;
    // end of the string that contains pos0: first offset > pos0 (32 probes per round)
    long long e;
    {
        long long lo = 0, hi = p.n_strings;              // the answer is in [lo, hi]; offsets[n_strings] = n_bytes > pos0
        while (lo < hi) {
            const long long step = (hi - lo + 31) / 32;
            const long long c = lo + step * lane;
            const bool gt = c >= hi || p.offsets[c] > pos0;       // monotone over the lanes
            const unsigned b = __ballot_sync(0xFFFFFFFFu, gt);
            if (b == 0u) lo = lo + 31 * step + 1;
            else {
                const int f = __ffs(b) - 1;
                const long long nh = lo + step * f;
                if (f > 0) lo = lo + step * (f - 1) + 1;
                hi = nh < hi ? nh : hi;
            }
        }
        e = p.offsets[lo];
    }
    struct G { const uint8_t *in; long long q, n; __device__ uint32_t operator[](int k) const { long long a = q + k; return a < n ? (uint32_t)in[a] : 0u; } };
    // the character in front of pos0 (we are strictly inside the string, so it exists)
    uint32_t prev_w;
    {
        long long pp = pos0 - 1;
        for (int k = 0; k < 8 && pp > 0 && (in[pp] & 0xC0u) == 0x80u; ++k) --pp;
        prev_w = classify_at(G{in, pp, p.n_bytes}, t);
    }
    // 32 bytes per trip, one byte per lane; the rules are evaluated for the characters that begin in the first ZONE
    // bytes (their next and after-next characters begin inside the 32 bytes), then the window moves on by ZONE
    constexpr int ZONE = 24, AHEAD = 4;
    bool any = false;
    for (long long q0 = pos0; q0 < e; q0 += AHEAD * ZONE) {
      // the bytes of AHEAD windows are fetched together (the walk runs into text nobody has touched yet: DRAM latency)
      uint32_t bytes[AHEAD];
#pragma unroll
      for (int g = 0; g < AHEAD; ++g) {
          const long long pos = q0 + g * ZONE + lane;
          bytes[g] = pos < e ? (uint32_t)in[pos] : 0x80u;
      }
#pragma unroll
      for (int g = 0; g < AHEAD; ++g) {
        const long long q = q0 + g * ZONE;
        if (q >= e) break;
        const long long pos = q + lane;
        const bool inb = pos < e;
        const uint32_t byte = bytes[g];
        const bool lead = inb && (byte & 0xC0u) != 0x80u;
        const unsigned leads = __ballot_sync(0xFFFFFFFFu, lead);
        uint32_t w = 0;
        if (lead) w = byte < 0x80u ? (uint32_t)t.ascii_feat[byte] : classify_at(G{in, pos, p.n_bytes}, t);
        const unsigned above = lane == 31 ? 0u : (leads & (0xFFFFFFFFu << (lane + 1)));
        const unsigned above2 = above & (above - 1u);
        const unsigned below = leads & ((1u << lane) - 1u);
        const uint32_t nw = __shfl_sync(0xFFFFFFFFu, w, above ? __ffs(above) - 1 : 0);
        const uint32_t aw = __shfl_sync(0xFFFFFFFFu, w, above2 ? __ffs(above2) - 1 : 0);
        uint32_t pw = __shfl_sync(0xFFFFFFFFu, w, below ? 31 - __clz(below) : 0);
        if (!below) pw = prev_w;
        const bool has_next = above != 0u, has_an = above2 != 0u;
        bool closer = false, mk = false;
        const bool ev = lead && lane < ZONE;
        if (ev) {
            const uint32_t full = make_word(pw, w, nw, aw, false, !has_next, !has_an);
            uint32_t cnt, sy;
            eval_rules(p.rules, full, cnt, mk, sy);
            closer = ((full >> 5) & 1u) || !has_next;
        }
        const unsigned bc = __ballot_sync(0xFFFFFFFFu, ev && closer), bm = __ballot_sync(0xFFFFFFFFu, ev && mk);
        if (bc) {
            const int first = __ffs(bc) - 1;
            return any || (bm & (first == 31 ? 0xFFFFFFFFu : ((2u << first) - 1u))) != 0u;
        }
        any = any || bm != 0u;
        if (any) return true;
        const unsigned zone = leads & ((1u << ZONE) - 1u);
        if (zone) prev_w = __shfl_sync(0xFFFFFFFFu, w, 31 - __clz(zone));
      }
    }
    return any;
}

// =====================================================================================================
// Decoupled look-back (single chain, 16-byte aggregate records, LB_WINDOW predecessors per step)
// =====================================================================================================
constexpr int LB_PER_LANE = 2;
constexpr int LB_WINDOW = 32 * LB_PER_LANE;

__device__ __forceinline__ uint4 ld_rec(const void *p)
{
    uint4 r;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_rec(void *p, uint4 v)
{
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

struct Prefix { unsigned long long G, base, K; int x; };

// spin until tile `idx` has published at least `min_state` for this launch; returns the record
__device__ __forceinline__ uint4 wait_rec(const AggRec *agg, long long idx, unsigned epoch, unsigned min_state, Result *result, bool &ok)
{
    uint4 r;
    unsigned spins = 0;
    for (;;) {
        r = ld_rec(agg + idx);
        if ((r.x >> 2) == epoch && (r.x & 3u) >= min_state) break;
        if (++spins > SPIN_LIMIT || (((spins & 1023u) == 0u) && ld_volatile_u32(&result->abort_flag))) {
            atomicOr(&result->error, 1u);
            st_volatile_u32(&result->abort_flag, 1u);
            ok = false;
            break;
        }
    }
    return r;
}

// Exclusive prefix of `tile` (warp 0, all lanes).  Walks back LB_WINDOW tiles at a time until it meets an
// inclusive prefix.  An aggregate is only valid for a tile that no block-mask backlog enters, i.e. when the
// inclusive prefix it is chained to carries no backlog and every aggregate between them leaves none
// (backlog-out for backlog-in 0 is stored in the record).  If that does not hold (rare: a whitespace chunk
// with several marks, or a chunk longer than the halo) the walk waits for the inclusive prefix of the tile
// right after the offending one -- that tile recomputes with its real backlog -- and starts over.
static __device__ Prefix lookback(long long tile, const Params &p, int lane)
{
    Prefix out;
    out.G = 0; out.base = 0; out.K = 0; out.x = 0;
    if (tile == 0) return out;
    for (int restart = 0;; ++restart) {
        unsigned long long sum_n = 0, sum_k = 0;     // characters / tokens of the consumed aggregates
        unsigned long long lf_part = 0; bool lf_found = false;
        long long viol = -1;                         // newest tile whose successor's aggregate must not be used
        int x_in = 0; bool x_set = false;
        bool ok = true, done = false;
        for (long long newest = tile - 1; !done; newest -= LB_WINDOW) {
            // lane l covers tiles first .. first + LB_PER_LANE - 1 (older lanes = older tiles)
            const long long first = newest - (long long)(31 - lane) * LB_PER_LANE - (LB_PER_LANE - 1);
            int rj = -1;                              // newest inclusive element of this lane
            unsigned long long rG = 0, rB = 0, rK = 0; int rx = 0;
            unsigned ln = 0, lk = 0, llf = 0; bool lhas = false; long long lviol = -1; int lastv = 0;
#ifdef LATOK_PROFILE
            long long _lt0 = clock64();
#endif
            // all records of this lane in flight at once; re-poll only the ones not yet published
            uint4 rec[LB_PER_LANE];
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) { rec[j] = make_uint4(0, 0, 0, 0); if (first + j >= 0) rec[j] = ld_rec(p.agg + (first + j)); }
            {
                unsigned spins = 0;
                for (;;) {
                    bool pending = false;
#pragma unroll
                    for (int j = 0; j < LB_PER_LANE; ++j)
                        if (first + j >= 0 && !((rec[j].x >> 2) == p.epoch && (rec[j].x & 3u) != 0u)) { rec[j] = ld_rec(p.agg + (first + j)); pending = true; }
                    if (!pending) break;
#ifdef LATOK_PROFILE
                    if (lane == 31) atomicAdd(&p.result->prof[14], 1ull);
#endif
                    if (++spins > SPIN_LIMIT || (((spins & 1023u) == 0u) && ld_volatile_u32(&p.result->abort_flag))) {
                        atomicOr(&p.result->error, 1u);
                        st_volatile_u32(&p.result->abort_flag, 1u);
                        ok = false;
                        break;
                    }
                }
            }
#ifdef LATOK_PROFILE
            if (lane == 31) { long long _t = clock64(); atomicAdd(&p.result->prof[6], (unsigned long long)(_t - _lt0)); _lt0 = _t; }
#endif
            // the newest inclusive record of this lane: fetch its prefix
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) if (first + j >= 0 && (rec[j].x & 3u) == 2u) rj = j;
            if (rj >= 0) {
                __threadfence();
                const IncRec *ir = p.inc + (first + rj);
                const uint4 a = ld_rec(ir), b = ld_rec(reinterpret_cast<const uint4 *>(ir) + 1);
                rG = a.x | ((unsigned long long)a.y << 32); rB = a.z | ((unsigned long long)a.w << 32);
                rK = b.x | ((unsigned long long)b.y << 32); rx = (int)b.z;
            }
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) {
                const long long idx = first + j;
                if (idx < -1) continue;
                if (idx == -1) { if (rj < 0) { rj = j; rG = rB = rK = 0; rx = 0; } continue; }
                if (j <= rj) continue;                          // superseded by (or is) the inclusive record
                const uint4 r = rec[j];
                const unsigned n = r.y & 0xFFFFu, lf1 = r.y >> 16, k = r.z & 0xFFFFu; const int v = (int)(r.z >> 16);
                if (lf1) { llf = ln + (lf1 - 1u); lhas = true; }
                ln += n; lk += k;
                if (v != 0 && idx != tile - 1) lviol = idx;      // its successor needs a real backlog
                if (idx == tile - 1) lastv = v;
            }
            const unsigned has_reset = __ballot_sync(0xFFFFFFFFu, rj >= 0);
            const int Lr = has_reset ? 31 - __clz(has_reset) : -1;
#ifdef LATOK_PROFILE
            if (lane == 0) { atomicAdd(&p.result->prof[13], 1ull); if (Lr >= 0) atomicAdd(&p.result->prof[8], (unsigned long long)((31 - Lr) * LB_PER_LANE)); }
#endif
            const bool contrib = lane >= Lr;          // lanes older than the newest inclusive element are superseded
            // characters / tokens
            const unsigned wn = __reduce_add_sync(0xFFFFFFFFu, contrib ? ln : 0u), wk = __reduce_add_sync(0xFFFFFFFFu, contrib ? lk : 0u);
            // newest string start among the consumed aggregates of this window
            const unsigned hasm = __ballot_sync(0xFFFFFFFFu, contrib && lhas);
            if (!lf_found && hasm) {
                const int H = 31 - __clz(hasm);
                const unsigned older = __reduce_add_sync(0xFFFFFFFFu, (contrib && lane < H) ? ln : 0u);
                lf_part = (unsigned long long)older + __shfl_sync(0xFFFFFFFFu, llf, H);
                lf_found = true;
            } else if (lf_found) lf_part += wn;       // this whole window lies before the string start found earlier
            sum_n += wn; sum_k += wk;
            // newest offending tile of this window (64-bit max through two 32-bit reductions on the offset from `newest`)
            const int voff = (contrib && lviol >= 0) ? (int)(newest - lviol) : 0x7FFFFFFF;   // smaller offset = newer
            const int vmin = __reduce_min_sync(0xFFFFFFFFu, voff);
            if (vmin != 0x7FFFFFFF && viol < 0) viol = newest - vmin;
            if (!x_set) { x_in = __shfl_sync(0xFFFFFFFFu, lastv, 31); x_set = true; }
            if (!__all_sync(0xFFFFFFFFu, ok)) { out.x = 0; return out; }    // watchdog tripped: error flag is set
#ifdef LATOK_PROFILE
            if (lane == 31) { long long _t = clock64(); atomicAdd(&p.result->prof[7], (unsigned long long)(_t - _lt0)); }
#endif
            if (Lr >= 0) {
                const unsigned long long G0 = __shfl_sync(0xFFFFFFFFu, rG, Lr), B0 = __shfl_sync(0xFFFFFFFFu, rB, Lr);
                const unsigned long long K0 = __shfl_sync(0xFFFFFFFFu, rK, Lr);
                const int x0 = __shfl_sync(0xFFFFFFFFu, rx, Lr);
                const bool consumed_any = sum_n != 0 || sum_k != 0 || __shfl_sync(0xFFFFFFFFu, rj, Lr) != LB_PER_LANE - 1 || Lr != 31 || newest != tile - 1;
                if (x0 != 0 && consumed_any && viol < 0) {
                    // the inclusive prefix carries a backlog into the first consumed aggregate
                    const long long ridx = newest - (long long)(31 - Lr) * LB_PER_LANE - (LB_PER_LANE - 1) + __shfl_sync(0xFFFFFFFFu, rj, Lr);
                    viol = ridx;
                }
                out.G = G0 + sum_n; out.K = K0 + sum_k; out.base = lf_found ? G0 + lf_part : B0;
                out.x = consumed_any ? x_in : x0;
                done = true;
            }
        }
        if (viol < 0) return out;
        // wait for the tile after the offending one to publish its exact inclusive prefix, then walk again
        bool ok2 = true;
        wait_rec(p.agg, viol + 1, p.epoch, 2u, p.result, ok2);
        if (lane == 0) atomicAdd(&p.result->prof[15], 1ull);
        if (!ok2) return out;
    }
}

__device__ __forceinline__ void nb_sync(int id, int cnt) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(cnt) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int cnt) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(cnt) : "memory"); }

// Feature word of the multi-byte character whose four bytes (lead byte >= 0xC0 in the low byte, then up to three
// continuation bytes; whatever follows a shorter character is ignored) are `v` -- the same decode and look-up as
// classify_at, without the length branches, so that lanes holding 2-, 3- and 4-byte characters
// stay converged and two characters can be in flight at once.
__device__ __forceinline__ uint32_t mb_features(uint32_t v, const Tables &t)
{
    const int L = __clz((int)~(v << 24)) - 1;                  // continuation bytes: 1..3 (>= 4: invalid lead byte)
    const uint32_t c1 = (v >> 8) & 0x3Fu, c2 = (v >> 16) & 0x3Fu, c3 = (v >> 24) & 0x3Fu;
    const uint32_t cp4 = ((v & (0x3Fu >> L)) << 18) | (c1 << 12) | (c2 << 6) | c3;
    const uint32_t cp = cp4 >> (6 * (3 - L) & 31);
    const uint32_t cl = min(cp, t.low_limit - 1u);
    const uint32_t blk = t.stage1[cl >> 7];
    const uint32_t b = t.stage2[blk * 64u + ((cl & 127u) >> 1)];
    uint32_t fw = t.class_feat[(b >> ((cl & 1u) * 4u)) & 15u];
    // the three rare cases behind one test: beyond the two-stage table, an over-long form of an ASCII character
    // (cp - 0x80 wraps), an invalid lead byte 0xF8..0xFF
    if (__builtin_expect(cp - 0x80u >= t.low_limit - 0x80u || L > 3, 0)) {
        if (cp >= t.low_limit) fw = (cp >= t.high_first && cp <= t.high_last) ? t.high_feat : 0u;
        if (cp < 0x80u) fw = t.ascii_feat[cp];
        if (L > 3) fw = 0u;
    }
    return fw;
}

// Backlog through one thread's characters (latok.c:218-244 in scan form): x += 1 at a mark, x = 0 at a
// string start, a closer (space / end of string) is "hot" if x >= 1 when it is reached, a space then takes
// one off and the end of a string clears it.  Driven by the (rare) marks; closers are only visited while x > 0.
__device__ __forceinline__ int eval_backlog(int x, uint32_t Mm, uint32_t FmA, uint32_t S, uint32_t Lm, uint32_t &HOT)
{
    HOT = 0;
    const uint32_t CL = S | Lm;
    uint32_t remP = 0xFFFFFFFFu, remC = 0xFFFFFFFFu;   // positions still ahead for raising events / closers
    for (;;) {
        if (x == 0) {
            const uint32_t m = Mm & remP;
            if (!m) break;
            const uint32_t b = m & (0u - m);
            x = 1;
            remC = ~(b - 1u);               // closers at or after the mark
            remP = remC & ~b;               // events strictly after it
        } else {
            const uint32_t pe = (Mm | FmA) & remP, ce = CL & remC;
            const uint32_t bp = pe & (0u - pe), bc = ce & (0u - ce);
            if (!bp && !bc) break;
            if (bp && (!bc || bp <= bc)) {
                if (FmA & bp) x = 0;
                if (Mm & bp) ++x;
                remC = ~(bp - 1u);
                remP = remC & ~bp;
            } else {
                HOT |= bc;
                if (S & bc) --x;
                if (Lm & bc) x = 0;            // nothing is carried past the end of a string (the next start resets it anyway)
                remC = ~(bc - 1u) & ~bc;
            }
        }
    }
    return x;
}

}  // namespace latok
