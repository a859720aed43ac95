// latok_tok5.cuh -- tokenize kernel v5 (split mask + token spans + CSR offsets) for sm_100a.
//
// Work decomposition
//   range  = what ONE WARP analyses on its own: a 4 KB window of the flat UTF-8 buffer, of which it owns the
//            characters from just after the first chunk closer (space / end of string) found in the first 116
//            bytes up to and including the first closer found in the 116 bytes after byte 3968.  Neighbouring
//            ranges look at the same bytes and agree, so (almost) no block-mask state crosses a range boundary.
//   step   = 1 KB of a range: lane l holds bytes [32l, 32l+32) as bit-planes (32 characters per register).
//   tile   = the NW (9 or 11, see Geometry) consecutive ranges of one CTA; one decoupled look-back record per tile
//            (service warp).
//
// Per range (compute warp, no CTA-wide barrier anywhere on this path):
//   pass A  forward over the steps, software-pipelined (base planes of step j+1, then context + rules of step j):
//           byte -> bit-plane transpose, bit-sliced ASCII classification, class-table patch for multi-byte
//           characters, squeeze to character space, prev/next/after-next context (latok.c:68-73,99-134), rule
//           sums (latok.c:318-341), and the block mask's forward half as a carry-propagating add
//           (latok.c:218-244 when no chunk holds two marks; a step that does is evaluated mark by mark)
//   pass C  backward over the steps: blank the chunks whose closer is hot, split values
//           (default_tokenizer.py:121-132), token flags (default_tokenizer.py:148-158), counts
//   -> the service warp sums the ranges of the tile, publishes the aggregate, looks back, hands the prefix down
//   pass D  CSR offsets by one lane per string; then forward over the steps: split bytes and (start,end) pairs staged
//           per step in shared memory and written with aligned 16-byte stores; in the token-feature instantiation the
//           rows of the step's tokens in the order of their ordinals (lane t sums row 32 i + t from the planes of the
//           lane-word the token ended in, fetched by shuffle), staged and written as whole 16-byte chunks.
// Rare paths, one mechanism (resolve()): every range posts, with its counts, how it transforms a block-mask backlog
// (x -> max(x + u, f0): u = marks - closers, f0 = what it leaves when nothing enters), the marks in front of its first
// closer and whether it begins / ends at a chunk closer.  The service warp composes these over the ranges of the tile:
// the backlog that really enters every range (several marks in a chunk, a backlog from the previous tile) and, for a
// range that ends inside a chunk (a space-free run longer than the search windows), whether that chunk's closer will be
// hot (a pending mark, a mark in a later range, or -- past the end of the tile -- the look-ahead walk).  A range whose
// result depends on something it assumed differently is analysed again (the ORDINARY analysis, with the real values) by
// the service warp itself, at once: the warp that owns the range is busy with its next tile by then.
// The warps run one tile ahead of the look-back: analysis of tile k+1, then pass D of tile k, whose state waits in
// place of its input bytes (two window buffers per warp; Parked owns that layout).  What the analysis of a range found
// goes to one RangeRec per (slot, range) in Ctl, which the service warp, the prefix of every warp and pass D read.
// Tickets are taken by the first warp that is ready for the next tile, so ticket order follows start order and
// predecessors publish first.
//
// No tensor cores: nothing here is a dense contraction; the bound is HBM bandwidth.
#pragma once
#include "latok_chain.cuh"

namespace latok {
namespace v5 {

constexpr int STEP = 1024;
constexpr int HALO = 128;                // the last HALO bytes of a range's window are the first of the next range's
constexpr int HLANES = HALO / 32;
constexpr int NMB = 7;                   // feature planes a non-ASCII character can have (ALPHA .. SYMBOL)
constexpr int MARGIN = 12;               // characters starting in the last 12 window bytes lack forward context
constexpr int LPAD = 16;                 // bytes in front of the window (previous character)
constexpr int SSTAGE = 5 * 36 * 4;          // pass D: bit stage (up to 5 value planes, 36 words each)
constexpr int TCAP = 320;                // tokens staged per step; steps with more write their pairs directly
constexpr int TSTAGE = (TCAP + 2) * 8;
constexpr int FLIST = 512;               // token-feature mode: token ends per step that are written in the order of their ordinals
constexpr int FSTAGE = 832;              // ... row stage: up to 15 bytes left of the trip before + 32 * 25 bytes, in 16-byte chunks
enum { BAR_AGG = 1, BAR_PRE = 3 };
static_assert(HALO % 32 == 0, "geometry");
static_assert(TSTAGE >= STEP + 64, "the token stage doubles as the byte stage of partly owned split-mask chunks");
static_assert(TSTAGE >= 1024 + FSTAGE && FSTAGE >= 15 + 32 * NFEAT + 8 && FSTAGE % 16 == 0, "token-feature mode: tails + row stage live in the token stage");

// The kernel exists in two geometries; the host picks one per batch (tokenize5_plan, latok_tok5.cu).  Long strings: 4 KB
// ranges, 9 compute warps per CTA -- fewer range boundaries inside space-free runs.  Short strings: 3 KB ranges, 11
// compute warps per CTA at 80 registers -- more warps in flight, which is what the instruction-bound regular path gains
// from.  Token features run in the long geometry only (the 25 planes per lane want its 96 registers).
template <int RS_, int NW_, bool FEATS_>
struct Geometry {
    static constexpr bool FEATS = FEATS_;    // the token-feature instantiation exists
    static constexpr int NW = NW_;           // compute warps per CTA (warp 0 is the service warp)
    static constexpr int NTH = (NW + 1) * 32;
    static constexpr int RS = RS_;           // steps per range
    static constexpr int WIN = RS * STEP;
    static constexpr int RANGE = WIN - HALO;
    static constexpr int XBYTES = LPAD + WIN + 16;
    static constexpr int CTAS = 2;           // CTAs per SM the default-rules instantiation is compiled for
    static_assert(RANGE % 16 == 0, "geometry");
    static_assert((NW - 1) * RANGE + WIN < 65536, "what a tile owns lies in its NW windows: its sums fit the 16-bit fields of AggRec");
};
using LongGeometry = Geometry<4, 9, true>;
using ShortGeometry = Geometry<3, 11, false>;

// What the analysis of a range posts: the characters it owns [c_lo, c_hi) (range-relative; n_own = c_hi - c_lo), the tokens
// counted in them, its last owned string start (lft, relative to c_lo; -1: none), the block-mask backlog it leaves (v) and --
// for a range that begins inside a chunk -- how it transforms a backlog: x -> max(x + u, v), mb1 marks in front of its
// first closer (resolve()).  One record per (slot, range of the tile); the owner of range i is compute warp i.
struct RangeRec {
    enum : int {
        HAVE = 1,            // the range holds data
        CLOSED = 2,          // it ends at a chunk closer
        LO_FOUND = 4,        // it begins at a chunk closer (else u and mb1 are set)
        HOLDS_CLOSER = 8,    // it owns a chunk closer
        GUESSED_HOT = 16,    // (a range that ends inside a chunk) its first analysis assumed that chunk closed hot
    };
    int c_lo, c_hi, n_own, ntok, lft, v, u, mb1, flags;
};
template <class Geom>
struct Ctl {
    int tile_id[2], tk_cnt[2], tk_flag[2];
    int pad0[4];
    Prefix slot[2];                      // the prefix in front of the tile, handed down by the service warp (x unused)
    RangeRec rec[2][Geom::NW];
    int tokstep[Geom::NW][2][Geom::RS];  // tokens per step
    int nsa[Geom::NW][2][Geom::RS];      // first split after the step (range-relative character index, -1: none)
};

// The state of one lane-word while it waits between the passes:
//   after pass A : CNT[NC] SYM[NY] | S HOT  F packed
//   after pass C : V[NV]   E       | S lead F packed
// Pass C rewrites V, E, lead and packed and leaves S and F as pass A stored them: pass D reads them.  The slot of the hot
// closers takes the lane-word's lead-byte mask: the window's string-start map (bit = byte), whose slot has become that
// mask in pass A, is rebuilt by the analysis of the next window before pass D reads it.
// Default rules: 8 words IN PLACE of the lane-word's 32 input bytes (pass A parks a step after it has read the next one),
// as two 16-byte halves 512 bytes apart inside the step's 1 KB (word w at js*256 + (w >> 2)*128 + ln*4 + (w & 3)), so the
// 128-bit accesses of a quarter warp fall into 32 different banks (a 32-byte lane stride makes them collide in pairs).
// Generic rules: WORDS words in a row, in a buffer of their own (plan()).
template <bool kDefault>
struct Parked {
    static constexpr int NC = kDefault ? 3 : 4;     // split-count planes
    static constexpr int NY = kDefault ? 1 : 4;     // sym-count planes
    static constexpr int NV = kDefault ? 3 : 5;     // split-value planes
    static constexpr int WORDS = kDefault ? 8 : 12;
    static_assert(!kDefault || WORDS * 4 == 32, "the in-place state takes the lane-word's 32 bytes");
    static_assert(NC + NY <= WORDS - 4 && NV + 1 <= WORDS - 4, "layout");
    uint32_t *t;
    __device__ __forceinline__ Parked(uint32_t *base, int js, int ln) : t(kDefault ? base + js * 256 + ln * 4 : base + (js * 32 + ln) * WORDS) {}
    // the words of step js, once read, as scratch: at least 1 KB
    __device__ __forceinline__ static uint16_t *scratch(uint32_t *base, int js) { return reinterpret_cast<uint16_t *>(Parked(base, js, 0).t); }
    __device__ __forceinline__ uint32_t s() const { return w(W_S); }
    __device__ __forceinline__ uint32_t f() const { return w(W_F); }
    __device__ __forceinline__ uint32_t packed() const { return w(W_K); }
    __device__ __forceinline__ uint32_t e() const { return w(W_E); }          // after pass C
    __device__ __forceinline__ uint32_t lead() const { return w(W_H); }       // after pass C

    __device__ __forceinline__ void store_a(const uint32_t (&cnt)[NC], const uint32_t (&sym)[NY], uint32_t S, uint32_t hot, uint32_t F, uint32_t pk) const
    {
        if (kDefault) {
            *reinterpret_cast<uint4 *>(t) = make_uint4(cnt[0], cnt[1], cnt[2], sym[0]);
            *reinterpret_cast<uint4 *>(t + 128) = make_uint4(S, hot, F, pk);
        } else {
#pragma unroll
            for (int q = 0; q < NC; ++q) t[q] = cnt[q];
#pragma unroll
            for (int q = 0; q < NY; ++q) t[NC + q] = sym[q];
            t[W_S] = S; t[W_H] = hot; t[W_F] = F; t[W_K] = pk;
        }
    }
    __device__ __forceinline__ void load_a(uint32_t (&cnt)[NC], uint32_t (&sym)[NY], uint32_t &S, uint32_t &hot, uint32_t &F, uint32_t &pk) const
    {
        if (kDefault) {
            const uint4 a = *reinterpret_cast<const uint4 *>(t), b = *reinterpret_cast<const uint4 *>(t + 128);
            cnt[0] = a.x; cnt[1] = a.y; cnt[2] = a.z; sym[0] = a.w; S = b.x; hot = b.y; F = b.z; pk = b.w;
        } else {
#pragma unroll
            for (int q = 0; q < NC; ++q) cnt[q] = t[q];
#pragma unroll
            for (int q = 0; q < NY; ++q) sym[q] = t[NC + q];
            S = t[W_S]; hot = t[W_H]; F = t[W_F]; pk = t[W_K];
        }
    }
    __device__ __forceinline__ void store_c(const uint32_t (&v)[NV], uint32_t E, uint32_t lead, uint32_t pk) const
    {
        if (kDefault) *reinterpret_cast<uint4 *>(t) = make_uint4(v[0], v[1], v[2], E);
        else {
#pragma unroll
            for (int q = 0; q < NV; ++q) t[q] = v[q];
            t[W_E] = E;
        }
        w(W_H) = lead; w(W_K) = pk;
    }
    __device__ __forceinline__ void load_c(uint32_t (&v)[NV], uint32_t &E, uint32_t &S, uint32_t &F, uint32_t &pk) const
    {
        if (kDefault) {
            const uint4 a = *reinterpret_cast<const uint4 *>(t), b = *reinterpret_cast<const uint4 *>(t + 128);
            v[0] = a.x; v[1] = a.y; v[2] = a.z; E = a.w; S = b.x; F = b.z; pk = b.w;
        } else {
#pragma unroll
            for (int q = 0; q < NV; ++q) v[q] = t[q];
            E = t[W_E]; S = t[W_S]; F = t[W_F]; pk = t[W_K];
        }
    }

  private:
    static constexpr int W_E = NV, W_S = WORDS - 4, W_H = WORDS - 3, W_F = WORDS - 2, W_K = WORDS - 1;
    __device__ __forceinline__ uint32_t &w(int i) const { return t[kDefault && i >= 4 ? 124 + i : i]; }
};
static_assert(FLIST * 2 <= STEP, "token-feature mode: the token-end list lives in a step's parked state");

struct Plan {
    int tables, ctl, mbar, sbm0, warp0, x[2], sst, tst, sbm, temp[2], per_warp, total;
};
template <class Geom>
__host__ __device__ inline Plan plan(const TableLayout &tl, bool is_default)
{
    Plan s; int o = 0;
    auto take = [&](int bytes) { int r = o; o += (bytes + 15) & ~15; return r; };
    s.tables = take(tl.stage2 - tl.lutv);    // split-value LUT, ASCII / class feature words, stage 1; stage 2 (16 KB) stays in global memory (L1)
    s.ctl = take((int)sizeof(Ctl<Geom>));
    s.mbar = take(8 * 2 * Geom::NW);
    s.sbm0 = take(Geom::RS * 32 * 4);           // string map of a window the service warp analyses again
    s.warp0 = o;
    s.x[0] = take(Geom::XBYTES); s.x[1] = take(Geom::XBYTES);
    s.sst = take(SSTAGE);
    s.tst = take(TSTAGE);
    s.sbm = take(Geom::RS * 32 * 4);
    for (int b = 0; b < 2; ++b)                 // parked state (default rules: in place of the window's bytes)
        s.temp[b] = is_default ? s.x[b] + LPAD : take(Geom::RS * 32 * Parked<false>::WORDS * 4);
    s.per_warp = o - s.warp0;
    s.total = s.warp0 + Geom::NW * s.per_warp;
    return s;
}

#ifdef LATOK_PROFILE
#define PROF5(i) do { if (lane == 0) { long long _t = clock64(); atomicAdd(&p.result->clocks.phase[i], (unsigned long long)(_t - _prof_t)); _prof_t = _t; } } while (0)
#else
#define PROF5(i) do { } while (0)
#endif

#define LIKELY(x) (__builtin_expect(!!(x), 1))
#define UNLIKELY(x) (__builtin_expect(!!(x), 0))
constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int CINF = 0x3FFFFFFF;

// packed per-lane-word scalars: chars n (6 bits) | first char index c0 (13) << 6 | tokens before (11) << 19 | prev-is-space << 30
__device__ __forceinline__ uint32_t pack_ncp(int n, int c0, int ps) { return (uint32_t)n | ((uint32_t)c0 << 6) | ((uint32_t)ps << 30); }
__device__ __forceinline__ int pk_n(uint32_t k) { return (int)(k & 63u); }
__device__ __forceinline__ int pk_c0(uint32_t k) { return (int)((k >> 6) & 8191u); }
__device__ __forceinline__ int pk_tp(uint32_t k) { return (int)((k >> 19) & 2047u); }
__device__ __forceinline__ uint32_t pk_ps(uint32_t k) { return (k >> 30) & 1u; }

__device__ __forceinline__ int bfind32(uint32_t x) { int r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x)); return r; }   // index of the highest set bit (-1: none)
__device__ __forceinline__ int ld_vs32(const int *p) { int v; asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p))); return v; }
__device__ __forceinline__ void st_vs32(int *p, int v) { asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory"); }

// What ranges [0, end) of a tile add to the prefix, from their records (warp-wide, end <= NW): the service warp sums the
// whole tile, a compute warp the ranges in front of its own
template <int NW>
__device__ __forceinline__ TileSum sum_ranges(const RangeRec (&rec)[NW], int end, int lane)
{
    const RangeRec a = rec[lane < NW ? lane : 0];
    const bool in = lane < end;
    const int mn = in ? a.n_own : 0;
    int pn = mn;                                   // inclusive prefix of characters over the ranges
#pragma unroll
    for (int d = 1; d < NW; d <<= 1) { const int t = __shfl_up_sync(FULL, pn, d); if (lane >= d) pn += t; }
    const unsigned hl = __ballot_sync(FULL, in && a.lft >= 0);
    const int lv = __shfl_sync(FULL, pn - mn + a.lft, hl ? 31 - __clz(hl) : 0);
    return TileSum{__reduce_add_sync(FULL, mn), __reduce_add_sync(FULL, in ? a.ntok : 0), hl ? lv : -1};
}

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
            mk = rule_mark(p.rules, full);
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

template <class Geom, bool kDefault, bool kFeats>
__global__ void __launch_bounds__(Geom::NTH, kDefault ? Geom::CTAS : 1) tokenize5_kernel(const Params p)
{
    constexpr int NW = Geom::NW, NTH = Geom::NTH, RS = Geom::RS, WIN = Geom::WIN, RANGE = Geom::RANGE, XBYTES = Geom::XBYTES;
    using PS = Parked<kDefault>;
    constexpr int NC = PS::NC, NY = PS::NY, NV = PS::NV;
    extern __shared__ __align__(128) unsigned char smem[];
    const Plan sp = plan<Geom>(p.tl, kDefault);
    uint8_t *tableS = smem + sp.tables;
    Ctl<Geom> &ctl = *reinterpret_cast<Ctl<Geom> *>(smem + sp.ctl);
    unsigned long long *mbar = reinterpret_cast<unsigned long long *>(smem + sp.mbar);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cw = warp - 1;                  // compute warp number (warp 0, the CTA's oldest warp, is the service warp)

    if (ld_volatile_u32(&p.result->error) & 2u) return;  // offsets failed validation in tile_index_kernel

    // ---- one-time per CTA: tables into shared memory, barriers, flags
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.table_blob + p.tl.lutv);
        const int n16 = (p.tl.stage2 - p.tl.lutv) / 16;
        for (int i = threadIdx.x; i < n16; i += NTH) reinterpret_cast<uint4 *>(tableS)[i] = __ldg(src + i);
        if (threadIdx.x == 0) {
            for (int w = 0; w < 2 * NW; ++w) mbar_init(mbar + w, 1);
            for (int b = 0; b < 2; ++b) { ctl.tile_id[b] = 0; ctl.tk_cnt[b] = 0; ctl.tk_flag[b] = 0; }
        }
    }
    __syncthreads();
    const bool want_spans = (p.what & 2u) != 0u, want_splits = (p.what & 1u) != 0u;
    const int ntiles_i = (int)p.ntiles;

    Tables tb;
    tb.ascii_feat = reinterpret_cast<const uint16_t *>(tableS + (p.tl.ascii_feat - p.tl.lutv));
    tb.class_feat = reinterpret_cast<const uint16_t *>(tableS + (p.tl.class_feat - p.tl.lutv));
    tb.stage1 = reinterpret_cast<const latok_stage1_t *>(tableS + (p.tl.stage1 - p.tl.lutv));
    tb.stage2 = p.table_blob + p.tl.stage2;
    tb.low_limit = p.tl.low_limit; tb.high_first = p.tl.high_first; tb.high_last = p.tl.high_last; tb.high_feat = p.tl.high_feat;

    // =================================================================================================
    // compute warps
    // =================================================================================================
    // the buffers of compute warp `w`: a compute warp works on its own; the service warp, when it repeats the analysis of a
    // range (resolve()), on those of the warp that owns the range
    auto wbase_of = [&](int w) -> unsigned char * { return smem + sp.warp0 + w * sp.per_warp; };
    unsigned char *wbase = smem + sp.warp0 + (cw < 0 ? 0 : cw) * sp.per_warp;      // (own buffers: output path of the compute warps)
    uint8_t *sst = wbase + (sp.sst - sp.warp0);
    int2 *tst = reinterpret_cast<int2 *>(wbase + (sp.tst - sp.warp0));
    auto Xof = [&](int w, int b) -> uint8_t * { return wbase_of(w) + (sp.x[b] - sp.warp0); };
    // string-start map / lead masks of the window under analysis (the service warp has a scratch of its own: the owner
    // of the range is busy with its next tile)
    auto sbm_of = [&](int w) -> uint32_t * {
        return reinterpret_cast<uint32_t *>(warp == 0 ? smem + sp.sbm0 : wbase_of(w) + (sp.sbm - sp.warp0));
    };
    auto tempof = [&](int w, int b) -> uint32_t * { return reinterpret_cast<uint32_t *>(wbase_of(w) + (sp.temp[b] - sp.warp0)); };
    const uint32_t *lutv = reinterpret_cast<const uint32_t *>(tableS);
#ifdef LATOK_PROFILE
    long long _prof_t = clock64();
#endif
    if (warp != 0) for (int i = lane; i < 5 * 36; i += 32) reinterpret_cast<uint32_t *>(sst)[i] = 0;     // bit stage of pass D
    __syncwarp();

    // ---- window load: TMA bulk copy of the 16-byte aligned interior, plain loads for the ragged end
    auto begin_load = [&](long long r, int b) -> bool {
        if (r >= p.nranges) return false;
        uint8_t *X = Xof(cw, b);
        const long long wl = r * (long long)RANGE - LPAD;          // global position of X[0]
        const long long lo = wl < 0 ? 0 : wl;
        long long hi = wl + XBYTES;
        const long long full16 = p.n_bytes & ~15LL;
        if (hi > full16) hi = full16;
        const int tma_bytes = hi > lo ? int(hi - lo) : 0;
        fence_proxy_async();
        __syncwarp();
        if (lane == 0 && tma_bytes > 0) {
            mbar_expect_tx(mbar + 2 * cw + b, (uint32_t)tma_bytes);
            tma_load_1d(X + (lo - wl), p.in + lo, (uint32_t)tma_bytes, mbar + 2 * cw + b);
        }
        const int a_end = int(lo - wl), b_beg = a_end + tma_bytes;
        for (int i = lane; i < a_end; i += 32) X[i] = 0;
        for (int i = b_beg + lane; i < XBYTES; i += 32) {
            const long long g = wl + i;
            X[i] = g < p.n_bytes ? p.in[g] : (uint8_t)0;
        }
        return tma_bytes > 0;
    };
    auto plain_load = [&](long long r, int w, int b) {          // repeated analysis: fetch the window again
        uint8_t *X = Xof(w, b);
        const long long wl = r * (long long)RANGE - LPAD;
        for (int i = lane * 16; i < XBYTES; i += 512) {
            const long long g = wl + i;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (g >= 0 && g + 16 <= p.n_bytes) v = *reinterpret_cast<const uint4 *>(p.in + g);
            else if (g + 16 > 0 && g < p.n_bytes) {
                uint32_t w4[4] = {0, 0, 0, 0};
                for (int q = 0; q < 16; ++q)
                    if (g + q >= 0 && g + q < p.n_bytes) w4[q >> 2] |= (uint32_t)p.in[g + q] << (8 * (q & 3));
                v = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
            *reinterpret_cast<uint4 *>(X + i) = v;
        }
        __syncwarp();
    };

    // Exact block-mask forward pass over one step (latok.c:218-244 in scan form): every lane-word becomes a backlog
    // transfer function x -> max(x + u, v) (string start = reset, mark = +1, space = one off but not below 0, end of
    // string = reset), a warp scan composes them, then each lane walks its own events once with the backlog that
    // really enters it.  Returns the hot closers; `x` is the backlog entering the step, `out` leaves this lane-word.
    auto lane_fn_scan = [&](uint32_t Mm, uint32_t FmA, uint32_t S, uint32_t Lm) -> Fn {      // inclusive scan over the lanes
        Fn f = fn_id();
        {
            uint32_t evs = Mm | FmA | S | Lm;
            while (evs) {
                const uint32_t b = evs & (0u - evs); evs ^= b;
                if (FmA & b) f = fn_compose(f, Fn{NEG, 0});
                if (Mm & b) f = fn_compose(f, Fn{1, NEG});
                if (S & b) f = fn_compose(f, Fn{-1, 0});
                if (Lm & b) f = fn_compose(f, Fn{NEG, 0});
            }
        }
        Fn inc = f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int ou = __shfl_up_sync(FULL, inc.u, d), ov = __shfl_up_sync(FULL, inc.v, d);
            if (lane >= d) inc = fn_compose(Fn{ou, ov}, inc);
        }
        return inc;
    };
    auto exact_step = [&](int x, uint32_t Mm, uint32_t FmA, uint32_t S, uint32_t Lm, int &out) -> uint32_t {
        const Fn inc = lane_fn_scan(Mm, FmA, S, Lm);
        const int eu = __shfl_up_sync(FULL, inc.u, 1), ev2 = __shfl_up_sync(FULL, inc.v, 1);
        const int xin = lane ? fn_apply(Fn{eu, ev2}, x) : x;
        uint32_t HOT = 0;
        out = xin;
        if (xin != 0 || Mm) out = eval_backlog(xin, Mm, FmA, S, Lm, HOT);
        return HOT;
    };
    // ---- string-start map of a window (bit = byte position), from the offsets of the strings that begin in it.  Needs
    // nothing of the window itself: the compute warps build it while the window is still on its way (the two dependent
    // global loads overlap the TMA copy).
    auto build_map = [&](const long long r, const int w) {
        if (r >= p.nranges) return;
        uint32_t *sbmS = sbm_of(w);
        const long long w0 = r * (long long)RANGE;
#pragma unroll
        for (int j = 0; j < RS; ++j) sbmS[j * 32 + lane] = 0;
        __syncwarp();
        const long long wend = w0 + WIN;
        for (long long s = p.tile_first_str[r] + lane; s <= p.n_strings; s += 32) {
            const long long o = p.offsets[s];
            if (o >= wend) break;
            const int wb = int(o - w0);
            atomicOr(&sbmS[wb >> 5], 1u << (wb & 31));
        }
        __syncwarp();
    };

    // ================================================================================================= analysis
    // Analyses range r in buffer `buf` of compute warp `w` and returns its record.  x_init: block-mask backlog entering the
    // range; far_init: the chunk open at the end of the range (a range that does not end at a chunk closer) will be closed
    // hot.  The first analysis of every range assumes that nothing enters and (far_init = -1) that an open last chunk WILL
    // be closed hot; the service warp orders a repeat with the real values where that changes the result (resolve()).
    auto analyze = [&](const long long r, const int buf, const int w, const int x_init, const int far_init) -> RangeRec {
        const long long w0 = r * (long long)RANGE;
        const bool have = r < p.nranges, last_range = r == p.nranges - 1;
        uint8_t *X = Xof(w, buf);
        uint32_t *tempS = tempof(w, buf);
        uint32_t *sbmS = sbm_of(w);
        int c_lo = 0, c_hi = CINF, n_own = 0, ntok_range = 0, lft = -1, v_out = 0;
        bool closed = true, lo_found = true, guessed_hot = false;
        // backlog transfer summary of the owned characters: marks - closers, a string boundary (= reset), marks in front of
        // the first closer, whether there is a closer at all
        int d_mc = 0, mb1 = 0; uint32_t rs_any = 0; bool seen_cl = false;
        auto finish = [&]() -> RangeRec {
            RangeRec a;
            a.c_lo = c_lo; a.c_hi = c_hi; a.n_own = n_own; a.ntok = ntok_range; a.lft = lft >= 0 ? lft - c_lo : -1; a.v = v_out;
            a.flags = (have ? RangeRec::HAVE : 0) | (closed ? RangeRec::CLOSED : 0) | (lo_found ? RangeRec::LO_FOUND : 0) |
                      (seen_cl ? RangeRec::HOLDS_CLOSER : 0) | (guessed_hot ? RangeRec::GUESSED_HOT : 0);
            a.u = 0; a.mb1 = 0;
            if (have && !lo_found) {               // (the summary exists)
                a.u = __any_sync(FULL, rs_any != 0u) ? NEG : __reduce_add_sync(FULL, d_mc);
                a.mb1 = min(__reduce_add_sync(FULL, mb1), 1 << 20);
            }
            return a;
        };
        if (!have) {
            c_hi = 0;
            v_out = x_init;
            return finish();
        }
        // ---- the character in front of the window: prev-context of the window's first character.  Matters only when the
        // range owns that character, i.e. no closer is found in the head window (then the range begins inside a chunk), and
        // for the feature rows of the head zone in token-feature mode.  A blank or a newline in the first 100 bytes is a
        // closer for sure, so almost every range skips this.
        uint32_t prevLB = 0;
        if (w0 > 0) {
            bool skip = false;
            if (!kFeats) {
                const uint32_t w4 = lane < 25 ? *reinterpret_cast<const uint32_t *>(X + LPAD + 4 * lane) : 0u;
                const uint32_t t1 = w4 ^ 0x20202020u, t2 = w4 ^ 0x0A0A0A0Au;
                skip = __any_sync(FULL, ((((t1 - 0x01010101u) & ~t1) | ((t2 - 0x01010101u) & ~t2)) & 0x80808080u) != 0u);
            }
            if (!skip) {
                const uint8_t *q = X + LPAD - 1;
                int back = 0;
                while (back < 3 && (q[-back] & 0xC0u) == 0x80u) ++back;
                const uint32_t w = classify_at(q - back, tb);
                prevLB = (w & 1u) | (((w >> 1) & 1u) << 1) | (((w >> 3) & 1u) << 2) | (((w >> 5) & 1u) << 3) | (((w >> 6) & 1u) << 4);
            }
        }
        const bool term_in_win = p.n_bytes < w0 + WIN;
        const long long rem64 = p.n_bytes - w0;
        const int nb_win = rem64 > (long long)(WIN + 64) ? WIN + 64 : (int)rem64;      // data bytes from the window start on (clamped)
        const int jt = last_range ? int((p.n_bytes - w0) >> 10) : -1;       // step / lane / bit of the end of the data
        const int lt = last_range ? int(((p.n_bytes - w0) >> 5) & 31) : 0, bt = last_range ? int((p.n_bytes - w0) & 31) : 0;

        // pipeline registers: base planes of the step that awaits its context
        uint32_t Pp[NBASE], Fp = 0, leadp = 0; int np = 0, c0p = 0;
#pragma unroll
        for (int f = 0; f < NBASE; ++f) Pp[f] = 0;
        int crun = 0;                    // characters of the range so far
        int xb = x_init;                 // block-mask backlog entering the next step (regular evaluation; 0 almost always)

#pragma unroll 1
        for (int j = 0; j <= RS; ++j) {
            // -------------------------------------------------------------- base planes of step j
            uint32_t Pc[NBASE], Fc = 0, leadc = 0; int nc = 0, c0c = 0;
#pragma unroll
            for (int f = 0; f < NBASE; ++f) Pc[f] = 0;
            if (j < RS) {
                const uint8_t *src = X + LPAD + j * STEP + lane * 32;
                const uint4 q0 = *reinterpret_cast<const uint4 *>(src), q1 = *reinterpret_cast<const uint4 *>(src + 16);
                const uint32_t wds[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
                uint32_t b[8];
                bytes_to_planes(wds, b);
                const int rem = nb_win - (j * STEP + lane * 32);
                const int vhi = min(max(rem, 0), 32);
                const uint32_t valid = mask_lt_nn(vhi);
                const uint32_t sb = sbmS[j * 32 + lane];
                leadc = (~(b[7] & ~b[6]) & valid) | sb;
                sbmS[j * 32 + lane] = leadc;                            // from here on the slot holds the lead-byte mask
                uint32_t mm = b[7] & b[6] & valid;                      // lead bytes of multi-byte characters
                classify_ascii(b, Pc);
                // multi-byte characters: decode + class table, features patched in at the lead byte, then the continuation
                // bytes are squeezed out.  Sparse (at most one such character per lane-word, e.g. an emoji in a tweet): one
                // look-up, run-by-run squeeze.  Dense (accented Latin, CJK): two characters per trip (independent look-up
                // chains, no branch on the character's length) and a five-stage compress.
                auto four_bytes = [&](int k) -> uint32_t {
                    const uint32_t *w = reinterpret_cast<const uint32_t *>(src + (k & ~3));
                    return __funnelshift_r(w[0], w[1], 8 * (k & 3));
                };
                Fc = sb;
                if (LIKELY(!__any_sync(FULL, (mm & (mm - 1u)) != 0u))) {
                    if (mm) {
                        const int k = __ffs(mm) - 1;
                        const uint32_t fw = mb_features(four_bytes(k), tb), bitk = 1u << k;
                        // (a character outside ASCII has none of TWITTER @ : / . -- planes 7..11 -- unless it is an over-long
                        // form of an ASCII character)
#pragma unroll
                        for (int f = 0; f < NMB; ++f) if (fw & (1u << f)) Pc[f] |= bitk;
                        if (UNLIKELY(fw >> NMB)) {
#pragma unroll
                            for (int f = NMB; f < NBASE; ++f) if (fw & (1u << f)) Pc[f] |= bitk;
                        }
                    }
                    squeeze_planes<NBASE>(Pc, Fc, leadc, valid);
                } else {
                    while (mm) {
                        const int k0 = __ffs(mm) - 1; mm &= mm - 1;
                        const bool two = mm != 0u;
                        const int k1 = two ? __ffs(mm) - 1 : k0; mm &= mm - 1;
                        const uint32_t v0 = four_bytes(k0), v1 = four_bytes(k1);
                        const uint32_t fw0 = mb_features(v0, tb), fw1 = two ? mb_features(v1, tb) : 0u;
                        const uint32_t bit0 = 1u << k0, bit1 = 1u << k1;
#pragma unroll
                        for (int f = 0; f < NMB; ++f) {
                            if (fw0 & (1u << f)) Pc[f] |= bit0;
                            if (fw1 & (1u << f)) Pc[f] |= bit1;
                        }
                        if (UNLIKELY((fw0 | fw1) >> NMB)) {
#pragma unroll
                            for (int f = NMB; f < NBASE; ++f) {
                                if (fw0 & (1u << f)) Pc[f] |= bit0;
                                if (fw1 & (1u << f)) Pc[f] |= bit1;
                            }
                        }
                    }
                    const uint32_t del = leadc ? (~leadc & valid) : 0u;
                    if (__any_sync(FULL, __popc(del & ~(del >> 1)) > LATOK_SQUEEZE_RUNS)) squeeze_planes_log<NBASE>(Pc, Fc, leadc);
                    else squeeze_planes<NBASE>(Pc, Fc, leadc, valid);
                }
                nc = __popc(leadc);
                int sc = nc;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(FULL, sc, d); if (lane >= d) sc += t; }
                c0c = crun + sc - nc;
                crun += __shfl_sync(FULL, sc, 31);
                if (UNLIKELY(j == jt)) c_hi = __shfl_sync(FULL, c0c + __popc(leadc & mask_lt(bt)), lt);
            }
            // -------------------------------------------------------------- context + rules of step j-1
            if (j > 0) {
                const int js = j - 1;
                const int n = np, c0 = c0p;
                const uint32_t Fm = Fp, lead = leadp;
                uint32_t *P = Pp;
                const uint32_t myLB = n > 0 ? ((((P[PL_A] >> (n - 1)) & 1u)) | (((P[PL_N] >> (n - 1)) & 1u) << 1) |
                                               (((P[PL_LO] >> (n - 1)) & 1u) << 2) | (((P[PL_SP] >> (n - 1)) & 1u) << 3) |
                                               (((P[PL_SY] >> (n - 1)) & 1u) << 4))
                                            : 0u;
                uint32_t LB = __shfl_up_sync(FULL, myLB, 1);
                if (lane == 0) LB = prevLB;
                prevLB = __shfl_sync(FULL, myLB, 31);
                const int nl = (lane + 1) & 31;
                const uint32_t XA = __shfl_sync(FULL, lane == 0 ? Pc[PL_A] : P[PL_A], nl), XN = __shfl_sync(FULL, lane == 0 ? Pc[PL_N] : P[PL_N], nl);
                const uint32_t XLO = __shfl_sync(FULL, lane == 0 ? Pc[PL_LO] : P[PL_LO], nl), XSP = __shfl_sync(FULL, lane == 0 ? Pc[PL_SP] : P[PL_SP], nl);
                const uint32_t XAT = __shfl_sync(FULL, lane == 0 ? Pc[PL_AT] : P[PL_AT], nl), XSL = __shfl_sync(FULL, lane == 0 ? Pc[PL_SL] : P[PL_SL], nl);
                const uint32_t XF = __shfl_sync(FULL, lane == 0 ? Fc : Fm, nl);
                const unsigned trel = (unsigned)(nb_win - (js * STEP + lane * 32));
                const bool has_term = trel < 32u;                 // the end-of-data terminator is this lane-word's last character
                const uint32_t REAL = mask_lt(n - (has_term ? 1 : 0));
                uint32_t TRUST = REAL;
                if (js == RS - 1 && lane == 31 && !term_in_win) TRUST &= mask_lt_nn(__popc(lead & mask_lt_nn(32 - MARGIN)));
                auto next1 = [&](uint32_t Xc, uint32_t Xn) -> uint32_t {
                    const uint32_t l = Xc | __funnelshift_lc(0u, Xn, n), h = __funnelshift_lc(Xn, 0u, n);
                    return __funnelshift_r(l, h, 1);
                };
                auto next2 = [&](uint32_t Xc, uint32_t Xn) -> uint32_t {
                    const uint32_t l = Xc | __funnelshift_lc(0u, Xn, n), h = __funnelshift_lc(Xn, 0u, n);
                    return __funnelshift_r(l, h, 2);
                };
                const uint32_t Lm_raw = next1(Fm, XF), L2m = next2(Fm, XF);
                const uint32_t nF = ~Lm_raw, aF = ~(Lm_raw | L2m), pF = ~Fm;
                const uint32_t Sraw = P[PL_SP];
                uint32_t full[NFEAT];
#pragma unroll
                for (int f = 0; f < NBASE; ++f) full[f] = P[f];
                full[12] = ((P[PL_A] << 1) | (LB & 1u)) & pF;                 // PREV_ALPHA
                full[13] = next1(P[PL_A], XA) & nF;                           // NEXT_ALPHA
                full[14] = ((P[PL_N] << 1) | ((LB >> 1) & 1u)) & pF;          // PREV_ALPHA_NUM
                full[15] = next1(P[PL_N], XN) & nF;                           // NEXT_ALPHA_NUM
                full[16] = ((P[PL_LO] << 1) | ((LB >> 2) & 1u)) & pF;         // PREV_LOWER
                full[17] = next1(P[PL_LO], XLO) & nF;                         // NEXT_LOWER
                full[18] = ((P[PL_SP] << 1) | ((LB >> 3) & 1u)) | Fm;         // PREV_SPACE  (start of string = space)
                full[19] = next1(P[PL_SP], XSP) | Lm_raw;                     // NEXT_SPACE  (end of string = space)
                full[20] = ((P[PL_SY] << 1) | ((LB >> 4) & 1u)) & pF;         // PREV_SYMBOL
                full[21] = next1(P[PL_AT], XAT) & nF;                         // NEXT_AT
                full[22] = next1(P[PL_SL], XSL) & nF;                         // NEXT_SLASH
                full[23] = next2(P[PL_A], XA) & aF;                           // AFTER_NEXT_ALPHA
                full[24] = next2(P[PL_SL], XSL) & aF;                         // AFTER_NEXT_SLASH
                uint32_t CNT[NC], SYC[NY], Mraw;
                if (kDefault) {
                    // C_SPLIT: SPACE + SYMBOL + PREV_SYMBOL + UPPER*NEXT_LOWER + UPPER*PREV_LOWER (default_tokenizer.py:49-55);
                    // up to 4 (UPPER is a Unicode property that some SYMBOL characters carry too), 5 with C_SYM: three planes
                    const uint32_t t1 = full[5], t2 = full[6], t3 = full[20], t4 = full[4] & full[17], t5 = full[4] & full[16];
                    const uint32_t s1 = t1 ^ t2 ^ t3, c1 = (t1 & t2) | (t3 & (t1 ^ t2));
                    const uint32_t s2 = t4 ^ t5, c2 = t4 & t5;
                    CNT[0] = s1 ^ s2;
                    const uint32_t c3 = s1 & s2;
                    CNT[1] = c1 ^ c2 ^ c3;
                    CNT[2] = (c1 & c2) | (c3 & (c1 ^ c2));
                    // C_MASK (default_tokenizer.py:80-91)
                    Mraw = (full[7] & full[18] & full[13]) | (full[11] & full[18] & full[21] & full[23]) |
                           (full[8] & full[14] & full[15]) | (full[9] & full[22] & full[24] & full[12]);
                    // C_SYM: SYMBOL*NEXT_SPACE (default_tokenizer.py:100-102)
                    SYC[0] = full[6] & full[19];
                } else {
                    auto term = [&](uint32_t mask) -> uint32_t {
                        uint32_t a = 0xFFFFFFFFu;
#pragma unroll
                        for (int f = 0; f < NFEAT; ++f) a &= full[f] | (((mask >> f) & 1u) - 1u);
                        return a;
                    };
                    auto add1 = [&](uint32_t *c, int nb, uint32_t t) {
                        for (int q = 0; q < nb; ++q) { const uint32_t k = c[q] & t; c[q] ^= t; t = k; }
                    };
#pragma unroll
                    for (int q = 0; q < NC; ++q) CNT[q] = 0;
#pragma unroll
                    for (int q = 0; q < NY; ++q) SYC[q] = 0;
                    Mraw = 0;
                    for (int i = 0; i < p.rules.n_split; ++i) add1(CNT, NC, term(p.rules.split[i]));
                    for (int i = 0; i < p.rules.n_mask; ++i) Mraw |= term(p.rules.mask[i]);
                    for (int i = 0; i < p.rules.n_sym; ++i) add1(SYC, NY, term(p.rules.sym[i]));
                }
                if (kFeats) {
                    // token-feature mode: the 25 feature planes of the lane-word go to a global scratch for pass D
                    uint32_t *pl = p.planes + (((size_t)r * RS + js) * NFEAT) * 32 + lane;
#pragma unroll
                    for (int f = 0; f < NFEAT; ++f) pl[f * 32] = full[f];
                }
                // ---- chunk-aligned ownership (both neighbours look at the same bytes)
                const uint32_t CLr = (Sraw | Lm_raw) & REAL;
                if (js == 0 && r > 0) {
                    uint32_t cand = lane < HLANES ? CLr : 0u;
                    if (lane == HLANES - 1) cand &= mask_lt(__popc(lead & mask_lt(32 - MARGIN)));
                    const unsigned bl = __ballot_sync(FULL, cand != 0u);
                    lo_found = bl != 0u;
                    const int fl = bl ? __ffs(bl) - 1 : 0;
                    const int cv = __shfl_sync(FULL, c0 + __ffs(cand), fl);
                    c_lo = lo_found ? cv : 0;
                }
                if (js == RS - 1 && !last_range) {
                    uint32_t cand = lane >= 32 - HLANES ? CLr : 0u;
                    if (lane == 31) cand &= mask_lt(__popc(lead & mask_lt(32 - MARGIN)));
                    const unsigned bh = __ballot_sync(FULL, cand != 0u);
                    closed = bh != 0u;
                    const int fl = bh ? __ffs(bh) - 1 : 32 - HLANES;
                    const int cv = __shfl_sync(FULL, closed ? c0 + __ffs(cand) : c0, fl);
                    c_hi = cv;
                }
                // ---- forward half of the block mask, common case: a carry-propagating add per lane-word
                uint32_t HOTorM;
                {
                    // characters the block mask runs over: the owned ones (c_hi is still "infinite" before the last step)
                    const uint32_t ACTf = range_mask(c0, c_lo, c_hi) & TRUST;
                    const uint32_t Mm = Mraw & ACTf, CL = CLr & ACTf;
                    // (summary for resolve(): the range as a backlog transfer function, marks in front of its first closer)
                    // -- kept only for ranges that begin inside a chunk (the others are asked again if a backlog enters them)
                    if (UNLIKELY(!lo_found)) {
                        d_mc += __popc(Mm) - __popc(CL);
                        rs_any |= (Fm | Lm_raw) & ACTf;
                    }
                    if (UNLIKELY(!lo_found && !seen_cl)) {
                        const unsigned Gc = __ballot_sync(FULL, CL != 0u);
                        const int fl = Gc ? __ffs(Gc) - 1 : 32;
                        // (a mark on a closer comes first: the first closer's own mark counts -- generic rules only, the
                        // default mask rows never fire on a closer)
                        const uint32_t upto = kDefault ? (CL & (0u - CL)) - 1u : CL ^ (CL - 1u);
                        mb1 += __popc(lane < fl ? Mm : (lane == fl ? (Mm & upto) : 0u));
                        seen_cl = Gc != 0u;
                    }
                    uint32_t co;
                    (void)chunk_carry(Mm, CL, 0u, co);
                    const unsigned G = __ballot_sync(FULL, co != 0u), Pg = __ballot_sync(FULL, CL == 0u && co == 0u);
                    const unsigned long long sum = (unsigned long long)(G | Pg) + (unsigned long long)G + (unsigned long long)(xb != 0 ? 1u : 0u);
                    const uint32_t cin = (((uint32_t)sum ^ Pg) >> lane) & 1u;
                    const uint32_t T = chunk_carry(Mm, CL, cin, co);
                    // chunk_carry drops a mark on a closer: under generic rules such a step is evaluated mark by mark
                    const uint32_t exact = (Mm & ~CL & T) | (kDefault ? 0u : (Mm & CL));
                    if (LIKELY(xb < 2 && !__any_sync(FULL, exact != 0u))) {
                        HOTorM = T & CL;
                        xb = (int)((sum >> 32) & 1u);
                    } else {
                        // a chunk with several marks (or a backlog of several): this step mark by mark
                        int out;
                        HOTorM = exact_step(xb, Mm, Fm & ACTf, Sraw & ACTf, Lm_raw & ACTf, out);
                        xb = __shfl_sync(FULL, out, 31);
                    }
                }
                // ---- park the step for pass C (step js+1 has been read already)
                PS(tempS, js, lane).store_a(CNT, SYC, Sraw, HOTorM, Fm, pack_ncp(n, c0, (int)((LB >> 3) & 1u)) | ((XF & 1u) << 31));
            }
#pragma unroll
            for (int f = 0; f < NBASE; ++f) Pp[f] = Pc[f];
            Fp = Fc; leadp = leadc; np = nc; c0p = c0c;
        }
        PROF5(1);
        if (c_hi == CINF) c_hi = crun;           // (defensive; every range sets it)
        n_own = c_hi - c_lo;
        if (n_own < 0) n_own = 0;
        v_out = xb;
        if (lane == 0) {                           // (statistics)
            if (xb != 0) atomicAdd(&p.result->stats.backlog_out, 1ull);
            if (!lo_found) atomicAdd(&p.result->stats.open_head, 1ull);
            if (!closed) atomicAdd(&p.result->stats.open_tail, 1ull);
        }
        __syncwarp();
        // character ends its string: the next character (possibly in the next lane-word) starts one
        auto L_of = [&](uint32_t Fm, uint32_t pk) -> uint32_t {
            const int n = pk_n(pk);
            return n > 0 ? ((Fm >> 1) | ((pk >> 31) << (n - 1))) : 0u;
        };
        auto real_mask = [&](int js, int n) -> uint32_t {
            const bool has_term = (unsigned)(nb_win - (js * STEP + lane * 32)) < 32u;
            return mask_lt(n - (has_term ? 1 : 0));
        };
        // First analysis of a range that ends inside a chunk: a guess whether that chunk will be closed hot (the service warp
        // knows better later, resolve()).  Yes if a mark is pending at the end; yes if the range also BEGINS inside the chunk
        // or the open part is long (a space-free run of that length nearly always holds a mark somewhere); no for a short
        // open part without a mark (a long word or URL-less stretch at the range end).
        bool far_guess = false;
        if (UNLIKELY(!closed)) {
            far_guess = !lo_found || xb != 0;
            if (!far_guess) {
                int open_len = n_own;
#pragma unroll 1
                for (int js = RS - 1; js >= 0; --js) {
                    const PS t(tempS, js, lane);
                    const uint32_t pk = t.packed();
                    const int n = pk_n(pk), c0 = pk_c0(pk);
                    const uint32_t CLo = (t.s() | L_of(t.f(), pk)) & range_mask(c0, c_lo, c_hi) & real_mask(js, n);
                    const unsigned hb = __ballot_sync(FULL, CLo != 0u);
                    if (hb) {
                        const int pos = __shfl_sync(FULL, c0 + 31 - (int)__clz(CLo), 31 - __clz(hb));
                        open_len = c_hi - pos - 1;
                        break;
                    }
                }
                far_guess = open_len >= 512;
            }
        }
        guessed_hot = far_init < 0 ? far_guess : (far_init != 0);
        PROF5(2);
        // ---------------------------------------------------------------- pass C: blanked chunks, values, tokens
        {
            uint32_t bin_step = far_init < 0 ? (far_guess ? 1u : 0u) : (uint32_t)far_init;
            int nsa_carry = -1;
            int lft_max = -1;
#pragma unroll 1
            for (int js = RS - 1; js >= 0; --js) {
                const PS t(tempS, js, lane);
                uint32_t CNT[NC], SYC[NY], Sraw, HOT, Fm, pk;
                t.load_a(CNT, SYC, Sraw, HOT, Fm, pk);
                const int n = pk_n(pk), c0 = pk_c0(pk);
                const uint32_t REAL = real_mask(js, n);
                const uint32_t OWN = range_mask(c0, c_lo, c_hi) & REAL;
                const uint32_t CL = (Sraw | L_of(Fm, pk)) & OWN;
                HOT &= CL;
                const bool hasCL = CL != 0u;
                const bool firstHot = hasCL && (HOT & (CL & (0u - CL))) != 0u;
                const unsigned H = __ballot_sync(FULL, hasCL), FH = __ballot_sync(FULL, firstHot);
                const unsigned above = lane == 31 ? 0u : (H & (0xFFFFFFFFu << (lane + 1)));
                const uint32_t bin = above ? ((FH >> (__ffs(above) - 1)) & 1u) : bin_step;
                if (H) bin_step = (FH >> (__ffs(H) - 1)) & 1u;
                const uint32_t Zm = flood_down(HOT, CL, bin);
                const uint32_t keepm = ~Zm | Sraw;             // block mask = 1
                // split values: splits = split_cnt * block_mask + sym; splits[0] = 1 (default_tokenizer.py:121-132)
                uint32_t V[NV];
                if (kDefault) {
                    const uint32_t x0 = CNT[0] & keepm, x1 = CNT[1] & keepm, x2 = CNT[2] & keepm, y = SYC[0];
                    V[0] = x0 ^ y;
                    const uint32_t k0 = x0 & y;
                    V[1] = x1 ^ k0;
                    V[2] = x2 ^ (x1 & k0);
                } else {
                    uint32_t carry = 0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint32_t xq = CNT[q] & keepm, y = SYC[q];
                        V[q] = xq ^ y ^ carry;
                        carry = (xq & y) | (carry & (xq ^ y));
                    }
                    V[4] = carry;
                }
                V[0] |= Fm;
#pragma unroll
                for (int q = 1; q < NV; ++q) V[q] &= ~Fm;
                uint32_t SPLIT = 0;
#pragma unroll
                for (int q = 0; q < NV; ++q) SPLIT |= V[q];
                const uint32_t PS = (Sraw << 1) | pk_ps(pk);
                const uint32_t E = ((SPLIT & ~Sraw) | (~SPLIT & PS & ~Fm)) & OWN;     // a token is counted at this character
                int ts = __popc(E);
                const int mytok = ts;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int q = __shfl_up_sync(FULL, ts, d); if (lane >= d) ts += q; }
                const int tot = __shfl_sync(FULL, ts, 31);
                ntok_range += tot;
                // first split that can end a token, for the steps before this one
                const uint32_t SPq = SPLIT & mask_lt(n) & range_mask(c0, c_lo, closed ? c_hi + 1 : c_hi);
                const unsigned hs = __ballot_sync(FULL, SPq != 0u);
                const int firstsp = __shfl_sync(FULL, c0 + __ffs(SPq) - 1, hs ? __ffs(hs) - 1 : 0);
                if (lane == 0) { ctl.tokstep[w][buf][js] = tot; ctl.nsa[w][buf][js] = nsa_carry; }
                if (hs) nsa_carry = firstsp;
                const uint32_t FO = Fm & OWN;
                if (FO) lft_max = max(lft_max, c0 + 31 - __clz(FO));
                // state for pass D (the window's map is rebuilt by the next analysis: the lead mask moves into the state)
                t.store_c(V, E, sbmS[js * 32 + lane], (pk & 0xC007FFFFu) | ((uint32_t)(ts - mytok) << 19));
            }
            lft = __reduce_max_sync(FULL, lft_max);
        }
        const RangeRec a = finish();
        PROF5(3);
        return a;
    };

    // =================================================================================================
    // service warp: tile aggregate, backlog / hot-tail resolution, look-back, prefix hand-down
    // =================================================================================================
    if (warp == 0) {
        for (int k = 0;; ++k) {
            const int s = k & 1;
            TileSum sum;                                       // tile totals from what the ranges have posted (ctl.rec)
            // lane i < NW: what range i posted with its FIRST analysis (nothing entering): backlog left (sf0), flags,
            // and -- only for ranges that begin inside a chunk (LO_FOUND clear) -- marks - closers (su; NEG: a string
            // boundary resets the backlog) and the marks in front of the first closer (smb1) ...
            int su = 0, sf0 = 0, smb1 = 0, sflags = RangeRec::CLOSED | RangeRec::LO_FOUND;
            // ... what it has been analysed with so far, and the backlog it left the last time
            int x_used = 0, far_used = 0, v_last = 0;
            // Backlog entering / hot tail of every range, given the backlog `x_tile` that enters the tile.  A range whose
            // result depends on something other than what it was analysed with is analysed AGAIN -- by this warp, at once:
            // the warp that owns the range is busy with its next tile and would only get to it ~10 us later, with the whole
            // look-back chain waiting (the window is fetched again into the owner's buffer of this tile, which the owner
            // does not touch before the prefix is handed down; the string map goes to a scratch of the service warp).
            // A range that begins at a chunk closer has no summary: if a backlog enters it after all, what it leaves is known
            // once it has been analysed again, and the ranges behind it follow in the next round (rare, short cascades).
            // Returns the backlog leaving the tile.
            auto resolve = [&](int x_tile) -> int {
                // nothing enters, nothing is left, every range ends at a closer: almost every tile
                if (x_tile == 0 && !__any_sync(FULL, lane < NW && (sflags & RangeRec::HAVE) != 0 &&
                                                          (sf0 != 0 || (sflags & RangeRec::CLOSED) == 0 || x_used != 0)))
                    return 0;
                const long long tile_w = ld_vs32(&ctl.tile_id[s]);
                int x_out = x_tile;
                for (;;) {
                    int xin = x_tile, x = x_tile, xend = 0;
                    bool known = true, kin = false, kend = false;    // (x known: entering range i / at its end)
#pragma unroll 1
                    for (int i = 0; i < NW; ++i) {
                        const int ui = __shfl_sync(FULL, su, i), fi = __shfl_sync(FULL, sf0, i), fl = __shfl_sync(FULL, sflags, i);
                        const int xu = __shfl_sync(FULL, x_used, i), vl = __shfl_sync(FULL, v_last, i);
                        if (lane == i) { xin = x; kin = known; }
                        if (known) {
                            if ((fl & RangeRec::HAVE) == 0) { /* no data: passes the backlog on */ }
                            else if ((fl & RangeRec::LO_FOUND) == 0) x = max(x + ui, fi);
                            else if (x == 0) x = fi;
                            else if (x == xu) x = vl;                 // it has been analysed with exactly this backlog
                            else known = false;
                        }
                        if (lane == i) { xend = x; kend = known; }
                    }
                    x_out = x;
                    const bool all_known = known;
                    const bool have = lane < NW && (sflags & RangeRec::HAVE) != 0;
                    const bool open = have && (sflags & RangeRec::CLOSED) == 0;           // the range ends inside a chunk
                    int far = far_used;
                    bool walk = false;
                    {
                        const unsigned Bm = __ballot_sync(FULL, lane < NW && smb1 > 0);
                        const unsigned Bc = __ballot_sync(FULL, lane < NW && (sflags & RangeRec::HOLDS_CLOSER) != 0);
                        const unsigned Bn = __ballot_sync(FULL, lane < NW && (sflags & RangeRec::HAVE) == 0);
                        if (open && kend) {
                            far = 0;
                            if (xend > 0) far = 1;
                            else {
                                // the first later range that holds a mark in front of its first closer / a closer / no data
                                const unsigned dec = (Bm | Bc | Bn) & (0xFFFFFFFEu << lane) & mask_lt(NW);
                                if (dec) far = (int)((Bm >> (__ffs(dec) - 1)) & 1u);
                                else walk = true;                            // the chunk runs on past the end of the tile
                            }
                        }
                    }
                    if (__any_sync(FULL, walk)) {
                        const bool any = walk_ahead(p, tb, (tile_w + 1) * (long long)NW * RANGE, lane);
                        if (walk) far = any ? 1 : 0;
                        if (lane == 0) atomicAdd(&p.result->walks, 1ull);
                    }
                    // the backlog that enters matters where there is a closer to meet it (a range without a summary -- it begins
                    // at a closer -- is assumed to hold one); a range that lies inside one chunk only needs to know whether
                    // that chunk will be closed hot
                    const bool x_matters = (sflags & (RangeRec::LO_FOUND | RangeRec::HOLDS_CLOSER)) != 0;
                    const bool need = have && kin && ((xin != x_used && x_matters) || far != far_used);
                    unsigned todo = __ballot_sync(FULL, need);
                    if (!todo) {
                        if (!all_known && lane == 0) atomicOr(&p.result->error, 1u);      // (cannot happen: every round makes a range known)
                        break;
                    }
                    {   // (statistics: repeat rounds, ranges repeated, of those because of the hot-tail guess)
                        const unsigned fb = __ballot_sync(FULL, need && far != far_used);
                        if (lane == 0) {
                            atomicAdd(&p.result->stats.repeat_rounds, 1ull); atomicAdd(&p.result->stats.ranges_repeated, (unsigned long long)__popc(todo));
                            atomicAdd(&p.result->stats.repeats_hot_tail, (unsigned long long)__popc(fb));
                        }
                    }
                    if (need) { x_used = xin; far_used = far; }
                    while (todo) {
                        const int i = __ffs(todo) - 1; todo &= todo - 1;
                        const int xi = __shfl_sync(FULL, xin, i), fi = __shfl_sync(FULL, far, i);
                        const long long r = tile_w * NW + i;
                        plain_load(r, i, s);
                        build_map(r, i);
                        const RangeRec a = analyze(r, s, i, xi, fi);
                        if (lane == 0) {                       // (the rest does not depend on what enters the range)
                            ctl.rec[s][i].ntok = a.ntok; ctl.rec[s][i].v = a.v;
                        }
                        if (lane == i) v_last = a.v;
                    }
                    __threadfence_block();
                    __syncwarp();
                    sum = sum_ranges(ctl.rec[s], NW, lane);
                }
                return x_out;
            };
            nb_sync(BAR_AGG + s, NTH);               // every range of the tile has been analysed and posted
            sum = sum_ranges(ctl.rec[s], NW, lane);
            if (lane < NW) {
                const RangeRec a = ctl.rec[s][lane];
                su = a.u; sf0 = a.v; smb1 = a.mb1; sflags = a.flags; v_last = a.v;
                far_used = (a.flags & RangeRec::GUESSED_HOT) ? 1 : 0;
            }
            const long long tile = ld_vs32(&ctl.tile_id[s]);
            if (tile >= p.ntiles) break;
            // The aggregate is published under the assumption that no backlog enters the tile (true for almost every tile).
            // A tile that begins inside a chunk (a long space-free run is passing through) most likely does get one: it
            // publishes nothing before it knows (its successors would have to wait for its inclusive prefix anyway) and
            // settles once, with the backlog that really enters.
            const bool begins_inside = tile > 0 && (__shfl_sync(FULL, sflags, 0) & (RangeRec::HAVE | RangeRec::LO_FOUND)) == RangeRec::HAVE;
            int v = 0;
            if (!begins_inside) {
                v = resolve(0);
                if (lane == 0) publish_agg(p.agg + tile, p.epoch, AGG_AGGREGATE, sum, v);
            }
            const Prefix pre = lookback(tile, p, lane);
            if (begins_inside || pre.x != 0) {
#ifdef LATOK_PROFILE
                const long long _s1 = clock64();
#endif
                v = resolve(pre.x);
#ifdef LATOK_PROFILE
                if (lane == 0) { atomicAdd(&p.result->clocks.resolve, (unsigned long long)(clock64() - _s1)); atomicAdd(&p.result->clocks.resolve_calls, 1ull); }
#endif
            }
            if (lane == 0) {
                Prefix inc = advance(pre, sum);
                inc.x = v;
                publish_inc(p.inc + tile, inc);
                __threadfence();
                publish_agg(p.agg + tile, p.epoch, AGG_INCLUSIVE, sum, v);
                Prefix &sl = ctl.slot[s];            // (not x: storing it costs the short geometry a spill)
                sl.G = pre.G; sl.base = pre.base; sl.K = pre.K;
                __threadfence_block();
            }
            __syncwarp();
            nb_arrive(BAR_PRE + s, NTH);
        }
        return;
    }

    // ================================================================================================= output
    auto output = [&](const long long r, const int buf, unsigned long long G_in, unsigned long long K_in, unsigned long long base_in) {
        const RangeRec ri = ctl.rec[buf][cw];
        const bool have = (ri.flags & RangeRec::HAVE) != 0, closed = (ri.flags & RangeRec::CLOSED) != 0;
        const bool lo_found = (ri.flags & RangeRec::LO_FOUND) != 0;
        // (the last range is tested as r == p.nranges - 1 where it matters: r stays live anyway, a bool held across pass D
        // costs the token-feature instantiation spills)
        if (!have) return;
        const int c_lo = ri.c_lo, c_hi = ri.c_hi, n_own = ri.n_own, ntok_range = ri.ntok;
        const long long w0 = r * (long long)RANGE;
        const long long rem64 = p.n_bytes - w0;
        const int nb_win = rem64 > (long long)(WIN + 64) ? WIN + 64 : (int)rem64;
        uint32_t *tempS = tempof(cw, buf);
        if (K_in + (unsigned long long)ntok_range > (unsigned long long)p.cap_tokens && lane == 0) atomicOr(&p.result->error, 4u);
        if (G_in + (unsigned long long)n_own > (unsigned long long)p.n_bytes || K_in + (unsigned long long)ntok_range > (unsigned long long)p.n_bytes + 1ull) {
            if (lane == 0 && atomicOr(&p.result->error, 8u) == 0u) {
                FaultRec &f = p.result->fault;
                f.range = (unsigned long long)r; f.G_in = G_in; f.K_in = K_in;
                f.n_own = n_own; f.ntok = ntok_range; f.c_lo = c_lo; f.c_hi = c_hi;
            }
            return;
        }
        // range-relative character index of the first character of the string that is open at c_lo (may be negative)
        int cur_base = c_lo - (int)(long long)(G_in - base_in);
        int ktok = 0;                      // tokens of the range before this step
        unsigned fc[7] = {0, 0, 0, 0, 0, 0, 0};      // token-feature mode: sums of the token open at the end of the previous step
        bool fc_hit = false;                          // ... and whether its first character has been seen
        // token-feature rows: aligned base of the rows of this range, byte phase of relative row 0 in it, the relative
        // ordinals that may be written ([f_kmin, f_kmax): row capacity of the caller's array)
        uint32_t *f_base = nullptr; int f_phase = 0, f_kmin = 0, f_kmax = 0, f_ph16 = 0; int8_t *f_g16 = nullptr;
        if (kFeats) {
            const unsigned long long fb = K_in * (unsigned long long)NFEAT;
            f_ph16 = (int)(fb & 15ull);
            f_g16 = p.feats + (fb - (unsigned long long)f_ph16);
            f_phase = (int)(fb & 3ull);
            f_base = reinterpret_cast<uint32_t *>(p.feats + (fb - (unsigned long long)f_phase));
            f_kmin = K_in > 0ull ? -1 : 0;
            const long long room = p.cap_tokens - (long long)K_in;
            f_kmax = room > (long long)(1 << 28) ? (1 << 28) : (room < -1 ? -1 : (int)room);
        }
        const bool spans_direct_all = !closed || !lo_found ||
                                      K_in + (unsigned long long)ntok_range > (unsigned long long)p.cap_tokens;   // (the direct path checks every pair)
        // ---------------------------------------------------------------- CSR offsets of the strings that start in this range
        // (first: in token-feature mode the step loop below reuses the state of a step, once read, as scratch)
        // (one lane per string; the character / token counts in front of a byte position come from the parked state)
        {
            __syncwarp();
            const long long wend = w0 + WIN;
            for (long long q = p.tile_first_str[r] + lane;; q += 32) {
                const long long o = q <= p.n_strings ? p.offsets[q] : 0x7FFFFFFFFFFFFFFFLL;
                const bool in = o < wend;
                if (in) {
                    const int wb = int(o - w0);
                    const int js = wb >> 10, tl = (wb >> 5) & 31;
                    const PS t(tempS, js, tl);
                    const uint32_t l_pk = t.packed(), l_E = t.e(), l_lead = t.lead();
                    const int l_c0 = pk_c0(l_pk);
                    const int c = l_c0 + __popc(l_lead & mask_lt_nn(wb & 31));
                    const bool mine = r == p.nranges - 1 ? (c >= c_lo) : (c >= c_lo && c < c_hi);
                    if (mine) {
                        int kb = 0;
                        for (int q2 = 0; q2 < js; ++q2) kb += ctl.tokstep[cw][buf][q2];
                        p.char_off[q] = (long long)(G_in + (unsigned long long)(c - c_lo));
                        p.tok_off[q] = (long long)K_in + kb + pk_tp(l_pk) + __popc(l_E & mask_lt(c - l_c0));
                    }
                }
                if (!__all_sync(FULL, in)) break;
            }
        }
#pragma unroll 1
        for (int js = 0; js < RS; ++js) {
            uint32_t V[NV], E, Sraw, Fm, pk;
            PS(tempS, js, lane).load_c(V, E, Sraw, Fm, pk);
            const int n = pk_n(pk), c0 = pk_c0(pk), tp = pk_tp(pk);
            const int wrel = nb_win - (js * STEP + lane * 32);          // data bytes from this lane-word on
            const bool has_term = (unsigned)wrel < 32u;
            const uint32_t REAL = mask_lt(n - (has_term ? 1 : 0));
            const uint32_t OWN = range_mask(c0, c_lo, c_hi) & REAL;
            const int cstep0 = __shfl_sync(FULL, c0, 0), cstep1 = __shfl_sync(FULL, c0 + n, 31);
            const int cf = max(c_lo, cstep0), cend = min(c_hi, cstep1);     // owned characters of this step: [cf, cend)
            const int nb = cend - cf;
            const int ntok_step = ctl.tokstep[cw][buf][js];
            uint32_t SPLIT = 0;
#pragma unroll
            for (int q = 0; q < NV; ++q) SPLIT |= V[q];
            // ------------------------------------------------------------ split mask bytes
            // The value planes are compacted at the bit level: every lane ORs its characters into a per-step bit stream
            // in shared memory whose origin is the 16-byte boundary at or below the step's first character in the output,
            // then lane t expands stream bits [32t, 32t+32) into 32 bytes and stores them as two aligned 16-byte chunks.
            if (want_splits && nb > 0) {
                const long long Gs0 = (long long)G_in + (cstep0 - c_lo);           // output index of the step's first character
                const int a = (int)(Gs0 & 15);
                int8_t *obase = p.splits + (Gs0 - a);                               // 16-byte aligned
                uint32_t *bp = reinterpret_cast<uint32_t *>(sst);                   // [NV][36] words, kept zero between steps
                {
                    const int bpos = a + (c0 - cstep0);
                    const int w = bpos >> 5, sh = bpos & 31;
#pragma unroll
                    for (int q = 0; q < NV; ++q) {
                        const uint32_t v = V[q] & OWN;                               // nothing but owned characters enters the stream
                        if (v) {
                            atomicOr(&bp[q * 36 + w], v << sh);
                            const uint32_t hi = __funnelshift_l(v, 0u, sh);          // bits that spill into the next word
                            if (hi) atomicOr(&bp[q * 36 + w + 1], hi);
                        }
                    }
                }
                __syncwarp();
                const int bf = a + (cf - cstep0), be = bf + nb;                     // owned stream positions [bf, be)
                uint32_t Vs[NV];
#pragma unroll
                for (int q = 0; q < NV; ++q) { Vs[q] = bp[q * 36 + lane]; bp[q * 36 + lane] = 0; }
                uint32_t W[8];
                auto expand = [&](const uint32_t *Vx) {
                    if (kDefault) {
                        const uint32_t qlo = (Vx[0] & 0x0F0F0F0Fu) | ((Vx[1] & 0x0F0F0F0Fu) << 4);
                        const uint32_t qhi = ((Vx[0] >> 4) & 0x0F0F0F0Fu) | (Vx[1] & 0xF0F0F0F0u);
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            W[2 * g] = lutv[(qlo >> (8 * g)) & 0xFFu];
                            W[2 * g + 1] = lutv[(qhi >> (8 * g)) & 0xFFu];
                        }
                        if (Vx[2]) {
#pragma unroll
                            for (int g = 0; g < 8; ++g) W[g] += spread4((Vx[2] >> (4 * g)) & 15u) << 2;
                        }
                    } else {
#pragma unroll
                        for (int g = 0; g < 8; ++g) {
                            uint32_t w = 0;
#pragma unroll
                            for (int q = 0; q < NV; ++q) w += spread4((Vx[q] >> (4 * g)) & 15u) << q;
                            W[g] = w;
                        }
                    }
                };
                expand(Vs);
                const int p0 = 32 * lane;
                const uint4 c1 = make_uint4(W[0], W[1], W[2], W[3]), c2 = make_uint4(W[4], W[5], W[6], W[7]);
                if (p0 >= bf && p0 + 16 <= be) *reinterpret_cast<uint4 *>(obase + p0) = c1;
                if (p0 + 16 >= bf && p0 + 32 <= be) *reinterpret_cast<uint4 *>(obase + p0 + 16) = c2;
                // the (at most two) chunks that are only partly owned go through a byte stage
                uint8_t *bst = reinterpret_cast<uint8_t *>(tst);                    // (the token stage is idle here)
                *reinterpret_cast<uint4 *>(bst + p0) = c1;
                *reinterpret_cast<uint4 *>(bst + p0 + 16) = c2;
                if (UNLIKELY(be > 1024)) {          // stream positions 1024.. (the step holds up to 1025 characters, plus the alignment)
                    uint32_t Vt[NV];
#pragma unroll
                    for (int q = 0; q < NV; ++q) Vt[q] = bp[q * 36 + 32];
                    __syncwarp();
                    if (lane == 0) {
#pragma unroll
                        for (int q = 0; q < NV; ++q) { bp[q * 36 + 32] = 0; bp[q * 36 + 33] = 0; }
                    }
                    expand(Vt);
                    if (lane == 0) {
                        *reinterpret_cast<uint4 *>(bst + 1024) = make_uint4(W[0], W[1], W[2], W[3]);
                        *reinterpret_cast<uint4 *>(bst + 1040) = make_uint4(W[4], W[5], W[6], W[7]);
                    }
                }
                __syncwarp();
                {
                    const int hend = min((bf + 15) & ~15, be);                       // head: [bf, hend)
                    if (lane < hend - bf) obase[bf + lane] = (int8_t)bst[bf + lane];
                    const int tbeg = max(be & ~15, hend);                            // tail: [tbeg, be)
                    if (lane < be - tbeg) obase[tbeg + lane] = (int8_t)bst[tbeg + lane];
                }
                __syncwarp();
            }
            // (token-feature mode: the 25 feature planes of the lane-word, parked in HBM by pass A -- asked for here, used after
            // the spans, so that the L2 latency is covered)
            uint32_t Q[kFeats ? NFEAT : 1];
            if (kFeats) {
                const uint32_t *pl = p.planes + (((size_t)r * RS + js) * NFEAT) * 32 + lane;
#pragma unroll
                for (int f = 0; f < NFEAT; ++f) Q[f] = pl[f * 32];
            }
            // ------------------------------------------------------------ token spans
            // latest owned string start in the lanes before this one (else: the one open when the step began)
            const uint32_t FO = Fm & OWN;
            int lf_excl;
            {
                const int mine = FO ? c0 + 31 - __clz(FO) : -1;
                const unsigned has = __ballot_sync(FULL, FO != 0u);
                const unsigned below = has & mask_lt(lane);
                const int got = __shfl_sync(FULL, mine, below ? 31 - __clz(below) : 0);
                lf_excl = below ? got : cur_base;
                const int wlast = __shfl_sync(FULL, mine, has ? 31 - __clz(has) : 0);
                if (has) cur_base = wlast;      // (for the next step; this step uses lf_excl)
            }
            if (want_spans) {
                const unsigned long long Ks = K_in + (unsigned long long)ktok;
                const bool direct = spans_direct_all || ntok_step > TCAP;
                const int ka = (int)(Ks & 1ull);
                // one (start, end) pair per token; end = next split (a string start is always a split)
                const uint32_t SPq = SPLIT & mask_lt(n) & range_mask(c0, c_lo, closed ? c_hi + 1 : c_hi);
                const int myfirst = SPq ? c0 + __ffs(SPq) - 1 : -1;
                const unsigned hs = __ballot_sync(FULL, myfirst >= 0);
                int nextsplit;     // first split in the following lanes / steps (-1: none in this range)
                {
                    const unsigned above = lane == 31 ? 0u : (hs & (0xFFFFFFFFu << (lane + 1)));
                    const int got = __shfl_sync(FULL, myfirst, above ? __ffs(above) - 1 : 0);
                    nextsplit = above ? got : ctl.nsa[cw][buf][js];
                }
                const bool multi_f = __any_sync(FULL, (FO & (FO - 1u)) != 0u);      // two string starts inside one lane-word
                if (LIKELY(!direct && !multi_f)) {
                    // bit-reversed planes: __clz walks the tokens in ascending order, the first split after a token is the
                    // highest bit below it.  At most one string start per lane-word here.
                    // (positions are handled as q = 31 - position, the index FLO returns on the reversed planes)
                    uint32_t evr = __brev(E);
                    const uint32_t spr = __brev(SPq), e2r = __brev(E & ~SPLIT);     // e2r: the span began one character earlier
                    const int fq = FO ? (int)__clz(FO) : -64;                        // q of the string start inside this lane-word
                    const int offA = c0 - lf_excl + 31, offB = fq;                   // string-relative index = off - q
                    int2 *dp = tst + ka + tp;
                    // the lowest token bit is the only one that may have no split below it inside the lane-word: the loop
                    // does not test for that, the pair is put right afterwards
                    const uint32_t lowb = evr & (0u - evr);
                    const bool fix_last = evr != 0u && (spr & (lowb - 1u)) == 0u;
                    while (evr) {
                        const int q = bfind32(evr);                                  // FLO
                        const uint32_t below = (1u << q) - 1u;
                        evr &= below;
                        const int off = q <= fq ? offB : offA;
                        const int qe = bfind32(spr & below);                         // FLO; the first split after the token
                        *dp++ = make_int2(off - q - (int)((e2r >> q) & 1u), off - qe);
                    }
                    if (fix_last) {
                        const int ql = bfind32(lowb);
                        const int off = ql <= fq ? offB : offA;
                        dp[-1].y = nextsplit >= 0 ? off - 31 + (nextsplit - c0) : -1;
                    }
                } else {
                uint32_t ev = E;
                int rank = 0;
                int cbase = lf_excl;
                while (ev) {
                    const int i = __ffs(ev) - 1; ev &= ev - 1;
                    const uint32_t fb = FO & mask_lt(i + 1);
                    if (fb) cbase = c0 + 31 - __clz(fb);
                    const uint32_t ab = (i == 31) ? 0u : (SPq & (0xFFFFFFFEu << i));
                    const int endc = ab ? c0 + __ffs(ab) - 1 : nextsplit;
                    const int sidx = c0 + i - (((SPLIT >> i) & 1u) ? 0 : 1) - cbase;
                    const int eidx = endc >= 0 ? endc - cbase : -1;
                    if (!direct) tst[ka + tp + rank] = make_int2(sidx, eidx);
                    else {
                        const long long kk = (long long)Ks + tp + rank;
                        if (kk < p.cap_tokens) {
                            if (eidx >= 0) reinterpret_cast<int2 *>(p.spans)[kk] = make_int2(sidx, eidx);
                            else p.spans[2 * kk] = sidx;          // still open: a later range writes the end
                        }
                    }
                    ++rank;
                }
                }
                // a range whose head is not chunk-aligned: its first split that follows a non-space character ends the
                // token left open by earlier ranges
                if (UNLIKELY(!lo_found && r > 0)) {
                    const uint32_t PSr = (Sraw << 1) | pk_ps(pk);
                    // (a range that ends at a closer also answers for the character after it: the next range begins at a
                    // closer then and does not come here -- a token that covers this whole range may end exactly there)
                    const uint32_t END = SPLIT & ~PSr & mask_lt(n) & range_mask(c0, c_lo, (r == p.nranges - 1 || closed) ? c_hi + 1 : c_hi);
                    if (END) {
                        const int i = __ffs(END) - 1;
                        if (ktok + tp + __popc(E & mask_lt(i)) == 0) {
                            const uint32_t fb = FO & mask_lt(i);      // string starts strictly before the split
                            const int cb = fb ? c0 + 31 - __clz(fb) : lf_excl;
                            const long long kk = (long long)K_in - 1;
                            if (kk >= 0 && kk < p.cap_tokens) p.spans[2 * kk + 1] = c0 + i - cb;
                        }
                    }
                }
                if (!direct) {
                    // stage slot j <-> pair (Ks - ka) + j of the output, so 16-byte chunks line up; the first and last chunk
                    // may hold one pair only
                    __syncwarp();
                    int2 *gb = reinterpret_cast<int2 *>(p.spans) + (Ks - (unsigned long long)ka);
                    const int tot = ka + ntok_step;
                    // whole chunks: slots 2c, 2c + 1 for c in [ka, tot / 2); the two single pairs at the ends by lane 0 / 1
                    const int cend = tot >> 1;
                    for (int c = ka + lane; c < cend; c += 32)
                        *reinterpret_cast<uint4 *>(gb + 2 * c) = *reinterpret_cast<const uint4 *>(tst + 2 * c);
                    if (lane == 0 && ka != 0 && tot > 1) gb[1] = tst[1];
                    if (lane == 1 && (tot & 1) != 0 && tot - 1 >= ka) gb[tot - 1] = tst[tot - 1];
                    __syncwarp();
                }
            }
            // ------------------------------------------------------------ per-token feature sums (latok.c:342-354)
            if (kFeats) {
                // Every split that follows a non-space character ends a token; the lane that holds it sums the token's
                // characters back to its first one (a split): population counts of the 25 feature planes over the part
                // inside this lane-word, then the open tails of the lanes / steps / ranges before it.
                auto plane_sums = [&](uint32_t frag, unsigned acc[7]) {
#pragma unroll
                    for (int f = 0; f < NFEAT; ++f) acc[f >> 2] += (unsigned)__popc(Q[f] & frag) << (8 * (f & 3));   // <= 32 each: no carry
                };
                uint32_t *tailsS = reinterpret_cast<uint32_t *>(tst);               // [32 lanes][8]: open tail sums + "holds a split"
                const int high = max(min(n, c_hi - c0), 0);                          // characters below c_hi (head zone included)
                const uint32_t SPw = SPLIT & mask_lt_nn(high);
                {
                    const uint32_t frag = SPw ? (mask_lt_nn(high) & ~mask_lt_nn(31 - __clz(SPw))) : mask_lt_nn(high);
                    unsigned tl[7] = {0, 0, 0, 0, 0, 0, 0};
                    plane_sums(frag, tl);
                    *reinterpret_cast<uint4 *>(tailsS + lane * 8) = make_uint4(tl[0], tl[1], tl[2], tl[3]);
                    *reinterpret_cast<uint4 *>(tailsS + lane * 8 + 4) = make_uint4(tl[4], tl[5], tl[6], SPw ? 1u : 0u);
                }
                __syncwarp();
                // four uint8 additions with wrap-around (latok.c:342-354 sums in uint8) in five instructions; __vadd4 takes ten
                auto vadd = [](unsigned x, unsigned y) -> unsigned {
                    return ((x & 0x7F7F7F7Fu) + (y & 0x7F7F7F7Fu)) ^ ((x ^ y) & 0x80808080u);
                };
                auto add8 = [&](unsigned acc[7], const uint4 &a, const uint4 &b) {
                    acc[0] = vadd(acc[0], a.x); acc[1] = vadd(acc[1], a.y); acc[2] = vadd(acc[2], a.z); acc[3] = vadd(acc[3], a.w);
                    acc[4] = vadd(acc[4], b.x); acc[5] = vadd(acc[5], b.y); acc[6] = vadd(acc[6], b.z);
                };
                // open tails of the lanes below `t`, then of the steps before (fc*), then of the ranges before (osum chain)
                // (a tail holds at most 32 of a feature and so does the part summed so far: the first six additions cannot carry
                // from one byte into the next and are plain ones)
                auto walk_lanes = [&](int t, unsigned acc[7], bool &hit) {
                    for (int it = 0; t >= 0 && !hit; --t, ++it) {
                        const uint4 a = *reinterpret_cast<const uint4 *>(tailsS + t * 8), b = *reinterpret_cast<const uint4 *>(tailsS + t * 8 + 4);
                        if (it < 6) { acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w; acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; }
                        else add8(acc, a, b);
                        hit = b.w != 0u;
                    }
                    if (!hit) {
                        add8(acc, make_uint4(fc[0], fc[1], fc[2], fc[3]), make_uint4(fc[4], fc[5], fc[6], 0u));
                        hit = fc_hit;
                    }
                    for (long long rr = r - 1; !hit && rr >= 0; --rr) {            // ranges that do not begin at a closer only
                        const Open o = wait_open(p.osum + rr, p.epoch, p.result);
                        add8(acc, o.lo, o.hi);
                        hit = o.has_split;
                    }
                };
                {
                    // Every token end (a split that follows a non-space character) closes the token with the next ordinal, so
                    // the token ends of a step are rows kr0 .. kr0 + nrows - 1 of the [T, 25] array, in the order of the lanes.
                    const uint32_t PSr = (Sraw << 1) | pk_ps(pk);
                    uint32_t ev = SPLIT & ~PSr & mask_lt(n) & range_mask(c0, c_lo + 1, c_hi + 1);
                    // ordinal of the lane's first row, relative to the first token of the range (-1: the token began in an earlier range)
                    const int kr_first = ev ? ktok + tp + __popc(E & mask_lt_nn(__ffs(ev) - 1)) - 1 : 0;
                    const unsigned has_ev = __ballot_sync(FULL, ev != 0u);
                    const int kr0 = __shfl_sync(FULL, kr_first, has_ev ? __ffs(has_ev) - 1 : 0);
                    const int nrows = has_ev ? __shfl_sync(FULL, kr_first + __popc(ev) - 1, 31 - __clz(has_ev)) - kr0 + 1 : 0;
                    if (nrows > 0 && nrows <= FLIST) {
                        // Rows in the order of their ordinals, 32 per trip, one per lane -- whatever lane-word a token ended in
                        // (the lane-words of a warp hold between none and a dozen token ends: a loop of every lane over its own
                        // ones runs as long as the busiest lane, and its rows would leave the warp as scattered words).
                        // (1) every lane lists its token ends: lane-word, position, position of the split the token began at
                        uint16_t *list = PS::scratch(tempS, js);         // (the step's state has been read)
                        {
                            uint32_t e = ev; int idx = kr_first - kr0;
                            while (e) {
                                const int i = __ffs(e) - 1; e &= e - 1;
                                const uint32_t below = SPLIT & mask_lt_nn(i);
                                const uint32_t st = below ? (uint32_t)(31 - __clz(below)) : 0u;
                                list[idx++] = (uint16_t)((uint32_t)lane | ((uint32_t)i << 5) | (st << 10) | (below ? 0x8000u : 0u));
                            }
                        }
                        uint8_t *rst = reinterpret_cast<uint8_t *>(tst) + 1024;            // row stage: 15 + 32 * 25 bytes, behind the tails
                        for (int c = lane; c < FSTAGE / 16; c += 32) *reinterpret_cast<uint4 *>(rst + 16 * c) = make_uint4(0, 0, 0, 0);
                        __syncwarp();
                        // (2) the rows that may be written (row capacity of the caller's array; no row in front of the first token)
                        const int jlo = max(0, f_kmin - kr0), jhi = min(nrows, f_kmax - kr0);
                        // (3) the rows of the step are consecutive bytes of the array, one stream: stream offset x <-> gS + x, the
                        // stage holds the stream from offset gw (a multiple of 16) on, the rows of the next trip begin at stage
                        // position sp < 16
                        const int rb0 = f_ph16 + NFEAT * (kr0 + jlo);                       // first byte of the step's rows, from f_g16
                        int8_t *gS = f_g16 + (rb0 & ~15);
                        const int head = rb0 & 15;                                          // bytes of the first chunk that belong to the rows before
                        int sp = head, gw = 0;
                        for (int jb = jlo; jb < jhi; jb += 32) {
                            const int j = jb + lane;
                            const bool valid = j < jhi;
                            const uint32_t rec = valid ? (uint32_t)list[j] : (uint32_t)lane;
                            const int w = (int)(rec & 31u), i = (int)((rec >> 5) & 31u), st = (int)((rec >> 10) & 31u);
                            bool hit = (rec & 0x8000u) != 0u;
                            const uint32_t frag = valid ? (mask_lt_nn(i) & ~mask_lt_nn(st)) : 0u;
                            unsigned acc[7] = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll
                            for (int f = 0; f < NFEAT; ++f)
                                acc[f >> 2] += (unsigned)__popc(__shfl_sync(FULL, Q[f], w) & frag) << (8 * (f & 3));
                            if (valid && !hit) walk_lanes(w - 1, acc, hit);
                            // the 32 rows of the trip, staged at their byte phase: five plain word stores per row, the two words a
                            // row shares with its neighbours by atomicOr
                            const int nv = min(32, jhi - jb), send = sp + NFEAT * nv;
                            if (valid) {
                                const int pb = sp + NFEAT * lane;
                                const uint32_t S = 8u * (uint32_t)(pb & 3);
                                uint32_t *wq = reinterpret_cast<uint32_t *>(rst) + (pb >> 2);
                                atomicOr(wq, acc[0] << S);                                   // (shares its word with the row before)
                                wq[1] = __funnelshift_l(acc[0], acc[1], S); wq[2] = __funnelshift_l(acc[1], acc[2], S);
                                wq[3] = __funnelshift_l(acc[2], acc[3], S); wq[4] = __funnelshift_l(acc[3], acc[4], S);
                                wq[5] = __funnelshift_l(acc[4], acc[5], S);
                                atomicOr(wq + 6, __funnelshift_l(acc[5], acc[6], S));       // (... with the row after)
                            }
                            __syncwarp();
                            // whole 16-byte chunks leave as such; what is left of the stream (< 16 bytes) moves to the front of the
                            // stage for the next trip.  Only the step's first chunk (when the rows before end inside it) and its
                            // last one are shared with another step / warp: their bytes go singly.
                            const bool firstt = jb == jlo, lastt = jb + 32 >= jhi;
                            const int nfull = send >> 4, e0 = send & ~15;
                            const bool head_part = firstt && head > 0;
                            if (lane < 16) {
                                if (head_part && lane >= head && lane < send) gS[lane] = (int8_t)rst[lane];
                                if (lastt && !(head_part && e0 == 0) && e0 + lane < send) gS[gw + e0 + lane] = (int8_t)rst[e0 + lane];
                            }
                            const uint4 zero4 = make_uint4(0, 0, 0, 0);
                            const uint4 va = *reinterpret_cast<const uint4 *>(rst + 16 * lane);
                            const uint4 vb = lane + 32 < FSTAGE / 16 ? *reinterpret_cast<const uint4 *>(rst + 16 * (lane + 32)) : zero4;
                            const uint4 vr = (lane == 0 && !lastt) ? *reinterpret_cast<const uint4 *>(rst + 16 * nfull) : zero4;
                            __syncwarp();
                            *reinterpret_cast<uint4 *>(rst + 16 * lane) = vr;                // (lane 0: the remainder; zero everywhere else)
                            if (lane + 32 < FSTAGE / 16) *reinterpret_cast<uint4 *>(rst + 16 * (lane + 32)) = zero4;
                            if (lane >= (head_part ? 1 : 0) && lane < nfull) *reinterpret_cast<uint4 *>(gS + gw + 16 * lane) = va;
                            if (lane + 32 < nfull) *reinterpret_cast<uint4 *>(gS + gw + 16 * (lane + 32)) = vb;
                            __syncwarp();
                            gw += 16 * nfull; sp = send & 15;
                        }
                    } else if (nrows > 0) {
                    // (more token ends in one step than the list holds: every lane writes the rows of its own token ends as one
                    // byte stream -- whole aligned words, the bytes of a row that do not fill a word wait in `carry` for the
                    // next row, the bytes that share a word with a row of another lane go singly)
                    if (ev) {
                        // ordinal of the first row, relative to the first token of the range (-1: the token began in an earlier range)
                        int kr = ktok + tp + __popc(E & mask_lt_nn(__ffs(ev) - 1)) - 1;
                        if (kr < f_kmin) { ev &= ev - 1; ++kr; }                      // (no token in front of it at all)
                        int o = f_phase + NFEAT * kr;                                   // byte offset of the row from the aligned base
                        int cnt = o & 3, wo = o >> 2;                                   // bytes waiting in `carry`; next whole word
                        uint32_t carry = 0;
                        bool first = true;
                        while (ev && kr < f_kmax) {
                            const int i = __ffs(ev) - 1; ev &= ev - 1;
                            unsigned acc[7] = {0, 0, 0, 0, 0, 0, 0};
                            const uint32_t below = SPLIT & mask_lt_nn(i);
                            bool hit = below != 0u;
                            plane_sums(mask_lt_nn(i) & ~mask_lt_nn(hit ? 31 - __clz(below) : 0), acc);
                            if (!hit) walk_lanes(lane - 1, acc, hit);
                            const uint32_t S = 8u * (uint32_t)cnt;
                            const uint32_t o0 = carry | (acc[0] << S);
                            const uint32_t o1 = __funnelshift_l(acc[0], acc[1], S), o2 = __funnelshift_l(acc[1], acc[2], S);
                            const uint32_t o3 = __funnelshift_l(acc[2], acc[3], S), o4 = __funnelshift_l(acc[3], acc[4], S);
                            const uint32_t o5 = __funnelshift_l(acc[4], acc[5], S), o6 = __funnelshift_l(acc[5], acc[6], S);
                            uint32_t *w = f_base + wo;
                            if (first && cnt) {                  // the low bytes of this word belong to the row before
                                uint8_t *b = reinterpret_cast<uint8_t *>(w);
                                if (cnt <= 1) b[1] = (uint8_t)(o0 >> 8);
                                if (cnt <= 2) b[2] = (uint8_t)(o0 >> 16);
                                b[3] = (uint8_t)(o0 >> 24);
                            } else w[0] = o0;
                            w[1] = o1; w[2] = o2; w[3] = o3; w[4] = o4; w[5] = o5;
                            if (cnt == 3) { w[6] = o6; carry = 0; wo += 7; } else { carry = o6; wo += 6; }
                            cnt = (cnt + 1) & 3;
                            first = false;
                            ++kr;
                        }
                        if (!first && cnt) {                     // the last bytes share their word with the next row
                            uint8_t *b = reinterpret_cast<uint8_t *>(f_base + wo);
                            b[0] = (uint8_t)carry;
                            if (cnt >= 2) b[1] = (uint8_t)(carry >> 8);
                            if (cnt == 3) b[2] = (uint8_t)(carry >> 16);
                        }
                    }
                    }
                }
                // the token open at the end of this step, for the steps after it (the same walk from the last lane, by all)
                {
                    unsigned acc[7] = {0, 0, 0, 0, 0, 0, 0};
                    bool hit = false;
                    for (int t = 31, it = 0; t >= 0 && !hit; --t, ++it) {
                        const uint4 a = *reinterpret_cast<const uint4 *>(tailsS + t * 8), b = *reinterpret_cast<const uint4 *>(tailsS + t * 8 + 4);
                        if (it < 7) { acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w; acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; }
                        else add8(acc, a, b);
                        hit = b.w != 0u;
                    }
                    if (!hit) { add8(acc, make_uint4(fc[0], fc[1], fc[2], fc[3]), make_uint4(fc[4], fc[5], fc[6], 0u)); hit = fc_hit; }
#pragma unroll
                    for (int g = 0; g < 7; ++g) fc[g] = acc[g];
                    fc_hit = hit;
                }
                __syncwarp();
            }
            ktok += ntok_step;
        }
        if (kFeats) {
            // the token open at the end of the range, for ranges that do not begin at a chunk closer
            if (lane == 0) publish_open(p.osum + r, p.epoch, fc_hit, fc);
        }
        if (r == p.nranges - 1 && lane == 0) {
            p.result->n_chars = G_in + (unsigned long long)n_own;
            p.result->n_tokens = K_in + (unsigned long long)ntok_range;
        }
    };

    // ================================================================================================= main loop
    // ticket of iteration k (slot k & 1): taken by the first warp that gets here, the others read it
    auto next_tile = [&](int k) -> int {
        const int s = k & 1;
        int t = 0;
        if (lane == 0) {
            const int old = atomicAdd(&ctl.tk_cnt[s], 1);
            if (old == NW - 1) st_vs32(&ctl.tk_cnt[s], 0);       // everybody has been here: ready for iteration k + 2
            if (old == 0) {
                const unsigned long long tk = atomicAdd(p.ticket, 1ull) - p.ticket_base;
                t = tk < (unsigned long long)ntiles_i ? (int)tk : ntiles_i;
                st_vs32(&ctl.tile_id[s], t);
                __threadfence_block();
                st_vs32(&ctl.tk_flag[s], k + 1);
            } else {
                Watchdog wd{SPIN_TICKET, false};
                while (ld_vs32(&ctl.tk_flag[s]) != k + 1 && !wd.expired(p.result)) {}
                t = ld_vs32(&ctl.tile_id[s]);
            }
        }
        return __shfl_sync(FULL, t, 0);
    };
    auto post = [&](int s, const RangeRec &a) {
        if (lane == 0) {
            ctl.rec[s][cw] = a;
            __threadfence_block();
        }
        __syncwarp();
        nb_arrive(BAR_AGG + s, NTH);
    };
    auto wait_window = [&](int b, unsigned &phase_bits) {
        Watchdog wd{SPIN_WINDOW, false};
        while (!mbar_try_wait(mbar + 2 * cw + b, (phase_bits >> b) & 1u) && !wd.expired(p.result)) {}
        phase_bits ^= 1u << b;
    };
    // write out tile `tile` (iteration kk): wait for its prefix, then pass D
    auto finish_tile = [&](int tile, int kk) {
        const int s = kk & 1;
        const long long r = (long long)tile * NW + cw;
        nb_sync(BAR_PRE + s, NTH);
        PROF5(4);
        // own prefix: the tile's plus the ranges before this one
        const Prefix in = advance(ctl.slot[s], sum_ranges(ctl.rec[s], cw, lane));
        output(r, s, in.G, in.K, in.base);
        PROF5(5);
    };

    unsigned phase_bits = 0;
    bool pending[2] = {false, false};
    int tile_cur = next_tile(0), tile_prev = -1;
    if (tile_cur < ntiles_i) pending[0] = begin_load((long long)tile_cur * NW + cw, 0);
    for (int k = 0;; ++k) {
        const int s = k & 1;
        if (tile_cur < ntiles_i) {
            build_map((long long)tile_cur * NW + cw, cw);
            if (s == 0 ? pending[0] : pending[1]) wait_window(s, phase_bits);
            __syncwarp();
            PROF5(0);
            post(s, analyze((long long)tile_cur * NW + cw, s, cw, 0, -1));
        } else {
            nb_arrive(BAR_AGG + s, NTH);                 // tells the service warp that the tickets have run out
        }
        if (tile_prev >= 0) finish_tile(tile_prev, k - 1);
        if (tile_cur >= ntiles_i) break;
        const int tile_next = next_tile(k + 1);
        bool pn = false;
        if (tile_next < ntiles_i) pn = begin_load((long long)tile_next * NW + cw, s ^ 1);
        if (s == 0) pending[1] = pn; else pending[0] = pn;
        tile_prev = tile_cur; tile_cur = tile_next;
    }
}

template <class Geom, bool kDefault, bool kFeats>
static cudaError_t launch_one(const Params &p, int grid, cudaStream_t s)
{
    const size_t smem = (size_t)plan<Geom>(p.tl, kDefault).total;
    static size_t configured = 0;
    if (configured < smem) {
        cudaError_t e = cudaFuncSetAttribute(tokenize5_kernel<Geom, kDefault, kFeats>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = smem;
    }
    tokenize5_kernel<Geom, kDefault, kFeats><<<grid, Geom::NTH, smem, s>>>(p);
    return cudaGetLastError();
}

template <class Geom, bool kDefault, bool kFeats>
static int ctas_one(const TableLayout &tl)
{
    int nb = 0;
    const size_t smem = (size_t)plan<Geom>(tl, kDefault).total;
    cudaFuncSetAttribute(tokenize5_kernel<Geom, kDefault, kFeats>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, tokenize5_kernel<Geom, kDefault, kFeats>, Geom::NTH, smem) != cudaSuccess) { cudaGetLastError(); return 1; }
    return nb < 1 ? 1 : nb;
}

// The entry points of one geometry.  Each geometry is instantiated in a translation unit of its own (LongGeometry in
// latok_tok5.cu, ShortGeometry in latok_tok5_short.cu), so the two compile in parallel.
template <class Geom>
int ctas_per_sm(const TableLayout &tl, bool is_default, bool want_feats)
{
    if constexpr (Geom::FEATS) {
        if (want_feats) return is_default ? ctas_one<Geom, true, true>(tl) : ctas_one<Geom, false, true>(tl);
    } else if (want_feats) return 0;                          // no such instantiation (tokenize5_plan never asks for it)
    return is_default ? ctas_one<Geom, true, false>(tl) : ctas_one<Geom, false, false>(tl);
}

template <class Geom>
cudaError_t launch(const Params &p, int grid, cudaStream_t s)
{
    const bool feats = (p.what & 4u) != 0u;
    if constexpr (Geom::FEATS) {
        if (feats) return p.rules.is_default ? launch_one<Geom, true, true>(p, grid, s) : launch_one<Geom, false, true>(p, grid, s);
    } else if (feats) return cudaErrorInvalidValue;
    return p.rules.is_default ? launch_one<Geom, true, false>(p, grid, s) : launch_one<Geom, false, false>(p, grid, s);
}

extern template int ctas_per_sm<LongGeometry>(const TableLayout &, bool, bool);
extern template cudaError_t launch<LongGeometry>(const Params &, int, cudaStream_t);
extern template int ctas_per_sm<ShortGeometry>(const TableLayout &, bool, bool);
extern template cudaError_t launch<ShortGeometry>(const Params &, int, cudaStream_t);

}  // namespace v5
}  // namespace latok
