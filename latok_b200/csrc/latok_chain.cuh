// latok_chain.cuh -- what crosses from one CTA of the tokenize kernel (latok_tok5.cuh) to another: the decoupled look-back
// chain (an aggregate and an inclusive-prefix record per tile), the open-token sums of token-feature mode (a record per
// range), the look-back walk over the chain, and the watchdog of every spin loop of the kernel.  latok_internal.h declares
// the records, because the host sizes and clears them; on the device only the codec below reads or writes them.
// Every record is written and read as whole 16-byte words with relaxed accesses; where a word says that the others are
// valid, the writer fences between them and the reader fences after it has seen that word.
#pragma once
#include "latok_device.cuh"

namespace latok {
namespace v5 {

// =====================================================================================================
// Watchdog: no spin loop may hang the device
// =====================================================================================================
constexpr unsigned SPIN_TICKET = 1u << 26;   // a compute warp waits for the tile ticket another warp of its CTA takes
constexpr unsigned SPIN_WINDOW = 1u << 24;   // ... for the TMA copy of its window
constexpr unsigned SPIN_CHAIN = 1u << 23;    // a warp waits for a record of another CTA

// Counts the rounds of one spin loop.  expired() is true once the loop must give up: after `limit` rounds or, for a wait
// on another CTA (`chain`), as soon as another watchdog has tripped (abort_flag, read every 1024 rounds).  It sets error
// bit 0 then, and a chain wait raises abort_flag, so that the CTAs waiting behind this one give up too.
struct Watchdog {
    unsigned limit;
    bool chain;
    unsigned spins = 0;
    __device__ __forceinline__ bool expired(Result *res)
    {
        if (++spins <= limit && !(chain && (spins & 1023u) == 0u && ld_volatile_u32(&res->abort_flag))) return false;
        atomicOr(&res->error, 1u);
        if (chain) st_volatile_u32(&res->abort_flag, 1u);
        return true;
    }
};

// =====================================================================================================
// Records
// =====================================================================================================
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

// A record belongs to this launch when it carries the launch's epoch (Params::epoch).  The host counts the epoch up per
// launch and clears every epoch-stamped buffer when it wraps, so a record left by an earlier launch reads as unpublished.
__device__ __forceinline__ bool this_launch(unsigned rec_epoch, unsigned epoch) { return rec_epoch == epoch; }

// What ranges add to the prefix (a tile's: AggRec; the ranges of a tile in front of one of them: sum_ranges()): their
// characters and tokens, and the position of their last string start relative to their first character (-1: none)
struct TileSum { int n, ntok, lft; };

// The prefix in front of a tile (lookback(), handed down to the compute warps) or behind it (IncRec): characters and tokens,
// the global index of the first character of the string open there, and the block-mask backlog crossing there
struct Prefix { unsigned long long G, base, K; int x; };
// the prefix behind ranges that add `t` to `pre` (x stays the caller's)
__device__ __forceinline__ Prefix advance(const Prefix &pre, const TileSum &t)
{
    Prefix r = pre;
    r.G = pre.G + (unsigned long long)t.n;
    r.K = pre.K + (unsigned long long)t.ntok;
    if (t.lft >= 0) r.base = pre.G + (unsigned long long)t.lft;
    return r;
}

// ---- aggregate record (AggRec), one per tile: status = epoch << 2 | state, then n | (lft + 1) << 16, ntok | v << 16
enum : unsigned {
    AGG_AGGREGATE = 1,   // the tile's sums and backlog for no backlog entering it
    AGG_INCLUSIVE = 2,   // ... and its inclusive prefix is in IncRec
};
static_assert(((EPOCH_MASK << 2) >> 2) == EPOCH_MASK, "the launch epoch fits the upper 30 bits of AggRec::status");
struct Agg {
    unsigned epoch, state;
    TileSum sum;         // of the tile, for no backlog entering it
    int v;               // the backlog it leaves, ditto
    // published by this launch, in `min_state` or a later state
    __device__ __forceinline__ bool published(unsigned launch_epoch, unsigned min_state) const
    {
        return this_launch(epoch, launch_epoch) && state >= min_state;
    }
};
__device__ __forceinline__ Agg read_agg(uint4 r)
{
    return Agg{r.x >> 2, r.x & 3u, TileSum{(int)(r.y & 0xFFFFu), (int)(r.z & 0xFFFFu), (int)(r.y >> 16) - 1}, (int)(r.z >> 16)};
}
// (the fields fit 16 bits: Geometry asserts that a tile holds fewer than 2^16 bytes; tokens, string starts and the
// backlog are bounded by its characters)
__device__ __forceinline__ void publish_agg(AggRec *rec, unsigned epoch, unsigned state, const TileSum &t, int v)
{
    st_rec(rec, make_uint4(epoch << 2 | state, (unsigned)t.n | (unsigned)(t.lft + 1) << 16, (unsigned)t.ntok | (unsigned)v << 16, 0u));
}
// spins until tile `idx` has published `min_state` or a later state in this launch (false: the watchdog gave up)
__device__ __forceinline__ bool wait_agg(const AggRec *agg, long long idx, unsigned epoch, unsigned min_state, Result *res)
{
    Watchdog wd{SPIN_CHAIN, true};
    while (!read_agg(ld_rec(agg + idx)).published(epoch, min_state))
        if (wd.expired(res)) return false;
    return true;
}

// ---- inclusive-prefix record (IncRec), one per tile: valid once the tile's AggRec is in state AGG_INCLUSIVE
static_assert(offsetof(IncRec, base) == 8 && offsetof(IncRec, K) == 16 && offsetof(IncRec, x) == 24, "IncRec: G base | K x");
__device__ __forceinline__ void publish_inc(IncRec *rec, const Prefix &inc)
{
    st_rec(&rec->G, make_uint4((unsigned)inc.G, (unsigned)(inc.G >> 32), (unsigned)inc.base, (unsigned)(inc.base >> 32)));
    st_rec(&rec->K, make_uint4((unsigned)inc.K, (unsigned)(inc.K >> 32), (unsigned)inc.x, 0u));
}
__device__ __forceinline__ Prefix read_inc(const IncRec *rec)
{
    const uint4 a = ld_rec(&rec->G), b = ld_rec(&rec->K);
    return Prefix{a.x | (unsigned long long)a.y << 32, a.z | (unsigned long long)a.w << 32, b.x | (unsigned long long)b.y << 32, (int)b.z};
}

// ---- open-token sums (OpenSums, token-feature mode), one per range: the feature sums of the token open at the end of the
// range (7 words of four uint8 sums) and whether that token holds a split; valid once `epoch` is this launch's
static_assert(offsetof(OpenSums, epoch) == 4 && offsetof(OpenSums, sums) == 16, "OpenSums: has_split epoch | sums");
__device__ __forceinline__ void publish_open(OpenSums *rec, unsigned epoch, bool has_split, const unsigned (&sums)[7])
{
    st_rec(&rec->sums[0], make_uint4(sums[0], sums[1], sums[2], sums[3]));
    st_rec(&rec->sums[4], make_uint4(sums[4], sums[5], sums[6], 0u));
    __threadfence();
    st_rec(rec, make_uint4(has_split ? 1u : 0u, epoch, 0u, 0u));
}
struct Open { uint4 lo, hi; bool has_split; };   // sums[0..3], sums[4..7]
__device__ __forceinline__ Open wait_open(const OpenSums *rec, unsigned epoch, Result *res)
{
    Watchdog wd{SPIN_CHAIN, true};
    uint4 h;
    do h = ld_rec(rec);
    while (!this_launch(h.y, epoch) && !wd.expired(res));
    __threadfence();
    return Open{ld_rec(&rec->sums[0]), ld_rec(&rec->sums[4]), h.x != 0u};
}

// =====================================================================================================
// Decoupled look-back (single chain, LB_WINDOW predecessors per step)
// =====================================================================================================
constexpr int LB_PER_LANE = 2;
constexpr int LB_WINDOW = 32 * LB_PER_LANE;

// Exclusive prefix of `tile` (warp 0, all lanes).  Walks back LB_WINDOW tiles at a time until it meets an
// inclusive prefix.  An aggregate is only valid for a tile that no block-mask backlog enters, i.e. when the
// inclusive prefix it is chained to carries no backlog and every aggregate between them leaves none
// (backlog-out for backlog-in 0 is stored in the record).  If that does not hold (rare: a whitespace chunk
// with several marks, or a chunk longer than the halo) the walk waits for the inclusive prefix of the tile
// right after the offending one -- that tile recomputes with its real backlog -- and starts over.
static __device__ Prefix lookback(long long tile, const Params &p, int lane)
{
    Prefix out{0, 0, 0, 0};
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
            Prefix rp{0, 0, 0, 0};                    // ... its prefix
            unsigned ln = 0, lk = 0, llf = 0; bool lhas = false; long long lviol = -1; int lastv = 0;
#ifdef LATOK_PROFILE
            long long _lt0 = clock64();
#endif
            // all records of this lane in flight at once; re-poll only the ones not yet published
            uint4 rec[LB_PER_LANE];
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) { rec[j] = make_uint4(0, 0, 0, 0); if (first + j >= 0) rec[j] = ld_rec(p.agg + (first + j)); }
            {
                Watchdog wd{SPIN_CHAIN, true};
                for (;;) {
                    bool pending = false;
#pragma unroll
                    for (int j = 0; j < LB_PER_LANE; ++j)
                        if (first + j >= 0 && !read_agg(rec[j]).published(p.epoch, AGG_AGGREGATE)) { rec[j] = ld_rec(p.agg + (first + j)); pending = true; }
                    if (!pending) break;
#ifdef LATOK_PROFILE
                    if (lane == 31) atomicAdd(&p.result->clocks.lb_repolls, 1ull);
#endif
                    if (wd.expired(p.result)) { ok = false; break; }
                }
            }
#ifdef LATOK_PROFILE
            if (lane == 31) { long long _t = clock64(); atomicAdd(&p.result->clocks.lb_poll, (unsigned long long)(_t - _lt0)); _lt0 = _t; }
#endif
            // the newest inclusive record of this lane: fetch its prefix
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) if (first + j >= 0 && read_agg(rec[j]).state == AGG_INCLUSIVE) rj = j;
            if (rj >= 0) {
                __threadfence();
                rp = read_inc(p.inc + (first + rj));
            }
#pragma unroll
            for (int j = 0; j < LB_PER_LANE; ++j) {
                const long long idx = first + j;
                if (idx < -1) continue;
                if (idx == -1) { if (rj < 0) { rj = j; rp = Prefix{0, 0, 0, 0}; } continue; }
                if (j <= rj) continue;                          // superseded by (or is) the inclusive record
                const Agg a = read_agg(rec[j]);
                if (a.sum.lft >= 0) { llf = ln + (unsigned)a.sum.lft; lhas = true; }
                ln += (unsigned)a.sum.n; lk += (unsigned)a.sum.ntok;
                if (a.v != 0 && idx != tile - 1) lviol = idx;   // its successor needs a real backlog
                if (idx == tile - 1) lastv = a.v;
            }
            const unsigned has_reset = __ballot_sync(0xFFFFFFFFu, rj >= 0);
            const int Lr = has_reset ? 31 - __clz(has_reset) : -1;
#ifdef LATOK_PROFILE
            if (lane == 0) { atomicAdd(&p.result->clocks.lb_windows, 1ull); if (Lr >= 0) atomicAdd(&p.result->clocks.lb_superseded, (unsigned long long)((31 - Lr) * LB_PER_LANE)); }
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
            if (lane == 31) { long long _t = clock64(); atomicAdd(&p.result->clocks.lb_sum, (unsigned long long)(_t - _lt0)); }
#endif
            if (Lr >= 0) {
                const unsigned long long G0 = __shfl_sync(0xFFFFFFFFu, rp.G, Lr), B0 = __shfl_sync(0xFFFFFFFFu, rp.base, Lr);
                const unsigned long long K0 = __shfl_sync(0xFFFFFFFFu, rp.K, Lr);
                const int x0 = __shfl_sync(0xFFFFFFFFu, rp.x, Lr);
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
        const bool ok2 = wait_agg(p.agg, viol + 1, p.epoch, AGG_INCLUSIVE, p.result);
        if (lane == 0) atomicAdd(&p.result->stats.lookback_restarts, 1ull);
        if (!ok2) return out;
    }
}

}  // namespace v5
}  // namespace latok
