// latok_device.cuh -- device helpers of the kernels (latok_tok5.cuh: tokenize; latok_kernels.cu: parse matrix;
// latok_tokbytes.cu: token byte ranges): PTX wrappers, Unicode class look-up, the context features, the block-mask mark
// test and the backlog functions.  What crosses between the CTAs of the tokenize kernel (the look-back chain) is that
// kernel's own, in latok_chain.cuh; its look-ahead walk is in latok_tok5.cuh.
#pragma once
#include "latok_internal.h"
#include "latok_bits.h"

namespace latok {

constexpr int NEG = -(1 << 28);           // "-infinity" of the (max,+) backlog functions

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

// ---- block-mask mark of a character (the mask rows of combine_matrix_rows, latok.c:318-341; default_rules() fills C_MASK)
// (unrolled: constant row indices read the rows straight from the parameter bank and keep the caller's registers free)
__device__ __forceinline__ bool rule_mark(const RuleSet &rules, uint32_t w)
{
    bool mark = false;
#pragma unroll
    for (int i = 0; i < MAX_RULE_ROWS; ++i) mark |= i < rules.n_mask && (w & rules.mask[i]) == rules.mask[i];
    return mark;
}

// 4 feature bits -> 4 byte counters (bit k -> byte k)
__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

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
