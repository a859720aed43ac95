// latok_bits.h -- pure per-lane bit-plane primitives of the v5 tokenize kernel (host + device).
//
// A "lane-word" is 32 consecutive input bytes held by one thread.  Everything below works on 32-bit planes:
// bit j of a plane belongs to byte j (byte space) or, after squeeze_planes, to the lane-word's j-th character
// (character space).  The functions are __host__ __device__ so tests/test_host_cpu.py can check them on the CPU
// against the generated class table (tools/bits_selftest.cu) -- they contain no table look-ups.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define LATOK_HD __host__ __device__ __forceinline__
#else
#define LATOK_HD inline
#endif

namespace latok {

// feature plane numbers = the first twelve columns of the parse matrix (offsets.py:24-35 / latok.h:24-35)
enum { PL_A = 0, PL_N = 1, PL_NUM = 2, PL_LO = 3, PL_UP = 4, PL_SP = 5, PL_SY = 6, PL_TW = 7, PL_AT = 8, PL_CO = 9,
       PL_SL = 10, PL_PE = 11, NBASE = 12 };

LATOK_HD uint32_t bits_byte_perm(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t v = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((v >> (8 * ((sel >> (4 * i)) & 7u))) & 0xFFu) << (8 * i);
    return r;
#endif
}

// (a & M) | (b & ~M) for a constant mask M
template <uint32_t M>
LATOK_HD uint32_t bits_select(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__) && !defined(LATOK_NO_LOP3_ASM)
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(a), "r"(b), "n"(M));     // c ? a : b
    return r;
#else
    return (a & M) | (b & ~M);
#endif
}

// 32 bytes (w[i] = bytes 4i..4i+3, little endian) -> 8 bit-planes: bit j of b[k] = bit k of byte j.
// Step 1: two 4x4 byte transposes put byte (8q + r) into byte q of word r, so that bit position 8q + r' of
// register k after the 8x8 bit transpose (three delta-swap stages between register pairs) is character 8q + r'.
LATOK_HD void bytes_to_planes(const uint32_t w[8], uint32_t b[8])
{
    uint32_t u[8];
    {
        const uint32_t t0 = bits_byte_perm(w[0], w[2], 0x5140), t1 = bits_byte_perm(w[0], w[2], 0x7362);
        const uint32_t t2 = bits_byte_perm(w[4], w[6], 0x5140), t3 = bits_byte_perm(w[4], w[6], 0x7362);
        u[0] = bits_byte_perm(t0, t2, 0x5410); u[1] = bits_byte_perm(t0, t2, 0x7632);
        u[2] = bits_byte_perm(t1, t3, 0x5410); u[3] = bits_byte_perm(t1, t3, 0x7632);
    }
    {
        const uint32_t t0 = bits_byte_perm(w[1], w[3], 0x5140), t1 = bits_byte_perm(w[1], w[3], 0x7362);
        const uint32_t t2 = bits_byte_perm(w[5], w[7], 0x5140), t3 = bits_byte_perm(w[5], w[7], 0x7362);
        u[4] = bits_byte_perm(t0, t2, 0x5410); u[5] = bits_byte_perm(t0, t2, 0x7632);
        u[6] = bits_byte_perm(t1, t3, 0x5410); u[7] = bits_byte_perm(t1, t3, 0x7632);
    }
    // 8x8 bit transpose inside every byte column: element (register r, bit k) <-> (register k, bit r)
    // (bits_select: one LOP3 per half of a swap -- the compiler's own lowering of the masked form takes two)
#define LATOK_SWAP(i, j, s, m)                                       \
    {                                                                \
        const uint32_t lo = bits_select<(m)>(u[i], u[j] << (s));     \
        const uint32_t hi = bits_select<(m)>(u[i] >> (s), u[j]);     \
        u[i] = lo; u[j] = hi;                                        \
    }
    LATOK_SWAP(0, 4, 4, 0x0F0F0F0Fu) LATOK_SWAP(1, 5, 4, 0x0F0F0F0Fu) LATOK_SWAP(2, 6, 4, 0x0F0F0F0Fu) LATOK_SWAP(3, 7, 4, 0x0F0F0F0Fu)
    LATOK_SWAP(0, 2, 2, 0x33333333u) LATOK_SWAP(1, 3, 2, 0x33333333u) LATOK_SWAP(4, 6, 2, 0x33333333u) LATOK_SWAP(5, 7, 2, 0x33333333u)
    LATOK_SWAP(0, 1, 1, 0x55555555u) LATOK_SWAP(2, 3, 1, 0x55555555u) LATOK_SWAP(4, 5, 1, 0x55555555u) LATOK_SWAP(6, 7, 1, 0x55555555u)
#undef LATOK_SWAP
#pragma unroll
    for (int k = 0; k < 8; ++k) b[k] = u[k];
}

// The twelve base features of the ASCII characters as boolean functions of the byte's bit-planes
// (gettyperecord + the tests of latok.c:87-98 restricted to code points < 0x80; the truth table is
// LATOK_ASCII_FEAT in _gen/latok_tables.h and tools/bits_selftest.cu checks all 256 byte values against it).
// Bytes >= 0x80 get no features here; multi-byte characters are patched in from the class table.
LATOK_HD void classify_ascii(const uint32_t b[8], uint32_t P[NBASE])
{
    const uint32_t b0 = b[0], b1 = b[1], b2 = b[2], b3 = b[3], b4 = b[4], b5 = b[5], b6 = b[6], b7 = b[7];
    const uint32_t asc = ~b7;
    const uint32_t nz5 = b4 | b3 | b2 | b1 | b0;                  // low five bits != 0
    const uint32_t gt26 = b4 & b3 & (b2 | (b1 & b0));              // low five bits in 27..31
    const uint32_t alpha = asc & b6 & nz5 & ~gt26;                 // A-Z a-z
    const uint32_t upper = alpha & ~b5, lower = alpha & b5;
    const uint32_t num = asc & ~b6 & b5 & b4 & ~(b3 & (b2 | b1));  // 0-9
    const uint32_t alnum = alpha | num;
    const uint32_t row0 = asc & ~b6 & ~b5;                          // 0x00-0x1F
    const uint32_t sp_a = row0 & ~b4 & b3 & ~(b2 & b1) & (b2 | b1 | b0);   // 0x09-0x0D
    const uint32_t sp_b = row0 & b4 & b3 & b2;                      // 0x1C-0x1F
    const uint32_t is20 = asc & ~b6 & b5 & ~nz5;                    // ' '
    const uint32_t space = sp_a | sp_b | is20;
    const uint32_t is7f = b6 & b5 & b4 & b3 & b2 & b1 & b0;
    const uint32_t symbol = asc & (b6 | b5) & ~alnum & ~is20 & ~is7f;   // printable, not alphanumeric, not space
    const uint32_t r2 = asc & ~b6 & b5 & ~b4;                       // 0x20-0x2F
    const uint32_t lo_e = b3 & b2 & b1;                             // low nibble 0xE / 0xF
    const uint32_t period = r2 & lo_e & ~b0;                        // '.'
    const uint32_t slash = r2 & lo_e & b0;                          // '/'
    const uint32_t colon = asc & ~b6 & b5 & b4 & b3 & ~b2 & b1 & ~b0;   // ':'
    const uint32_t at = asc & b6 & ~b5 & ~nz5;                      // '@'
    const uint32_t hash = r2 & ~b3 & ~b2 & b1 & b0;                 // '#'
    const uint32_t dollar = r2 & ~b3 & b2 & ~b1 & ~b0;              // '$'
    const uint32_t caret = asc & b6 & ~b5 & b4 & b3 & b2 & b1 & ~b0;    // '^'
    P[PL_A] = alpha; P[PL_N] = alnum; P[PL_NUM] = num; P[PL_LO] = lower; P[PL_UP] = upper; P[PL_SP] = space;
    P[PL_SY] = symbol; P[PL_TW] = hash | dollar | at | caret; P[PL_AT] = at; P[PL_CO] = colon; P[PL_SL] = slash;
    P[PL_PE] = period;
}

LATOK_HD uint32_t bits_clz(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return (uint32_t)__clz((int)x);
#else
    return x ? (uint32_t)__builtin_clz(x) : 32u;
#endif
}
LATOK_HD uint32_t bits_brev(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __brev(x);
#else
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
    return (x >> 16) | (x << 16);
#endif
}
LATOK_HD uint32_t bits_low(int k) { return k <= 0 ? 0u : (k >= 32 ? 0xFFFFFFFFu : ((1u << k) - 1u)); }   // low k bits

// byte space -> character space: keep the positions in `lead`, squeeze the others out (stable).  `vmask` = the
// byte positions that hold data.  NP planes + one extra word (the string-start map) move together.
template <int NP>
LATOK_HD void squeeze_planes(uint32_t P[NP], uint32_t &F, uint32_t lead, uint32_t vmask)
{
    // (the planes hold nothing at continuation bytes: the ASCII classifier leaves bytes >= 0x80 empty and multi-byte
    // characters are patched in at their lead byte; only the string-start map can point at one, in malformed input)
    uint32_t del = lead ? (~lead & vmask) : 0u;
    F &= lead;
    while (del) {
        const int top = 31 - (int)bits_clz(del);
        const int r = (int)bits_clz(~(del << (31 - top)));   // run of deleted positions ending at `top`
        const int c = top - r;                                 // last kept position below the run (may be -1)
        const uint32_t keep = bits_low(c + 1);
#pragma unroll
        for (int f = 0; f < NP; ++f) P[f] = (P[f] & keep) | ((P[f] >> r) & ~keep);
        F = (F & keep) | ((F >> r) & ~keep);
        del &= keep;
    }
}

// The same result by a five-stage parallel-suffix compress (cost independent of the number of deleted runs):
// stage i moves every kept bit whose count of deleted positions below it has bit i set down by 2^i.
#ifndef LATOK_SQUEEZE_RUNS
#define LATOK_SQUEEZE_RUNS 4      // more deleted runs than this in some lane-word of the warp: use the compress
#endif
template <int NP>
LATOK_HD void squeeze_planes_log(uint32_t P[NP], uint32_t &F, uint32_t lead)
{
    F &= lead;
    if (!lead) return;
    uint32_t m = lead, mk = ~lead << 1;
#pragma unroll
    for (int f = 0; f < NP; ++f) P[f] &= lead;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        uint32_t mp = mk ^ (mk << 1);
        mp ^= mp << 2; mp ^= mp << 4; mp ^= mp << 8; mp ^= mp << 16;
        const uint32_t mv = mp & m;
        m = (m ^ mv) | (mv >> (1 << i));
#pragma unroll
        for (int f = 0; f < NP; ++f) { const uint32_t t = P[f] & mv; P[f] = (P[f] ^ t) | (t >> (1 << i)); }
        { const uint32_t t = F & mv; F = (F ^ t) | (t >> (1 << i)); }
        mk &= ~mp;
    }
}

// ---- block mask, common case (latok.c:218-244 when no whitespace chunk holds more than one mark) -------------
// CL = characters that close a chunk (space / last character of a string), M = marks, cin = a mark is pending in
// the chunk that is open at the first character.
// Returns T = (M & ~CL) + ~CL + cin: T & CL are the closers reached with a pending mark ("hot"), M & ~CL & T are
// marks that found another mark pending in their chunk, and the carry out of bit 31 (cout) says a mark is still
// pending after the last character.  Positions that hold no character must be 0 in CL and M; they pass the carry on.
// The result is exact unless (M & ~CL & T) | (M & CL) != 0; then the exact evaluation must be used.  A mark on a
// closer (never under the default rules; custom mask rows can fire on a space or on the last character of a
// string) is dropped here, while latok.c:218-244 takes it before that closer, which makes the closer hot.
LATOK_HD uint32_t chunk_carry(uint32_t M, uint32_t CL, uint32_t cin, uint32_t &cout)
{
    const uint32_t R = ~CL, A = M & R;
    const uint64_t t = (uint64_t)A + (uint64_t)R + (uint64_t)cin;
    cout = (uint32_t)(t >> 32);
    return (uint32_t)t;
}

// Characters blanked by the block mask: a hot closer and the run of non-closers below it; `bin` = the first
// closer ABOVE this lane-word is hot (so the open run at the top is blanked too).
LATOK_HD uint32_t flood_down(uint32_t HOT, uint32_t CL, uint32_t bin)
{
    const uint32_t Hr = bits_brev(HOT), Rr = ~bits_brev(CL);
    const uint32_t seed = ((Hr << 1) | bin) & Rr;
    const uint32_t Zr = Rr & ~(seed + Rr);
    return bits_brev(Zr) | HOT;
}

}  // namespace latok
