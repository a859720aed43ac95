// latok_tokbytes.cu -- token spans as BYTE ranges of the packed UTF-8 buffer (SURVEY §8 f1).
//
// The reference materialises every token with `text[s:e].strip()` (default_tokenizer.py:151-158, 47-59 % of its
// CPU time).  Here the (start, end) code-point pairs written by the tokenize kernel are turned into byte offsets into
// the flat buffer, already trimmed the way strip() trims them (a span holds whitespace only at its first character,
// SURVEY §8 A5), so that utf8[b:e] IS the token text and an Arrow-style (data, begin, end) view needs no Python loop.
//
//   lead_count_kernel   characters (non-continuation bytes) per 32-byte word, as an exclusive prefix inside each
//                       group of 4096 words + one total per group (reads B, writes B/8)
//   group_scan_kernel   exclusive prefix of the group totals (one CTA)
//                       (these two are launch_char_prefix, which the parse matrix of latok_kernels.cu uses too)
//   token_bytes_kernel  one lane per token: ASCII-only strings map index -> byte directly; other strings find the
//                       word by a galloping search on the prefix and the byte by a select on the word's lead mask
// All three are HBM/L2-bound integer kernels; no tensor cores.
#include "latok_device.cuh"

namespace latok {

constexpr int TB_CHUNK = 16;             // blocks of 32 tokens per warp visit (one string search per chunk)

// bit j = byte j of the 32-byte word at `pos` begins a character (is not a UTF-8 continuation byte 10xxxxxx);
// bytes at and beyond n_bytes count as no character
__device__ __forceinline__ uint32_t lead_mask32(const uint8_t *in, long long pos, long long n_bytes)
{
    uint32_t w[8];
    if (pos + 32 <= n_bytes) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(in + pos)), b = __ldg(reinterpret_cast<const uint4 *>(in + pos + 16));
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            uint32_t v = 0x80808080u;
            for (int j = 0; j < 4; ++j)
                if (pos + 4 * q + j < n_bytes) v = (v & ~(0xFFu << (8 * j))) | ((uint32_t)in[pos + 4 * q + j] << (8 * j));
            w[q] = v;
        }
    }
    uint32_t m = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const uint32_t cont = (w[q] >> 7) & ~(w[q] >> 6) & 0x01010101u;      // 1 at the low bit of every continuation byte
        m |= ((cont * 0x10204080u) >> 28) << (4 * q);                        // the four flags gathered into a nibble
    }
    return ~m;
}

// position of the r-th (0-based) set bit of m; m has more than r bits set
__device__ __forceinline__ int select32(uint32_t m, unsigned r)
{
    int pos = 0;
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const unsigned c = (unsigned)__popc((m >> pos) & ((1u << w) - 1u));
        if (r >= c) { r -= c; pos += w; }
    }
    return pos;
}

// characters per 32-byte word as an exclusive prefix inside each group of TB_GROUP words + one total per group
__global__ void __launch_bounds__(1024) lead_count_kernel(const uint8_t *in, long long n_bytes, long long nwords,
                                                          unsigned *word_local, unsigned *group_tot)
{
    __shared__ unsigned wtot[32];
    __shared__ unsigned carry_s;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const long long w0 = (long long)blockIdx.x * TB_GROUP;
    for (int it = 0; it < TB_GROUP / 1024; ++it) {
        const long long w = w0 + it * 1024 + threadIdx.x;
        const unsigned c = w < nwords ? (unsigned)__popc(lead_mask32(in, w * TB_WORD, n_bytes)) : 0u;
        unsigned inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const unsigned t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        unsigned before = carry_s;
        for (int q = 0; q < warp; ++q) before += wtot[q];
        if (w < nwords) word_local[w] = before + inc - c;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = before + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) group_tot[blockIdx.x] = carry_s;
}

__global__ void __launch_bounds__(1024) group_scan_kernel(const unsigned *group_tot, long long ngroups, unsigned long long *group_pref)
{
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long carry_s;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (long long base = 0; base < ngroups; base += 1024) {
        const long long i = base + threadIdx.x;
        const unsigned long long v = i < ngroups ? group_tot[i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        unsigned long long before = carry_s;
        for (int w = 0; w < warp; ++w) before += wsum[w];
        if (i < ngroups) group_pref[i] = before + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = before + inc;
        __syncthreads();
    }
}

struct TokBytesParams {
    const uint8_t *in;
    long long n_bytes;
    const long long *offsets, *char_off, *tok_off;
    long long n_strings, n_tokens;
    const int32_t *spans;
    long long *out;                 // [T,2]
    const unsigned *word_local;
    const unsigned long long *group_pref;
    const uint8_t *table_blob;
    TableLayout tl;
};

// One lane per token, 32 consecutive tokens per warp step.  The token's string comes from a bisection over the CSR
// offsets of the (at most 32) strings that begin inside the warp's token block; a character index becomes a byte
// offset by a galloping search over the per-word character prefix, started where the string's bytes-per-character
// ratio says the character should be, then a select on the word's lead mask.
__global__ void __launch_bounds__(256) token_bytes_kernel(const TokBytesParams p)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    Tables tb;
    tb.ascii_feat = reinterpret_cast<const uint16_t *>(p.table_blob + p.tl.ascii_feat);
    tb.class_feat = reinterpret_cast<const uint16_t *>(p.table_blob + p.tl.class_feat);
    tb.stage1 = reinterpret_cast<const latok_stage1_t *>(p.table_blob + p.tl.stage1); tb.stage2 = p.table_blob + p.tl.stage2;
    tb.low_limit = p.tl.low_limit; tb.high_first = p.tl.high_first; tb.high_last = p.tl.high_last; tb.high_feat = p.tl.high_feat;
    auto wp = [&](long long w) -> unsigned long long { return p.group_pref[w / TB_GROUP] + p.word_local[w]; };
    const long long nblk = (p.n_tokens + 31) / 32;
    const long long nchunk = (nblk + TB_CHUNK - 1) / TB_CHUNK;
    for (long long ch = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ch < nchunk; ch += warps) {
      // string of the chunk's first token: last s with tok_off[s] <= k (strings without tokens are skipped over); the
      // blocks after it start from the string of the previous block's last token
      long long sf = 0;
      if (lane == 0) {
          const long long kb = ch * TB_CHUNK * 32;
          long long lo = 0, hi = p.n_strings;            // tok_off[lo] <= kb < tok_off[hi] = n_tokens
          while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (p.tok_off[mid] <= kb) lo = mid; else hi = mid; }
          sf = lo;
      }
      sf = __shfl_sync(0xFFFFFFFFu, sf, 0);
      const long long blk_end = (ch + 1) * TB_CHUNK < nblk ? (ch + 1) * TB_CHUNK : nblk;
      auto load_tv = [&](long long first) -> long long {
          const long long sj = first + 1 + lane;
          return sj <= p.n_strings ? p.tok_off[sj] : 0x7FFFFFFFFFFFFFFFLL;
      };
      auto load_sp = [&](long long k) -> int2 { return k < p.n_tokens ? reinterpret_cast<const int2 *>(p.spans)[k] : make_int2(0, 0); };
      long long tv = load_tv(sf);
      int2 sp = load_sp(ch * TB_CHUNK * 32 + lane);
      for (long long blk = ch * TB_CHUNK; blk < blk_end; ++blk) {
        const long long k = blk * 32 + lane;
        const bool live = k < p.n_tokens;
        // first tokens of the 32 strings after sf; the lane's string = sf + #{j : tok_off[sf + 1 + j] <= k}
        int cnt = 0;
#pragma unroll
        for (int w = 16; w >= 1; w >>= 1) {
            const long long v = __shfl_sync(0xFFFFFFFFu, tv, cnt + w - 1);
            if (v <= k) cnt += w;
        }
        long long s = sf + cnt;
        const long long tv31 = __shfl_sync(0xFFFFFFFFu, tv, 31);
        if (live && cnt == 31 && tv31 <= k) {                             // more than 32 strings begin in this block: search
            long long lo = s, hi = p.n_strings;
            while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (p.tok_off[mid] <= k) lo = mid; else hi = mid; }
            s = lo;
        }
        // next block: starts from the string of this block's last token; its loads are issued before this block's work
        const int2 sp_cur = sp;
        {
            const unsigned lv = __ballot_sync(0xFFFFFFFFu, live);
            sf = __shfl_sync(0xFFFFFFFFu, s, 31 - __clz(lv));
            if (blk + 1 < blk_end) { tv = load_tv(sf); sp = load_sp(k + 32); }
        }
        if (!live) continue;
        const long long o0 = p.offsets[s], o1 = p.offsets[s + 1], c0 = p.char_off[s], c1 = p.char_off[s + 1];
        const unsigned len_b = (unsigned)(o1 - o0), len_c = (unsigned)(c1 - c0);
        const bool ascii = len_b == len_c;
        // Everything below is relative to the string and fits 32 bits (spans are int32): word wr = the 32-byte word
        // w_lo + wr of the text, wp(wr) = characters of THE STRING in front of that word (<= 0 for wr = 0 when the string
        // begins inside the word), taken modulo 2^32 from the 64-bit prefix
        const long long w_lo = o0 / TB_WORD;
        const int nw = (int)((o1 - 1) / TB_WORD - w_lo);                  // the string's last word
        const unsigned c0lo = (unsigned)c0, skew = (unsigned)(o0 - w_lo * TB_WORD);
        const unsigned *gp_lo = reinterpret_cast<const unsigned *>(p.group_pref);      // low halves (little endian)
        auto wp = [&](int wr) -> int {
            const long long w = w_lo + wr;
            return (int)(gp_lo[2 * (w / TB_GROUP)] + p.word_local[w] - c0lo);
        };
        // byte position (relative to the string) of its character number idx; idx == length: the end of the string;
        // `hint`: a word known to begin at or before the character (-1: none)
        int word_of_last = -1;
        const float ratio = __fdividef((float)len_b, (float)len_c);
        auto byte_of = [&](unsigned idx, int hint) -> unsigned {
            if (ascii) return idx;
            if (idx >= len_c) return len_b;
            const int g = (int)idx;
            int lo = 0, hi = nw, step = 1;
            if (hint >= 0) lo = hint;
            else {
                int probe = (int)((skew + (unsigned)((float)idx * ratio)) / TB_WORD);
                probe = probe > hi ? hi : probe;
                if (wp(probe) <= g) lo = probe;
                else {
                    int h = probe;                                        // wp(h) > g
                    while (h - step > lo && wp(h - step) > g) { h -= step; step <<= 1; }
                    lo = h - step > lo ? h - step : lo;
                    hi = h - 1; step = hi - lo + 1;                       // (no galloping up below: bisect [lo, hi])
                }
            }
            if (step == 1) {                                              // gallop up from lo (wp(lo) <= g)
                while (lo + step <= hi && wp(lo + step) <= g) { lo += step; step <<= 1; }
                if (lo + step - 1 < hi) hi = lo + step - 1;
            }
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (wp(mid) <= g) lo = mid; else hi = mid - 1;
            }
            word_of_last = lo;
            const int pos = select32(lead_mask32(p.in, (w_lo + lo) * TB_WORD, p.n_bytes), (unsigned)(g - wp(lo)));
            return (unsigned)lo * TB_WORD + (unsigned)pos - skew;
        };
        long long bs = o0 + byte_of((unsigned)sp_cur.x, -1);
        const long long be = o0 + byte_of((unsigned)sp_cur.y, word_of_last);
        // strip(): only the span's first character can be whitespace
        if (bs < be) {
            const uint8_t *q = p.in + bs;
            const uint32_t b0 = q[0];
            uint32_t w;
            int len = 1;
            if (b0 < 0x80u) w = tb.ascii_feat[b0];
            else {
                len = b0 >= 0xF0u ? 4 : (b0 >= 0xE0u ? 3 : 2);
                uint32_t v = b0;
                for (int j = 1; j < len && bs + j < p.n_bytes; ++j) v |= (uint32_t)q[j] << (8 * j);
                w = mb_features(v, tb);
            }
            if ((w >> PL_SP) & 1u) bs = bs + len < be ? bs + len : be;
        }
        reinterpret_cast<longlong2 *>(p.out)[k] = make_longlong2(bs, be);
      }
    }
}

cudaError_t launch_char_prefix(const uint8_t *in, long long n_bytes, unsigned *word_local, unsigned *group_tot,
                               unsigned long long *group_pref, cudaStream_t s)
{
    const long long nwords = char_prefix_words(n_bytes), ngroups = char_prefix_groups(n_bytes);
    lead_count_kernel<<<(unsigned)ngroups, 1024, 0, s>>>(in, n_bytes, nwords, word_local, group_tot);
    group_scan_kernel<<<1, 1024, 0, s>>>(group_tot, ngroups, group_pref);
    return cudaGetLastError();
}

// after launch_char_prefix on the same stream
cudaError_t launch_token_bytes(const uint8_t *in, long long n_bytes, const long long *offsets, const long long *char_off,
                               const long long *tok_off, long long n_strings, long long n_tokens, const int32_t *spans,
                               long long *out, const unsigned *word_local, const unsigned long long *group_pref,
                               const uint8_t *table_blob, const TableLayout &tl, int n_sm, cudaStream_t s)
{
    if (n_strings == 0 || n_tokens == 0) return cudaSuccess;
    TokBytesParams p;
    p.in = in; p.n_bytes = n_bytes; p.offsets = offsets; p.char_off = char_off; p.tok_off = tok_off;
    p.n_strings = n_strings; p.n_tokens = n_tokens;
    p.spans = spans; p.out = out; p.word_local = word_local; p.group_pref = group_pref;
    p.table_blob = table_blob; p.tl = tl;
    const long long want = (((n_tokens + 31) / 32 + TB_CHUNK - 1) / TB_CHUNK + 7) / 8;
    const long long cap = (long long)n_sm * 8 * 8;
    token_bytes_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, s>>>(p);
    return cudaGetLastError();
}

long long char_prefix_words(long long n_bytes) { return n_bytes / TB_WORD + 1; }
long long char_prefix_groups(long long n_bytes) { return (char_prefix_words(n_bytes) + TB_GROUP - 1) / TB_GROUP; }

}  // namespace latok
