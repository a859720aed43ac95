// latok_kernels.cu -- the parse matrix and the stand-alone helpers of the C ABI.
//
//   parse_matrix_kernel   the int8 [C,25] feature matrix (_gen_parse_matrix, latok.c:31-138): one warp per 32-byte word
//                         of the batch, one lane per byte; every character's 12 class bits plus its context bits
//   string_starts_kernel  the bitmap of string starts that tells parse_matrix_kernel where strings begin and end
//   tile_index_kernel     first string of every tokenize range, and the check of the offsets array
//   block_mask_kernel     stand-alone _gen_block_mask
//   combine_rows_kernel   stand-alone _combine_matrix_rows
//
// The tokenize kernel itself (split mask, spans, CSR offsets, token features) is in latok_tok5.cuh.
// No tensor cores: nothing here is a dense contraction.
#include "latok_device.cuh"

namespace latok {

// =====================================================================================================
// Bit o of `starts` is set when a string begins at byte o; offsets[n_strings] = n_bytes sets bit n_bytes, so the bitmap
// has n_bytes / 32 + 1 words (zeroed by the caller).  Empty strings set the bit of the string after them.
__global__ void string_starts_kernel(const long long *offsets, long long n_strings, uint32_t *starts, const Result *result)
{
    if (ld_volatile_u32(&result->error) & 2u) return;  // offsets failed validation in tile_index_kernel
    const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (s > n_strings) return;
    const long long o = offsets[s];
    atomicOr(&starts[o >> 5], 1u << (o & 31));
}

// bytes of the UTF-8 character whose lead byte is b
__device__ __forceinline__ int utf8_len(uint32_t b) { return b < 0xC0u ? 1 : b < 0xE0u ? 2 : b < 0xF0u ? 3 : 4; }

// One warp per 32-byte word w, lane l on byte 32 w + l.  Row of a character = characters in front of its word
// (launch_char_prefix) + lead bytes in front of it in the word.  The class words of the next and after-next
// characters come from the word itself or from the 8 bytes after it (lanes 0..7 also classify those), the previous
// character's from the word or from the 4 bytes in front of it (lanes 8..11).  The rows of a word are contiguous: they
// are staged in shared memory and written as consecutive bytes.
constexpr int PM_WARPS = 8;
__global__ void __launch_bounds__(PM_WARPS * 32) parse_matrix_kernel(const uint8_t *in, long long n_bytes, const uint32_t *starts,
                                                                     const unsigned *word_local, const unsigned long long *group_pref,
                                                                     const uint8_t *table_blob, const TableLayout tl, int8_t *matrix,
                                                                     const Result *result)
{
    __shared__ uint32_t rowS[PM_WARPS][32];
    if (ld_volatile_u32(&result->error) & 2u) return;  // offsets failed validation: the start bitmap was not built
    constexpr unsigned FULL = 0xFFFFFFFFu;
    Tables tb;
    tb.ascii_feat = reinterpret_cast<const uint16_t *>(table_blob + tl.ascii_feat);
    tb.class_feat = reinterpret_cast<const uint16_t *>(table_blob + tl.class_feat);
    tb.stage1 = reinterpret_cast<const latok_stage1_t *>(table_blob + tl.stage1); tb.stage2 = table_blob + tl.stage2;
    tb.low_limit = tl.low_limit; tb.high_first = tl.high_first; tb.high_last = tl.high_last; tb.high_feat = tl.high_feat;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *rows = rowS[warp];
    const long long nwords = n_bytes / TB_WORD + 1;
    for (long long w = (long long)blockIdx.x * PM_WARPS + warp; w < nwords; w += (long long)gridDim.x * PM_WARPS) {
        const long long base = w * TB_WORD, pos = base + lane;
        const long long xpos = lane < 8 ? base + 32 + lane : base - 12 + lane;
        const uint32_t b = pos < n_bytes ? in[pos] : 0x80u;
        const uint32_t xb = lane < 12 && xpos >= 0 && xpos < n_bytes ? in[xpos] : 0x80u;
        const bool lead = (b & 0xC0u) != 0x80u, xlead = (xb & 0xC0u) != 0x80u;
        const unsigned leads = __ballot_sync(FULL, lead), xleads = __ballot_sync(FULL, xlead);
        if (!leads) continue;
        const uint32_t cw = lead ? classify_at(in + pos, tb) : 0u, xw = xlead ? classify_at(in + xpos, tb) : 0u;
        // value v of the byte q = 0 .. 39 of the word (q >= 32: the bytes after it, held by lanes 0..7)
        auto at = [&](uint32_t v, uint32_t xv, int q) {
            const uint32_t a = __shfl_sync(FULL, v, q & 31), c = __shfl_sync(FULL, xv, (q - 32) & 31);
            return q < 32 ? a : c;
        };
        const int np = lane + utf8_len(b), ap = np + utf8_len(at(b, xb, np));     // next and after-next character
        const uint32_t nw = at(cw, xw, np), aw = at(cw, xw, ap);
        const unsigned below = leads & mask_lt(lane), xbelow = xleads & 0xF00u;
        const uint32_t pin = __shfl_sync(FULL, cw, below ? 31 - __clz(below) : 0);
        const uint32_t pout = __shfl_sync(FULL, xw, xbelow ? 31 - __clz(xbelow) : 0);
        const unsigned long long S = starts[w] | (w + 1 < nwords ? (unsigned long long)starts[w + 1] << 32 : 0ull);
        const bool F = (S >> lane) & 1u, L = (S >> np) & 1u, L2 = (S >> ap) & 1u;
        if (lead) rows[__popc(below)] = make_word(below ? pin : pout, cw, nw, aw, F, L, L2);
        __syncwarp();
        int8_t *dst = matrix + (group_pref[w / TB_GROUP] + word_local[w]) * NFEAT;
        for (int i = lane; i < __popc(leads) * NFEAT; i += 32) dst[i] = (int8_t)((rows[i / NFEAT] >> (i % NFEAT)) & 1u);
        __syncwarp();
    }
}

cudaError_t launch_parse_matrix(const uint8_t *in, long long n_bytes, const long long *offsets, long long n_strings,
                                uint32_t *starts, const unsigned *word_local, const unsigned long long *group_pref,
                                const uint8_t *table_blob, const TableLayout &tl, int8_t *matrix, const Result *result,
                                int n_sm, cudaStream_t s)
{
    const long long nwords = n_bytes / TB_WORD + 1;
    if (cudaError_t e = cudaMemsetAsync(starts, 0, (size_t)nwords * sizeof(uint32_t), s)) return e;
    string_starts_kernel<<<(unsigned)((n_strings + 256) / 256), 256, 0, s>>>(offsets, n_strings, starts, result);
    const long long want = (nwords + PM_WARPS - 1) / PM_WARPS, cap = (long long)n_sm * 8;
    parse_matrix_kernel<<<(unsigned)(want < cap ? want : cap), PM_WARPS * 32, 0, s>>>(in, n_bytes, starts, word_local, group_pref,
                                                                                    table_blob, tl, matrix, result);
    return cudaGetLastError();
}

// =====================================================================================================
// tile_first_str[t] = first string whose byte offset is >= t * TILE  (t = 0 .. ntiles; [ntiles] = S + 1).
// Also validates the offsets array.
__global__ void tile_index_kernel(const long long *offsets, long long n_strings, long long n_bytes,
                                  long long *first_str, long long ntiles, int TILE, Result *result)
{
    const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    long long t_begin = 0, t_end = -1;
    if (s <= n_strings) {
        const long long cur = offsets[s];
        const long long prev = s ? offsets[s - 1] : -1;
        bool bad = cur < 0 || cur > n_bytes || cur < prev || (s == 0 && cur != 0) || (s == n_strings && cur != n_bytes);
        if (bad) atomicOr(&result->error, 2u);
        else {
            t_begin = prev < 0 ? 0 : prev / TILE + 1;
            t_end = cur / TILE;
            if (t_end > ntiles - 1) t_end = ntiles - 1;
        }
        if (s == n_strings) first_str[ntiles] = n_strings + 1;
    }
    // short ranges: each lane writes its own; long ranges: the whole warp helps
    const long long len = t_end - t_begin + 1;
    if (len > 0 && len <= 4)
        for (long long t = t_begin; t <= t_end; ++t) first_str[t] = s;
    unsigned long_mask = __ballot_sync(0xFFFFFFFFu, len > 4);
    while (long_mask) {
        const int src = __ffs(long_mask) - 1; long_mask &= long_mask - 1;
        const long long b = __shfl_sync(0xFFFFFFFFu, t_begin, src), e = __shfl_sync(0xFFFFFFFFu, t_end, src);
        const long long ss = __shfl_sync(0xFFFFFFFFu, s, src);
        for (long long t = b + lane; t <= e; t += 32) first_str[t] = ss;
    }
}

cudaError_t launch_tile_index(const long long *offsets, long long n_strings, long long n_bytes,
                              long long *tile_first_str, long long ntiles, int tile_bytes, Result *result, cudaStream_t s)
{
    const int bs = 256;
    const long long n = n_strings + 1;
    const unsigned grid = (unsigned)((n + bs - 1) / bs);
    tile_index_kernel<<<grid, bs, 0, s>>>(offsets, n_strings, n_bytes, tile_first_str, ntiles, tile_bytes, result);
    return cudaGetLastError();
}

// =====================================================================================================
// Stand-alone _gen_block_mask(a1, a2) (latok.c:140-258) on caller arrays: one CTA, a forward sweep
// (backlog at every space) and a backward sweep (blank the chunks whose closing space is "hot").
constexpr int BM_NT = 1024;
__global__ void __launch_bounds__(BM_NT, 1)
block_mask_kernel(const int8_t *a1, long long s1, const int8_t *a2, long long s2, long long n, int8_t *out,
                  unsigned char *hot)
{
    __shared__ int scr[3 * 32 + 8];
    __shared__ int s_any_mark, s_any_space, s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_any_mark = 0; s_any_space = 0; s_carry = 0; }
    __syncthreads();
    bool am = false, as = false;
    for (long long i = tid; i < n; i += BM_NT) { am |= a1[i * s1] != 0; as |= a2[i * s2] != 0; }
    if (am) s_any_mark = 1;
    if (as) s_any_space = 1;
    __syncthreads();
    if (!s_any_mark || !s_any_space) {  // latok.c:191-196 / :211-216
        const int8_t v = s_any_mark ? 0 : 1;
        for (long long i = tid; i < n; i += BM_NT) out[i] = v;
        return;
    }
    const long long nchunks = (n + BM_NT - 1) / BM_NT;
    // forward: x = backlog; hot[i] = space i closes a blanked chunk
    for (long long ch = 0; ch < nchunks; ++ch) {
        const long long i = ch * BM_NT + tid;
        const bool mk = i < n && a1[i * s1] != 0, spc = i < n && a2[i * s2] != 0;
        Fn f = fn_id();
        if (mk) { f.u = 1; f.v = NEG + 1; }
        if (spc) { f.u = max(f.u - 1, NEG); f.v = max(f.v - 1, 0); }
        Fn inc = f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int ou = __shfl_up_sync(0xFFFFFFFFu, inc.u, d), ov = __shfl_up_sync(0xFFFFFFFFu, inc.v, d);
            if (lane >= d) inc = fn_compose(Fn{ou, ov}, inc);
        }
        int eu = __shfl_up_sync(0xFFFFFFFFu, inc.u, 1), ev = __shfl_up_sync(0xFFFFFFFFu, inc.v, 1);
        Fn wex = lane ? Fn{eu, ev} : fn_id();
        if (lane == 31) { scr[2 * warp] = inc.u; scr[2 * warp + 1] = inc.v; }
        __syncthreads();
        Fn base = fn_id(), tot = fn_id();
        for (int w = 0; w < BM_NT / 32; ++w) {
            Fn t = Fn{scr[2 * w], scr[2 * w + 1]};
            if (w < warp) base = fn_compose(base, t);
            tot = fn_compose(tot, t);
        }
        const int carry = s_carry;
        const int x = fn_apply(fn_compose(base, wex), carry) + (mk ? 1 : 0);
        if (i < n) hot[i] = (spc && x >= 1) ? 1 : 0;
        __syncthreads();
        if (tid == 0) s_carry = fn_apply(tot, carry);
        __syncthreads();
    }
    // backward: every non-space position takes the hot flag of the next space (or of the virtual end)
    if (tid == 0) s_carry = s_carry >= 1 ? 1 : 0;  // latok.c:239-244: marks left after the last space
    __syncthreads();
    for (long long ch = nchunks - 1; ch >= 0; --ch) {
        const long long i = ch * BM_NT + tid;
        const bool spc = i < n && a2[i * s2] != 0;
        const bool h = spc && hot[i];
        const unsigned H = __ballot_sync(0xFFFFFFFFu, spc), FH = __ballot_sync(0xFFFFFFFFu, h);
        if (lane == 0) { scr[2 * warp] = H != 0u; scr[2 * warp + 1] = H ? ((FH >> (__ffs(H) - 1)) & 1u) : 0u; }
        __syncthreads();
        const int carry = s_carry;
        int cin;
        const unsigned above = lane == 31 ? 0u : (H & (0xFFFFFFFFu << (lane + 1)));
        if (above) cin = (FH >> (__ffs(above) - 1)) & 1u;
        else {
            cin = carry;
            for (int w2 = warp + 1; w2 < BM_NT / 32; ++w2)
                if (scr[2 * w2]) { cin = scr[2 * w2 + 1]; break; }
        }
        if (i < n) out[i] = (spc || i == 0) ? 1 : (cin ? 0 : 1);
        int first = carry;
        for (int w2 = 0; w2 < BM_NT / 32; ++w2)
            if (scr[2 * w2]) { first = scr[2 * w2 + 1]; break; }
        __syncthreads();
        if (tid == 0) s_carry = first;
        __syncthreads();
    }
}

cudaError_t launch_block_mask(const int8_t *a1, long long s1, const int8_t *a2, long long s2, long long n,
                              int8_t *out, unsigned char *scratch, cudaStream_t s)
{
    if (n <= 0) return cudaSuccess;
    block_mask_kernel<<<1, BM_NT, 0, s>>>(a1, s1, a2, s2, n, out, scratch);
    return cudaGetLastError();
}

// =====================================================================================================
// Stand-alone _combine_matrix_rows(m, idxs) (latok.c:275-370): one thread per output column.
__global__ void combine_rows_kernel(const int8_t *m, long long m_rows, long long m_cols, long long sr, long long sc,
                                    const int8_t *idx, int idx_rows, int idx_cols, int8_t *out)
{
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= m_cols) return;
    const unsigned char *mu = reinterpret_cast<const unsigned char *>(m);
    unsigned char result = 0;
    if (idx_cols > 0) {          // "and" within a row, "or" across rows (:318-341)
        unsigned char row = 0;
        for (int i = 0; i < idx_rows; ++i) {
            for (int j = 0; j < idx_cols; ++j) {
                const unsigned char r = (unsigned char)idx[i * idx_cols + j];
                if (r < 255 && r < m_rows) {
                    const unsigned char v = mu[r * sr + k * sc];
                    row = j == 0 ? v : (unsigned char)(row * v);
                }
            }
            result = (unsigned char)(result + row);
        }
    } else {                     // 1-D: plain sum of the listed rows (:342-354)
        for (int j = 0; j < idx_rows; ++j) {
            const unsigned char r = (unsigned char)idx[j];
            if (r < 255 && r < m_rows) result = (unsigned char)(result + mu[r * sr + k * sc]);
        }
    }
    out[k] = (int8_t)result;
}

cudaError_t launch_combine_rows(const int8_t *m, long long m_rows, long long m_cols, long long stride_r,
                                long long stride_c, const int8_t *idx, int idx_rows, int idx_cols,
                                int8_t *out, cudaStream_t s)
{
    if (m_cols <= 0) return cudaSuccess;
    const int bs = 256;
    combine_rows_kernel<<<(unsigned)((m_cols + bs - 1) / bs), bs, 0, s>>>(m, m_rows, m_cols, stride_r, stride_c, idx,
                                                                         idx_rows, idx_cols, out);
    return cudaGetLastError();
}

}  // namespace latok
