/*
 * latok_oracle.c -- CPU restatement of LaTok's tokenization hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity checker for the CUDA
 * library in latok_b200/csrc.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load it; the product
 * (the latok_b200 package) never imports, links or calls anything under oracle/.
 *
 * Parity status: PINNED.  tests/test_oracle_cpu.py checks every function here
 * against (a) the reference's only golden vector, the executed notebook cell
 * notebooks/scratch/LaTokenizer.ipynb:1263-1430 (tests/golden/notebook_cell.json),
 * and (b) fixtures produced by the reference's own latok.c compiled in the build
 * container (oracle/Makefile target `ref`, generator tests/golden/make_golden.py).
 *
 * Each function cites the reference lines it restates (paths relative to the
 * reference checkout).  The code is a plain sequential restatement: one string
 * at a time, one character at a time, no vectorisation, no threads.
 *
 * The character-class lookup uses a sorted run list + binary search
 * (oracle/_gen/oracle_runs.h, generated from the committed ranges file), which
 * is structurally unrelated to the packed two-stage table the CUDA side uses.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "_gen/oracle_runs.h"

#define NFEAT 25

/* feature columns, latok/core/offsets.py:24-49 */
enum {
    F_ALPHA = 0, F_ALPHA_NUM, F_NUM, F_LOWER, F_UPPER, F_SPACE, F_SYMBOL, F_TWITTER,
    F_AT, F_COLON, F_SLASH, F_PERIOD,
    F_PREV_ALPHA, F_NEXT_ALPHA, F_PREV_ALPHA_NUM, F_NEXT_ALPHA_NUM, F_PREV_LOWER,
    F_NEXT_LOWER, F_PREV_SPACE, F_NEXT_SPACE, F_PREV_SYMBOL, F_NEXT_AT, F_NEXT_SLASH,
    F_AFTER_NEXT_ALPHA, F_AFTER_NEXT_SLASH
};

/* ---- A0: class lookup.  Restates gettyperecord (latok.c:15-29) composed with
 * the base-feature tests of latok.c:87-98; code points >= 0x110000 map to the
 * all-zero record exactly as latok.c:20-21 does. ---- */
uint16_t lo_base_features(uint32_t cp)
{
    if (cp >= 0x110000u) return 0;
    int lo = 0, hi = ORACLE_NRUNS - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (ORACLE_RUN_FIRST[mid] <= cp) lo = mid; else hi = mid - 1;
    }
    return ORACLE_RUN_FEAT[lo];
}

/* ---- A1: feature matrix.  Restates gen_parse_matrix, latok.c:31-138:
 * base columns :87-98, PREV/NEXT exchange :99-117, AFTER_NEXT :118-121,
 * end-of-string fills :122-134, row-0 initialisation :69-73. ---- */
void lo_parse_matrix(const uint32_t *cps, int64_t L, int8_t *m)
{
    for (int64_t i = 0; i < L; ++i) {
        int8_t *row = m + i * NFEAT;
        uint16_t f = lo_base_features(cps[i]);
        for (int k = 0; k < 12; ++k) row[k] = (int8_t)((f >> k) & 1);
        if (i > 0) {
            int8_t *prev = row - NFEAT;
            prev[F_NEXT_ALPHA] = row[F_ALPHA];
            prev[F_NEXT_ALPHA_NUM] = row[F_ALPHA_NUM];
            prev[F_NEXT_LOWER] = row[F_LOWER];
            prev[F_NEXT_SPACE] = row[F_SPACE];
            prev[F_NEXT_AT] = row[F_AT];
            prev[F_NEXT_SLASH] = row[F_SLASH];
            row[F_PREV_ALPHA] = prev[F_ALPHA];
            row[F_PREV_ALPHA_NUM] = prev[F_ALPHA_NUM];
            row[F_PREV_LOWER] = prev[F_LOWER];
            row[F_PREV_SPACE] = prev[F_SPACE];
            row[F_PREV_SYMBOL] = prev[F_SYMBOL];
        } else {
            /* start of string behaves as a space, latok.c:69-73,114-117 */
            row[F_PREV_ALPHA] = 0;
            row[F_PREV_ALPHA_NUM] = 0;
            row[F_PREV_LOWER] = 0;
            row[F_PREV_SPACE] = 1;
            row[F_PREV_SYMBOL] = 0;
        }
        if (i > 1) {
            int8_t *pp = row - 2 * NFEAT;
            pp[F_AFTER_NEXT_ALPHA] = row[F_ALPHA];
            pp[F_AFTER_NEXT_SLASH] = row[F_SLASH];
        }
        if (i + 1 >= L) {
            /* end of string behaves as a space, latok.c:122-130 */
            row[F_NEXT_ALPHA] = 0;
            row[F_NEXT_ALPHA_NUM] = 0;
            row[F_NEXT_AT] = 0;
            row[F_NEXT_LOWER] = 0;
            row[F_NEXT_SLASH] = 0;
            row[F_NEXT_SPACE] = 1;
        }
        if (i + 2 >= L) {
            row[F_AFTER_NEXT_SLASH] = 0;
            row[F_AFTER_NEXT_ALPHA] = 0;
        }
    }
}

/* ---- A2/A6: sum-of-products over selected rows.  Restates
 * combine_matrix_rows, latok.c:275-370.  `m` is addressed through byte strides
 * exactly like the NumPy array the reference receives (the tokenizer passes the
 * transposed view, strides (1,25)).  idx entries equal to -1 (255) are skipped
 * (:325,:347); arithmetic is unsigned char with wrap-around, reinterpreted as
 * int8 on return (:357-359).
 *   idx_cols > 0 : 2-D index matrix [idx_rows, idx_cols]   (:318-341)
 *   idx_cols == 0: 1-D index vector  [idx_rows]            (:342-354)
 * Like the reference, a 2-D row whose first entry is -1 keeps the previous
 * row's running product (an uninitialised read for the first row in the
 * reference); callers here always pass a valid first column. ---- */
void lo_combine_rows(const int8_t *m, int64_t n_cols, int64_t stride_r, int64_t stride_c,
                     const int8_t *idx, int idx_rows, int idx_cols, int8_t *out)
{
    const unsigned char *mu = (const unsigned char *)m;
    unsigned char *result = (unsigned char *)calloc((size_t)(n_cols > 0 ? n_cols : 1), 1);
    unsigned char *row = (unsigned char *)calloc((size_t)(n_cols > 0 ? n_cols : 1), 1);
    if (idx_cols > 0) {
        for (int i = 0; i < idx_rows; ++i) {
            for (int j = 0; j < idx_cols; ++j) {
                unsigned char r = (unsigned char)idx[i * idx_cols + j];
                if (r < 255) {
                    for (int64_t k = 0; k < n_cols; ++k) {
                        unsigned char v = mu[r * stride_r + k * stride_c];
                        if (j == 0) row[k] = v; else row[k] = (unsigned char)(row[k] * v);
                    }
                }
            }
            for (int64_t k = 0; k < n_cols; ++k) result[k] = (unsigned char)(result[k] + row[k]);
        }
    } else {
        for (int j = 0; j < idx_rows; ++j) {
            unsigned char r = (unsigned char)idx[j];
            if (r < 255)
                for (int64_t k = 0; k < n_cols; ++k)
                    result[k] = (unsigned char)(result[k] + mu[r * stride_r + k * stride_c]);
        }
    }
    for (int64_t k = 0; k < n_cols; ++k) out[k] = (int8_t)result[k];
    free(result);
    free(row);
}

/* ---- A3: block mask.  Restates gen_block_mask, latok.c:140-258, literally:
 * nonzero position lists (:178-201), no-mark case (:191-196), no-space case
 * (:211-216), the sequential merge in which each space serves at most one
 * pending mark (:218-238) and the tail (:239-244).  a1/a2 are strided int8. ---- */
void lo_block_mask(const int8_t *a1, int64_t s1, const int8_t *a2, int64_t s2, int64_t L, int8_t *out)
{
    int64_t n1 = 0, n2 = 0;
    int64_t *p1 = (int64_t *)malloc(sizeof(int64_t) * (size_t)(L > 0 ? L : 1));
    int64_t *p2 = (int64_t *)malloc(sizeof(int64_t) * (size_t)(L > 0 ? L : 1));
    for (int64_t i = 0; i < L; ++i) {
        if (a1[i * s1] != 0) p1[n1++] = i;
        if (a2[i * s2] != 0) p2[n2++] = i;
    }
    if (n1 == 0) {
        for (int64_t i = 0; i < L; ++i) out[i] = 1;
    } else if (n2 == 0) {
        for (int64_t i = 0; i < L; ++i) out[i] = 0;
    } else {
        for (int64_t i = 0; i < L; ++i) out[i] = 1;
        int64_t k1 = 0, v1 = p1[0], prev2 = 0;
        for (int64_t k2 = 0; k2 < n2; ++k2) {
            int64_t v2 = p2[k2];
            if (v2 >= v1) {
                for (int64_t q = prev2 + 1; q < v2; ++q) out[q] = 0;
                if (++k1 >= n1) break;
                v1 = p1[k1];
            }
            prev2 = v2;
        }
        if (k1 < n1)
            for (int64_t q = prev2 + 1; q < L; ++q) out[q] = 0;
    }
    free(p1);
    free(p2);
}

/* ---- A4: split mask.  Restates gen_split_mask, default_tokenizer.py:113-134:
 *   splits = comb(m.T, C_SPLIT) * block_mask(comb(m.T, C_MASK), m.T[SPACE]) + comb(m.T, C_SYM)
 *   splits[0] = 1
 * with int8 element-wise arithmetic.  Rule matrices are passed in
 * (build_combo_matrix layout, latok_utils.py:27-56) so user tokenizers can be
 * checked too.  Returns -1 for L == 0 (the reference raises IndexError, :132). ---- */
int lo_split_mask(const int8_t *m, int64_t L,
                  const int8_t *c_split, int sr, int sc,
                  const int8_t *c_mask, int mr, int mc,
                  const int8_t *c_sym, int yr, int yc, int8_t *splits)
{
    if (L <= 0) return -1;
    int8_t *a = (int8_t *)malloc((size_t)L), *b = (int8_t *)malloc((size_t)L);
    int8_t *bm = (int8_t *)malloc((size_t)L), *sy = (int8_t *)malloc((size_t)L);
    /* m.T has shape [25, L], strides (1, 25) */
    lo_combine_rows(m, L, 1, NFEAT, c_split, sr, sc, a);
    lo_combine_rows(m, L, 1, NFEAT, c_mask, mr, mc, b);
    lo_block_mask(b, 1, m + F_SPACE, NFEAT, L, bm);
    lo_combine_rows(m, L, 1, NFEAT, c_sym, yr, yc, sy);
    for (int64_t i = 0; i < L; ++i) splits[i] = (int8_t)((int8_t)(a[i] * bm[i]) + sy[i]);
    splits[0] = 1;
    free(a); free(b); free(bm); free(sy);
    return 0;
}

/* ---- A5: span read-off.  Restates the loop of tokenize/featurize,
 * default_tokenizer.py:148-158 and :174-191: nz = nonzero(splits); span k =
 * [nz[k], nz[k+1]) and the last one runs to L; a span is emitted iff
 * text[s:e].strip() is non-empty.  str.strip() removes leading/trailing
 * whitespace; the SPACE column marks exactly the str.isspace() code points
 * (checked in tests/test_oracle_cpu.py), so "non-empty after strip" == "some
 * character of the span is not SPACE".  spans[k] = untrimmed (s, e) as stored in
 * LaToken.start_idx/end_idx (:181-183,188-190); trimmed[k] = the (s', e') that
 * slice the stripped token text.  Returns the number of emitted spans. ---- */
int64_t lo_spans(const int8_t *splits, const int8_t *m, int64_t L, int32_t *spans, int32_t *trimmed)
{
    int64_t T = 0, s = -1;
    for (int64_t i = 0; i <= L; ++i) {
        if (i < L && splits[i] == 0) continue;
        if (s >= 0) {
            int64_t e = i, ts = s, te = e;
            while (ts < te && m[ts * NFEAT + F_SPACE]) ++ts;
            while (te > ts && m[(te - 1) * NFEAT + F_SPACE]) --te;
            if (te > ts) {
                spans[2 * T] = (int32_t)s;
                spans[2 * T + 1] = (int32_t)e;
                if (trimmed) { trimmed[2 * T] = (int32_t)ts; trimmed[2 * T + 1] = (int32_t)te; }
                ++T;
            }
        }
        s = i;
    }
    return T;
}

/* ---- A6: per-token feature vector.  Restates the 1-D branch of
 * combine_matrix_rows (latok.c:342-354) as called from featurize
 * (default_tokenizer.py:183,190): features[f] = sum over rows [s, e) of m[:, f]
 * in unsigned char with wrap, returned as int8.
 * Deliberate deviation (SURVEY.md Q5): the reference builds the row indices with
 * np.arange(..., dtype=int8), which wraps/raises for positions >= 128 and skips
 * position 255 (the -1 sentinel).  This restates the intended sum over all rows
 * of the span; it is identical to the reference wherever the reference is
 * defined (all positions <= 127 under NumPy 2, <= 254 under NumPy 1.15). ---- */
void lo_token_feats(const int8_t *m, const int32_t *spans, int64_t T, int8_t *feats)
{
    for (int64_t t = 0; t < T; ++t) {
        unsigned char acc[NFEAT];
        memset(acc, 0, sizeof acc);
        for (int64_t i = spans[2 * t]; i < spans[2 * t + 1]; ++i)
            for (int f = 0; f < NFEAT; ++f)
                acc[f] = (unsigned char)(acc[f] + (unsigned char)m[i * NFEAT + f]);
        for (int f = 0; f < NFEAT; ++f) feats[t * NFEAT + f] = (int8_t)acc[f];
    }
}

/* ---- Batch driver over code points: the per-string pipeline
 * _gen_parse_matrix -> gen_split_mask -> span loop -> token features
 * (default_tokenizer.py:137-191) applied to each string of a batch.  Empty
 * strings produce no characters and no tokens (the batch-API decision for
 * SURVEY.md Q1).  Any output pointer may be NULL to skip it.
 *   cps[char_off[s] .. char_off[s+1])  code points of string s
 *   splits  int8 [C]           matrix  int8 [C,25]
 *   spans   int32[T,2]         feats   int8 [T,25]
 *   tok_off int64[S+1]
 * Returns T. ---- */
int64_t lo_tokenize_batch_cps(const uint32_t *cps, const int64_t *char_off, int64_t S,
                              const int8_t *c_split, int sr, int sc,
                              const int8_t *c_mask, int mr, int mc,
                              const int8_t *c_sym, int yr, int yc,
                              int8_t *splits, int8_t *matrix, int32_t *spans, int64_t *tok_off,
                              int8_t *feats)
{
    int64_t T = 0, maxL = 1;
    for (int64_t s = 0; s < S; ++s)
        if (char_off[s + 1] - char_off[s] > maxL) maxL = char_off[s + 1] - char_off[s];
    int8_t *m = (int8_t *)malloc((size_t)maxL * NFEAT);
    int8_t *sp = (int8_t *)malloc((size_t)maxL);
    int32_t *tmp = (int32_t *)malloc(sizeof(int32_t) * 2 * (size_t)maxL);
    for (int64_t s = 0; s < S; ++s) {
        int64_t c0 = char_off[s], L = char_off[s + 1] - c0;
        if (tok_off) tok_off[s] = T;
        if (L == 0) continue;
        lo_parse_matrix(cps + c0, L, m);
        lo_split_mask(m, L, c_split, sr, sc, c_mask, mr, mc, c_sym, yr, yc, sp);
        int64_t n = lo_spans(sp, m, L, tmp, NULL);
        if (splits) memcpy(splits + c0, sp, (size_t)L);
        if (matrix) memcpy(matrix + c0 * NFEAT, m, (size_t)L * NFEAT);
        if (spans) memcpy(spans + 2 * T, tmp, sizeof(int32_t) * 2 * (size_t)n);
        if (feats) lo_token_feats(m, tmp, n, feats + T * NFEAT);
        T += n;
    }
    if (tok_off) tok_off[S] = T;
    free(m); free(sp); free(tmp);
    return T;
}

/* ---- UTF-8 front end for the CPU-baseline timing leg: decodes well-formed
 * (generalised: surrogates allowed, as Python's 'surrogatepass') UTF-8 into code
 * points, the job CPython's PyUnicode object has already done for the reference
 * (latok.c:47-55 reads code points via PyUnicode_READ).  Returns the number of
 * code points written; char_off[S+1] receives per-string code-point offsets. ---- */
int64_t lo_decode_utf8(const uint8_t *bytes, const int64_t *byte_off, int64_t S,
                       uint32_t *cps, int64_t *char_off)
{
    int64_t c = 0;
    for (int64_t s = 0; s < S; ++s) {
        char_off[s] = c;
        int64_t p = byte_off[s], e = byte_off[s + 1];
        while (p < e) {
            uint8_t b = bytes[p];
            uint32_t cp;
            int n;
            if (b < 0x80) { cp = b; n = 1; }
            else if (b >= 0xC0 && b < 0xE0) { cp = b & 0x1Fu; n = 2; }
            else if (b >= 0xE0 && b < 0xF0) { cp = b & 0x0Fu; n = 3; }
            else if (b >= 0xF0 && b < 0xF8) { cp = b & 0x07u; n = 4; }
            else { cp = 0x110000u; n = 1; }
            for (int k = 1; k < n; ++k)
                cp = (cp << 6) | ((p + k < e ? bytes[p + k] : 0) & 0x3Fu);
            cps[c++] = cp;
            p += n;
        }
    }
    char_off[S] = c;
    return c;
}
