/*
 * latok_b200.h -- C ABI of liblatok_b200.so: LaTok's tokenization hot path on one B200.
 *
 * This is the boundary a binding of the reference would call instead of its CPython extension
 * module `latok.latok` (reference: latok/core/src/latok/latok.c:373-378, built by setup.py:10-17)
 * and instead of the array-producing part of latok/core/default_tokenizer.py:113-191.
 * Plain pointers and sizes only; no Python, NumPy or torch types cross it.
 *
 * Conventions
 *   - every function returns 0 (LATOK_B200_OK) or a LATOK_B200_E* code; the message for the last
 *     failure on the calling thread is latok_b200_last_error().  This replaces
 *     PyErr_SetString(PyExc_ValueError, ...) + NULL (latok.c:40-50,151-171,292-312).
 *   - an engine owns one device, its streams, the Unicode class table and all device / pinned
 *     staging memory.  An engine is not thread-safe: one host thread at a time (the Python
 *     wrapper holds a lock per engine); use one engine per GPU.
 *   - text is a flat UTF-8 byte buffer plus an int64 offsets array of n_strings+1 entries
 *     (offsets[0]==0, non-decreasing, offsets[n_strings]==total bytes).  The bytes must be
 *     well-formed UTF-8; lone surrogates encoded the way Python's 'surrogatepass' does are
 *     accepted (they are legal in the `str` the reference reads, latok.c:47-55).
 *   - all character positions in the outputs are CODE-POINT indices, as in the reference
 *     (latok.c:53,58; default_tokenizer.py:148-158), not byte offsets.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     LATOK_B200_ECUDA.
 */
#ifndef LATOK_B200_H
#define LATOK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LATOK_B200_API __attribute__((visibility("default")))
#else
#define LATOK_B200_API
#endif

#define LATOK_B200_ABI_VERSION 2
#define LATOK_B200_NUM_FEATURES 25 /* FEATURE_COUNT, latok.h:49 / offsets.py:49 */

enum {
    LATOK_B200_OK = 0,
    LATOK_B200_EINVAL = 1,    /* bad argument (maps to ValueError) */
    LATOK_B200_ECUDA = 2,     /* CUDA runtime failure / no device (maps to RuntimeError) */
    LATOK_B200_ENOMEM = 3,    /* host or device allocation failed */
    LATOK_B200_ESTATE = 4,    /* call out of order (e.g. fetch before submit) */
    LATOK_B200_EINTERNAL = 5  /* device-side watchdog or consistency check tripped */
};

/* what one submit computes; OR them together */
enum {
    LATOK_B200_SPLITS = 1, /* int8 split mask per character    (gen_split_mask, default_tokenizer.py:113-134) */
    LATOK_B200_SPANS = 2,  /* token spans + per-string CSR      (tokenize/featurize loop, :148-158,:174-191)   */
    LATOK_B200_FEATS = 4,  /* int8[T,25] per-token feature sums (featurize, :181-191 -> latok.c:342-354)       */
    LATOK_B200_MATRIX = 8, /* int8[C,25] feature matrix         (_gen_parse_matrix, latok.c:31-138)            */
    LATOK_B200_SPANS16 = 16 /* compact results: spans come back as uint16[T,2] (half the device -> host bytes);
                               implies SPANS; fetch fails with EINVAL if a string has >= 65 536 characters          */
};

typedef struct latok_b200_engine latok_b200_engine;

/* ---- library ---------------------------------------------------------------------------- */
LATOK_B200_API int latok_b200_abi_version(void);
LATOK_B200_API const char *latok_b200_last_error(void);
/* number of visible CUDA devices (0 and LATOK_B200_OK on a box without a GPU driver) */
LATOK_B200_API int latok_b200_device_count(int *count);

/* ---- engine lifetime (replaces module init, latok.c:394-416, which holds no state) -------- */
/* max_batch_bytes / max_strings size the device and pinned buffers up front; both grow on demand. */
LATOK_B200_API int latok_b200_create(int device, size_t max_batch_bytes, int64_t max_strings, latok_b200_engine **out);
LATOK_B200_API int latok_b200_destroy(latok_b200_engine *e);

/* ---- tokenizer rules (the reference's extension point: combo matrices,
 *      latok_utils.py:27-56 + default_tokenizer.py:39-110).  Each matrix is int8 [rows, cols],
 *      row-major, feature column indices padded with -1; rows are AND-ed, then summed.
 *      Defaults = C_SPLIT / C_MASK / C_SYM of default_tokenizer.py:108-110.
 *      Restriction: the split matrix must contain the row [SPACE_IDX] (every whitespace
 *      character is a split point), which is what makes "drop an all-whitespace span"
 *      equal to the reference's `text[s:e].strip()` test.
 *      A batch is tokenized with the rules in force when it is submitted: set_rules between a submit
 *      and its fetch (pipeline depth 2) applies to later submits only. */
LATOK_B200_API int latok_b200_set_rules(latok_b200_engine *e,
                         const int8_t *split, int split_rows, int split_cols,
                         const int8_t *mask, int mask_rows, int mask_cols,
                         const int8_t *sym, int sym_rows, int sym_cols);

/* ---- batch hot path ---------------------------------------------------------------------
 * A submitted batch lives in one of the engine's TWO sets of device / pinned staging buffers until it is released.
 * Pipeline depth 1 (default): every submit replaces the batch in flight; sizes / fetch refer to it.
 * Pipeline depth 2: two batches may be in flight; sizes / fetch / fetch_token_bytes / last_stats refer to the OLDEST
 * one and latok_b200_release() retires it.  The loop
 *     submit(0); for i: { submit(i+1); fetch(i); release(); }
 * on ONE host thread overlaps the host -> device copy and the kernels of batch i+1 with the device -> host copy of
 * batch i (separate copy-in, compute and copy-out streams; this is the double buffering of the north star).
 * Changing the depth drops the batches in flight. */
LATOK_B200_API int latok_b200_set_pipeline_depth(latok_b200_engine *e, int depth);
/* Host buffers in: stages pageable memory through the set's pinned buffers (pinned caller memory, e.g. from
 * latok_b200_host_alloc, goes straight to the device), cudaMemcpyAsync on the copy-in stream, kernels on the compute
 * stream.  Returns once the work is enqueued.  ESTATE if `depth` batches are already in flight. */
LATOK_B200_API int latok_b200_submit(latok_b200_engine *e, const uint8_t *utf8, const int64_t *offsets,
                      int64_t n_strings, uint32_t what);
/* Same, for text already resident in device memory (16-byte aligned d_utf8). */
LATOK_B200_API int latok_b200_submit_device(latok_b200_engine *e, const uint8_t *d_utf8, const int64_t *d_offsets,
                             int64_t n_strings, int64_t n_bytes, uint32_t what);
/* Waits for the kernels of the (oldest) batch in flight; C = total characters, T = total emitted tokens. */
LATOK_B200_API int latok_b200_sizes(latok_b200_engine *e, int64_t *n_chars, int64_t *n_tokens);
/* Copies results into caller (host) buffers on the copy-out stream and waits for them; any pointer may be NULL to
 * skip that output.  cap_chars / cap_tokens / cap_strings = what the caller's arrays have room for (characters,
 * tokens, strings); EINVAL (nothing is written) when the batch needs more.
 *   splits       int8  [C]      split mask, values 0..n (counts, not booleans)
 *   char_offsets int64 [S+1]    first character of each string in `splits` / `matrix`
 *   spans        int32 [T,2]    (start_idx, end_idx) per token, untrimmed, string-relative
 *                               (uint16 [T,2] when LATOK_B200_SPANS16 was requested)
 *   tok_offsets  int64 [S+1]    first token of each string in `spans` / `tok_feats`
 *   tok_feats    int8  [T,25]   per-token feature sums (uint8 wrap-around viewed as int8)
 *   matrix       int8  [C,25]   the parse matrix
 */
LATOK_B200_API int latok_b200_fetch(latok_b200_engine *e, int64_t cap_chars, int64_t cap_tokens, int64_t cap_strings,
                     int8_t *splits, int64_t *char_offsets, void *spans, int64_t *tok_offsets, int8_t *tok_feats,
                     int8_t *matrix);
/* Retires the oldest batch in flight (its set may be submitted into again). */
LATOK_B200_API int latok_b200_release(latok_b200_engine *e);
LATOK_B200_API int latok_b200_in_flight(latok_b200_engine *e, int *n);
/* Token spans as BYTE ranges of the flat UTF-8 buffer, trimmed the way the reference trims a token with
 * `text[s:e].strip()` (default_tokenizer.py:151-158; SURVEY 8 f1): utf8[byte_spans[2k] : byte_spans[2k+1]] is the
 * text of token k, so tokens can be sliced from the packed buffer (or viewed as an Arrow-style string array)
 * without touching Python strings.  Needs LATOK_B200_SPANS at submit and the submitted text still in place
 * (host submits: until the next submit; device submits: the caller's buffer).  byte_spans is int64 [T,2] in host
 * memory, or in device memory when on_device != 0, with room for cap_tokens tokens (EINVAL if the batch has more).
 * Runs three small kernels after the tokenize kernel. */
LATOK_B200_API int latok_b200_fetch_token_bytes(latok_b200_engine *e, int64_t cap_tokens, int64_t *byte_spans, int on_device);
/* device time of those kernels for the last call (harness) */
LATOK_B200_API int latok_b200_token_bytes_ms(latok_b200_engine *e, float *ms);
/* Device pointers of the same results (valid until the next submit); for device-side consumers. */
LATOK_B200_API int latok_b200_device_results(latok_b200_engine *e, const int8_t **splits, const int64_t **char_offsets,
                              const int32_t **spans, const int64_t **tok_offsets,
                              const int8_t **tok_feats, const int8_t **matrix);

/* ---- token vocabulary: corpus token counts and integer token ids on the device ------------------
 * The counterpart of a `collections.Counter` over the tokens of tokenize_batch, or of a dict lookup per token, without
 * a Python string per token (no counterpart in the reference, which yields token strings, default_tokenizer.py:151-158).
 * A vocabulary lives on one device; its keys are the exact trimmed token bytes (what fetch_token_bytes ranges select:
 * `text[s:e].strip()` as UTF-8 with lone surrogates encoded as 'surrogatepass' does); ids are dense, 0 .. n_keys - 1,
 * in the order of first occurrence (within a batch: token order).  A batch commits all at once or not at all.
 * Device memory held: the hash table (16 + 8 bytes per slot, at least 2 slots per key, power-of-two capacity, grown
 * 4x when the load passes one half), the key arena (key bytes + 16 bytes per key: offsets and counts) and 8 bytes per
 * token of the largest batch; encode also uses the engine's 16 bytes per token for the token byte ranges.
 * LATOK_B200_VOCAB_HASH_BITS=n (read at creation; tests only) keeps n bits of the hash to force collisions. */
typedef struct latok_b200_vocab latok_b200_vocab;
/* An empty vocabulary on e's device, sized for expected_keys keys (more grow the table). */
LATOK_B200_API int latok_b200_vocab_create(latok_b200_engine *e, int64_t expected_keys, latok_b200_vocab **out);
LATOK_B200_API int latok_b200_vocab_destroy(latok_b200_vocab *v);
/* The tokens of the engine's (oldest) batch in flight (needs LATOK_B200_SPANS and the submitted text still in place, as
 * for fetch_token_bytes).  add != 0: every token is counted, keys not in the vocabulary get the next ids; add == 0:
 * read-only, a token not in the vocabulary gets unk_id.  ids: int32 [T] in token order (CSR = tok_offsets of fetch),
 * in host memory or, with on_device != 0, in device memory (4-byte aligned); NULL skips them.  cap_tokens = room in
 * ids (EINVAL when the batch has more tokens).  Runs on the engine's compute stream after the batch's kernels;
 * EINVAL for a vocabulary on another device, or one that would pass 2^31 - 1 keys (nothing is committed then). */
LATOK_B200_API int latok_b200_vocab_encode(latok_b200_engine *e, latok_b200_vocab *v, int add, int32_t unk_id,
                                           int64_t cap_tokens, int32_t *ids, int on_device);
/* keys, their bytes, and the slots of the hash table (load = n_keys / table_slots); any pointer may be NULL */
LATOK_B200_API int latok_b200_vocab_size(latok_b200_vocab *v, int64_t *n_keys, int64_t *key_bytes, int64_t *table_slots);
/* Keys in id order into host buffers (any may be NULL): bytes [key_bytes], offsets [n_keys + 1] (key i =
 * bytes[offsets[i] : offsets[i + 1]]), counts int64 [n_keys].  cap_keys / cap_bytes = room, as in fetch. */
LATOK_B200_API int latok_b200_vocab_export(latok_b200_vocab *v, int64_t cap_keys, int64_t cap_bytes,
                                           uint8_t *bytes, int64_t *offsets, int64_t *counts);
/* Adds n_keys keys (host bytes + offsets [n_keys + 1]) with the ids n_keys_before + position and the given counts
 * (NULL: 0).  A key that is empty, repeated, or already in the vocabulary is EINVAL (nothing is added then). */
LATOK_B200_API int latok_b200_vocab_import(latok_b200_engine *e, latok_b200_vocab *v, const uint8_t *bytes,
                                           const int64_t *offsets, int64_t n_keys, const int64_t *counts);
/* Adds every key of src to dst with its src count: a key dst lacks gets the next id (new keys in src's id order), a
 * key dst has gets src's count added (Counter.update(other)).  src may be on any device; e is dst's engine.
 * map: int32 [n_keys(src)], the dst id of every src id, in host memory or (on_device != 0) in device memory on dst's
 * device; NULL skips it.  All or nothing, as for encode.  EINVAL when src == dst or the result would pass 2^31 - 1 keys. */
LATOK_B200_API int latok_b200_vocab_merge(latok_b200_engine *e, latok_b200_vocab *dst, const latok_b200_vocab *src,
                                          int32_t *map, int on_device);
/* Drops every key and count; keeps the table and arena allocations (for scratch vocabularies reused per batch). */
LATOK_B200_API int latok_b200_vocab_clear(latok_b200_vocab *v);
/* device time of the last encode / import / merge (token byte ranges and a merge's copy-in included; harness) */
LATOK_B200_API int latok_b200_vocab_last_ms(latok_b200_vocab *v, float *ms);

/* ---- measurement hooks (harness only) ----------------------------------------------------- */
/* CUDA-event bracket on the engine's compute stream around any number of submits. */
LATOK_B200_API int latok_b200_timer_begin(latok_b200_engine *e);
LATOK_B200_API int latok_b200_timer_end(latok_b200_engine *e, float *elapsed_ms); /* synchronises */
/* kernels launched by this engine since creation (the harness reports the delta) */
LATOK_B200_API int latok_b200_launch_count(latok_b200_engine *e, int64_t *launches);
/* device time of the tokenize kernel alone for the last submit, and number of tiles that had to
 * scan ahead beyond their halo to close a whitespace chunk */
LATOK_B200_API int latok_b200_last_stats(latok_b200_engine *e, float *tokenize_kernel_ms, int64_t *lookahead_walks);

/* ---- ingest: csv / csv.gz rows -> packed batch (host code; counterpart of the per-row loop of
 *      scripts/timing/time_tokenizer.py:25-40, `text = json.loads(row[column]).strip()`; SURVEY 8 f3) ------------- */
typedef struct latok_b200_reader latok_b200_reader;
/* `path` may be gzip-compressed; `column` is the csv column that holds the JSON-encoded text (the reference uses 1). */
LATOK_B200_API int latok_b200_reader_open(const char *path, int column, latok_b200_reader **out);
/* Packs up to max_rows further rows: their stripped UTF-8 is appended to utf8 (capacity utf8_cap bytes; pinned memory
 * from latok_b200_host_alloc goes to latok_b200_submit without another copy) and offsets[0..*n_rows] receives the
 * running byte offsets (offsets needs max_rows + 1 entries).  Stops early when the next row would not fit;
 * *n_rows == 0 means end of file.  A row without that column, or whose column is not a JSON string, is an error
 * (LATOK_B200_EINVAL), as it is in the reference's loop. */
LATOK_B200_API int latok_b200_reader_next(latok_b200_reader *r, int64_t max_rows, uint8_t *utf8, int64_t utf8_cap,
                           int64_t *offsets, int64_t *n_rows);
LATOK_B200_API int latok_b200_reader_close(latok_b200_reader *r);

/* ---- pinned host memory for callers that want zero-copy staging --------------------------- */
LATOK_B200_API int latok_b200_host_alloc(void **ptr, size_t bytes);
LATOK_B200_API int latok_b200_host_free(void *ptr);

/* ---- the reference extension module's three functions on caller arrays -------------------- */
/* _gen_parse_matrix(text) (latok.c:31-138): one string's UTF-8 -> int8[n_chars,25].
 * Call with out == NULL to obtain n_chars. */
LATOK_B200_API int latok_b200_gen_parse_matrix(latok_b200_engine *e, const uint8_t *utf8, int64_t n_bytes,
                                int64_t *n_chars, int8_t *out);
/* _gen_block_mask(a1, a2) (latok.c:140-258): strided int8 inputs of length n -> int8[n]. */
LATOK_B200_API int latok_b200_gen_block_mask(latok_b200_engine *e, const int8_t *a1, int64_t stride1,
                              const int8_t *a2, int64_t stride2, int64_t n, int8_t *out);
/* _combine_matrix_rows(m, idxs) (latok.c:275-370): m is int8 [m_rows, m_cols] addressed with byte
 * strides; idx is int8 [idx_rows, idx_cols] (2-D: rows AND-ed then summed) or, with
 * idx_cols == 0, a 1-D list of idx_rows row numbers to sum.  out is int8[m_cols]. */
LATOK_B200_API int latok_b200_combine_matrix_rows(latok_b200_engine *e, const int8_t *m, int64_t m_rows, int64_t m_cols,
                                   int64_t stride_row, int64_t stride_col,
                                   const int8_t *idx, int idx_rows, int idx_cols, int8_t *out);

#ifdef __cplusplus
}
#endif
#endif /* LATOK_B200_H */
