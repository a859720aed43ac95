// Internal structures shared by the kernels (latok_tok5.cuh, latok_kernels.cu, latok_tokbytes.cu, latok_vocab.cu) and
// the C-ABI host layer (latok_capi.cu).
#pragma once
#include "_gen/latok_table_types.h"   // latok_stage1_t (8 bits for UCD 11, 16 when a newer UCD needs more than 256 blocks)
#include <cuda_runtime.h>
#include <stdint.h>

namespace latok {

constexpr int NFEAT = 25;
constexpr int MAX_RULE_ROWS = 15;

// packed Unicode class table blob (built by latok_capi.cu from _gen/latok_tables.h)
struct TableLayout {
    // byte offsets inside the blob; every section is 16-byte aligned
    int lutv;         // u32[256]: 4 split-mask bytes for (value bit-plane 0 nibble | bit-plane 1 nibble << 4)
    int ascii_feat;   // u16[128]
    int class_feat;   // u16[16]
    int stage1;       // latok_stage1_t[stage1_len]
    int stage2;       // u8[stage2_len]
    int total;        // multiple of 16
    int stage1_len, stage2_len;
    uint32_t low_limit;
    uint32_t high_first, high_last, high_feat;  // the single non-empty run above low_limit
};

struct RuleSet {
    int n_split, n_mask, n_sym;
    int is_default;
    uint32_t split[MAX_RULE_ROWS + 1];
    uint32_t mask[MAX_RULE_ROWS + 1];
    uint32_t sym[MAX_RULE_ROWS + 1];
};

// ---- records that cross between the CTAs of the tokenize kernel (ONE look-back chain) ----------
// Every tile publishes a 16-byte aggregate as soon as it has finished computing (state 1), computed
// under the assumption that no block-mask backlog enters the tile (true for almost every tile), and
// later its inclusive prefix (state 2).  A reader reconstructs the backlog entering each aggregate it
// consumes; if that is non-zero it waits for that tile's inclusive prefix instead.
// The device reads and writes these records only through the codec of latok_chain.cuh.  AggRec and OpenSums carry the
// launch epoch (Params::epoch), so the host zeroes them only when they are allocated and when the epoch wraps.
constexpr unsigned EPOCH_MASK = (1u << 30) - 1;   // launch epochs wrap at 2^30: AggRec::status keeps two bits for the state
struct __align__(16) AggRec {
    unsigned status;   // epoch << 2 | state (1: aggregate, 2: the inclusive prefix in IncRec too; another epoch: none yet)
    unsigned n_lft;    // characters in the tile | (tile-relative index of its last string start + 1; 0: none) << 16
    unsigned ntok_v;   // tokens in the tile | backlog it leaves << 16, both for no backlog entering it
    unsigned pad;
};
struct __align__(16) IncRec {
    unsigned long long G;     // characters before the end of the tile
    unsigned long long base;  // global index of the first character of the string open at the end of the tile
    unsigned long long K;     // tokens counted before the end of the tile
    int x;                    // backlog leaving the tile
    int pad;
};
// token-feature mode only, one per range: feature sums of the token still open at the end of the range
struct __align__(16) OpenSums {
    unsigned has_split;       // that token holds a split
    unsigned epoch;           // the launch that published the record
    unsigned pad[2];
    unsigned sums[8];         // four uint8 sums per word, 25 features (sums[7] is 0)
};
static_assert(sizeof(AggRec) == 16 && sizeof(IncRec) == 32 && sizeof(OpenSums) == 48, "chain records are whole 16-byte words");

// Statistics of the tokenize kernel's rare paths, counted in every build (LATOK_B200_PRINT_PROF prints them)
struct KernelStats {
    unsigned long long repeat_rounds;       // rounds of repeated analyses (resolve())
    unsigned long long ranges_repeated;     // ranges analysed again
    unsigned long long repeats_hot_tail;    // ... of those, because the guess about a hot tail was wrong
    unsigned long long open_head;           // analyses of ranges that begin inside a chunk
    unsigned long long open_tail;           // ... that end inside one
    unsigned long long backlog_out;         // ... that leave a block-mask backlog
    unsigned long long lookback_restarts;   // look-back walks started again behind a tile that needs a real backlog
};
// The range whose prefix failed the consistency check of pass D (error bit 3)
struct FaultRec {
    unsigned long long range, G_in, K_in;
    long long n_own, ntok, c_lo, c_hi;
};
// LATOK_PROFILE builds: summed clock64() deltas and event counts (lane 0 / 31 of the warps that measure them)
struct ProfClocks {
    unsigned long long phase[6];            // compute warps: ticket + window wait, pass A, hot-tail guess, pass C, prefix wait, pass D
    unsigned long long resolve;             // service warp: resolve() with the backlog from the look-back
    unsigned long long resolve_calls;
    unsigned long long lb_poll;             // look-back: waiting for a window of records
    unsigned long long lb_sum;              // ... summing it
    unsigned long long lb_windows;          // windows walked
    unsigned long long lb_superseded;       // records skipped behind an inclusive prefix
    unsigned long long lb_repolls;          // polling rounds over records not yet published
};

struct Result {
    unsigned long long n_chars;
    unsigned long long n_tokens;
    unsigned long long walks;
    unsigned long long ticket;   // dynamic tile counter (zeroed with the rest of the struct before each launch)
    KernelStats stats;
    FaultRec fault;
    ProfClocks clocks;
    unsigned int error;      // bit 0: watchdog, bit 1: offsets not monotone, bit 2: token capacity exceeded, bit 3: inconsistent prefix (fault)
    unsigned int abort_flag;
};

struct Params {
    const uint8_t *in;
    long long n_bytes;
    const long long *offsets;   // [n_strings + 1]
    long long n_strings;
    const long long *tile_first_str;  // [ntiles + 1]
    long long ntiles;
    long long nranges;                // tile_first_str is indexed by range, ntiles counts tiles (Tok5Plan)
    int8_t *splits;
    long long *char_off;
    int32_t *spans;
    long long *tok_off;
    int8_t *feats;
    long long cap_tokens;
    uint32_t what;
    AggRec *agg;
    IncRec *inc;
    OpenSums *osum;
    uint32_t *planes;     // v5 token-feature mode: the 25 feature planes of every lane-word, [range][step][25][32 lanes]
    unsigned epoch;
    unsigned long long *ticket;
    unsigned long long ticket_base;
    Result *result;
    const uint8_t *table_blob;
    TableLayout tl;
    RuleSet rules;
};

// The tokenize kernel (latok_tok5.cu): one warp analyses a range of the text, a tile is the ranges of one CTA.  The plan
// picks the kernel's geometry for a batch and sizes its work; the launch runs that geometry.
struct Tok5Plan {
    bool short_geometry;
    int range_bytes;          // bytes from one range's start to the next's (launch_tile_index)
    long long nranges, ntiles;
    size_t plane_words;       // token-feature planes (Params::planes)
    int grid;                 // CTAs: ctas_per_sm x SMs, at most ntiles
};
Tok5Plan tokenize5_plan(long long n_bytes, long long n_strings, bool feats, const TableLayout &tl, bool is_default, int n_sm);
cudaError_t launch_tokenize5(const Tok5Plan &plan, const Params &p, cudaStream_t s);
cudaError_t launch_tile_index(const long long *offsets, long long n_strings, long long n_bytes,
                              long long *tile_first_str, long long ntiles, int tile_bytes, Result *result, cudaStream_t s);
cudaError_t launch_block_mask(const int8_t *a1, long long s1, const int8_t *a2, long long s2, long long n,
                              int8_t *out, unsigned char *scratch, cudaStream_t s);
cudaError_t launch_combine_rows(const int8_t *m, long long m_rows, long long m_cols, long long stride_r,
                                long long stride_c, const int8_t *idx, int idx_rows, int idx_cols,
                                int8_t *out, cudaStream_t s);

// characters in front of every 32-byte word of the text: group_pref[w / TB_GROUP] + word_local[w] (latok_tokbytes.cu)
constexpr int TB_WORD = 32;              // bytes per counted word (one 32-bit lead mask)
constexpr int TB_GROUP = 4096;           // words per group (128 KB of text)
long long char_prefix_words(long long n_bytes);
long long char_prefix_groups(long long n_bytes);
cudaError_t launch_char_prefix(const uint8_t *in, long long n_bytes, unsigned *word_local, unsigned *group_tot,
                               unsigned long long *group_pref, cudaStream_t s);
// token spans as trimmed byte ranges of the flat buffer (latok_tokbytes.cu), after launch_char_prefix
cudaError_t launch_token_bytes(const uint8_t *in, long long n_bytes, const long long *offsets, const long long *char_off,
                               const long long *tok_off, long long n_strings, long long n_tokens, const int32_t *spans,
                               long long *out, const unsigned *word_local, const unsigned long long *group_pref,
                               const uint8_t *table_blob, const TableLayout &tl, int n_sm, cudaStream_t s);
// the int8 [C,25] parse matrix (latok_kernels.cu), after launch_char_prefix; starts: char_prefix_words(n_bytes) words
cudaError_t launch_parse_matrix(const uint8_t *in, long long n_bytes, const long long *offsets, long long n_strings,
                                uint32_t *starts, const unsigned *word_local, const unsigned long long *group_pref,
                                const uint8_t *table_blob, const TableLayout &tl, int8_t *matrix, const Result *result,
                                int n_sm, cudaStream_t s);

// token vocabulary (latok_vocab.cu)
constexpr unsigned long long VOCAB_COMMITTED = 1ULL << 63;
struct __align__(16) VocabSlot { unsigned long long hash, ref; };    // hash 0: empty
struct VocabStatus {
    unsigned long long claims;     // slots claimed by the insert launch
    unsigned long long n_new;      // keys new in the batch, and their bytes (flag kernel)
    unsigned long long new_bytes;
    unsigned overflow;             // load limit passed or a probe sequence without a slot: the batch is run again
    unsigned pad;
    unsigned long long max_key;    // bytes of the longest key (WordPiece)
};
struct VocabParams {
    VocabSlot *table;
    unsigned long long mask;       // capacity - 1 (capacity a power of two)
    unsigned long long hmask;      // hash bits kept (LATOK_B200_VOCAB_HASH_BITS, a test seam)
    const uint8_t *text;           // the launch's keys: key k = text[rng[k].x, rng[k].y)
    const longlong2 *rng;
    long long n;
    uint8_t *arena;                // committed key id = arena[key_off[id], key_off[id + 1])
    long long *key_off;
    long long n_keys;
    unsigned long long *first_occ; // [capacity]
    uint32_t *slot;                // [n]
    int32_t *rank;                 // [n + 1]
    int32_t *ids;                  // [n] or NULL
    int32_t unk;
    unsigned long long *counts;    // [n_keys] or NULL
    const long long *weight;       // [n]: count of key k (a merge), or NULL: 1 per token
    VocabStatus *st;
    unsigned long long limit;      // new claims the load limit allows in this launch
    // WordPiece (ids = the pieces, [P]; unk = the id of an unknown word)
    const uint8_t *pre;            // continuation prefix, pre[0, plen), in device memory
    int plen;
    int max_chars;                 // a word of more characters is unk
    long long *wp_off;             // [n + 1]: pieces per word, then (after the scan) the first piece of every word
    int32_t *wp_first;             // [n]: the id of a one-piece word
};
enum VocabPhase { VOCAB_INSERT, VOCAB_LOOKUP, VOCAB_FLAG, VOCAB_LENS, VOCAB_COMMIT, VOCAB_COUNT, VOCAB_REHASH, VOCAB_MAX_KEY,
                  VOCAB_WP_COUNT, VOCAB_WP_WRITE };
cudaError_t launch_vocab(VocabPhase phase, const VocabParams &p, long long n_new, int n_sm, cudaStream_t s);
// rng[k] = (key_off[k], key_off[k + 1]) for k < n, on the device (a merge's source keys)
cudaError_t launch_vocab_ranges(const long long *key_off, long long n, longlong2 *rng, int n_sm, cudaStream_t s);
cudaError_t vocab_scan(int which, void *tmp, size_t *tmp_bytes, const VocabParams &p, long long n_new, long long key_bytes,
                       cudaStream_t s);

}  // namespace latok
