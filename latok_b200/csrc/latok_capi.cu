// latok_capi.cu -- host side of liblatok_b200.so: the C ABI declared in include/latok_b200.h.
//
// Owns device / pinned memory, streams and the packed Unicode class table, validates arguments
// (the reference reports errors with PyErr_SetString(PyExc_ValueError, ...), latok.c:40-50,
// 151-171, 292-312; here they become status codes + latok_b200_last_error()) and launches the
// kernels.  There is no CPU implementation of the path in this library.
#include "../../include/latok_b200.h"
#include "latok_internal.h"
#include "_gen/latok_tables.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

using namespace latok;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (call);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return fail(_e == cudaErrorMemoryAllocation ? LATOK_B200_ENOMEM : LATOK_B200_ECUDA,          \
                        "%s failed: %s", #call, cudaGetErrorString(_e));                                 \
    } while (0)

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;  // elements
    int ensure(size_t n, bool zero = false)
    {
        if (n <= cap) return 0;
        size_t want = n + n / 8 + 64;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        CU(cudaMalloc((void **)&p, want * sizeof(T)));
        if (zero) { CU(cudaMemset(p, 0, want * sizeof(T))); CU(cudaDeviceSynchronize()); }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

template <class T>
struct PinBuf {
    T *p = nullptr;
    size_t cap = 0;
    int ensure(size_t n)
    {
        if (n <= cap) return 0;
        size_t want = n + n / 8 + 64;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        CU(cudaMallocHost((void **)&p, want * sizeof(T)));
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// grows b to at least n elements, keeping its first `keep` (written on stream s)
template <class T>
int grow_keep(DevBuf<T> &b, size_t n, size_t keep, cudaStream_t s)
{
    if (n <= b.cap) return 0;
    const size_t want = n > 2 * b.cap ? n : 2 * b.cap;
    T *p = nullptr;
    CU(cudaMalloc((void **)&p, want * sizeof(T)));
    if (keep) CU(cudaMemcpyAsync(p, b.p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s));
    CU(cudaStreamSynchronize(s));
    if (b.p) cudaFree(b.p);
    b.p = p;
    b.cap = want;
    return 0;
}

uint32_t row_mask(const int8_t *row, int cols, bool &ok)
{
    uint32_t m = 0;
    for (int j = 0; j < cols; ++j) {
        int v = row[j];
        if (v == -1) continue;
        if (v < 0 || v >= NFEAT) { ok = false; return 0; }
        m |= 1u << v;
    }
    if (m == 0) ok = false;  // a row of only -1 has no defined value in the reference (latok.c:325-337)
    return m;
}

// default rules = C_SPLIT / C_MASK / C_SYM of default_tokenizer.py:49-55, 80-91, 100-102 (column
// numbers from offsets.py:24-48)
RuleSet default_rules()
{
    RuleSet r;
    memset(&r, 0, sizeof r);
    r.is_default = 1;
    const uint32_t split[] = {1u << 5, 1u << 6, 1u << 20, (1u << 4) | (1u << 17), (1u << 4) | (1u << 16)};
    const uint32_t mask[] = {(1u << 7) | (1u << 18) | (1u << 13), (1u << 11) | (1u << 18) | (1u << 21) | (1u << 23),
                             (1u << 8) | (1u << 14) | (1u << 15), (1u << 9) | (1u << 22) | (1u << 24) | (1u << 12)};
    const uint32_t sym[] = {(1u << 6) | (1u << 19)};
    r.n_split = 5; r.n_mask = 4; r.n_sym = 1;
    memcpy(r.split, split, sizeof split);
    memcpy(r.mask, mask, sizeof mask);
    memcpy(r.sym, sym, sizeof sym);
    return r;
}

bool same_rows(const uint32_t *a, int na, const uint32_t *b, int nb)
{
    if (na != nb) return false;
    std::vector<uint32_t> x(a, a + na), y(b, b + nb);
    for (auto v : x) {
        bool found = false;
        for (auto &w : y) if (w == v) { w = 0xFFFFFFFFu; found = true; break; }
        if (!found) return false;
    }
    return true;
}

}  // namespace

// One of the two sets of buffers a submitted batch lives in until it has been fetched.  Two sets alternate, so that
// (pipeline depth 2) batch i+1 is copied in and tokenized while batch i is copied out.
struct Batch {
    DevBuf<uint8_t> d_in;
    DevBuf<long long> d_off, d_first, d_char_off, d_tok_off;
    DevBuf<int8_t> d_splits, d_feats, d_matrix;
    DevBuf<int32_t> d_spans;
    DevBuf<uint32_t> d_spans16;                     // LATOK_B200_SPANS16: (start | end << 16) per token
    DevBuf<Result> d_result;
    PinBuf<Result> h_result;
    PinBuf<uint8_t> h_in;                           // pinned staging of pageable caller buffers
    PinBuf<long long> h_off;
    cudaEvent_t ev_h2d = nullptr;                   // inputs have arrived on the device (copy-in stream)
    cudaEvent_t ev_index = nullptr;                 // string index built (aux stream)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;   // around the tokenize kernel (timing)
    cudaEvent_t ev_kdone = nullptr;                 // last device work that touches this set (compute stream)
    bool submitted = false, sized = false, inputs_on_stream = false;
    const uint8_t *cur_in = nullptr;
    const long long *cur_off = nullptr;
    long long n_strings = 0, n_bytes = 0;
    uint32_t what = 0;
    long long n_chars = 0, n_tokens = 0, walks = 0;
    float kernel_ms = 0.f;
    void release()
    {
        d_in.release(); d_off.release(); d_first.release(); d_char_off.release(); d_tok_off.release();
        d_splits.release(); d_feats.release(); d_matrix.release(); d_spans.release(); d_spans16.release();
        d_result.release(); h_result.release(); h_in.release(); h_off.release();
        for (cudaEvent_t *ev : {&ev_h2d, &ev_index, &ev_k0, &ev_k1, &ev_kdone}) { if (*ev) cudaEventDestroy(*ev); *ev = nullptr; }
    }
};

struct latok_b200_engine {
    int device = 0;
    int n_sm = 0;
    // compute: kernels; aux: string index of the next batch while the previous one is tokenized;
    // s_in / s_out: host -> device and device -> host copies (PCIe is full duplex: the three overlap)
    cudaStream_t stream = nullptr, aux = nullptr, s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_b0 = nullptr, ev_b1 = nullptr;
    TableLayout tl{};
    RuleSet rules{};
    DevBuf<uint8_t> d_table, d_scratch, d_scratch2, d_scratch3;
    DevBuf<AggRec> agg;
    DevBuf<IncRec> inc;
    DevBuf<OpenSums> osum;
    DevBuf<uint32_t> d_planes;
    DevBuf<long long> d_tok_bytes;                  // token byte ranges (latok_b200_fetch_token_bytes)
    DevBuf<unsigned> d_blk_local, d_group_tot;      // characters in front of every 32-byte word (launch_char_prefix)
    DevBuf<unsigned long long> d_group_pref;
    DevBuf<uint32_t> d_starts;                      // string-start bitmap of the parse matrix
    float last_token_bytes_ms = 0.f;
    unsigned epoch = 0;
    long long launches = 0;
    Batch set[2];
    int depth = 1;                                  // batches that may be in flight (submitted, not yet released)
    int q[2] = {0, 0}, nq = 0;                      // the sets in flight, oldest first
    int last = 1;                                   // set of the most recent submit
    Batch *front() { return nq ? &set[q[0]] : nullptr; }
};

// for the other translation units of the library (latok_reader.cpp)
extern "C" int latok_b200_set_error_(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

static int set_device(latok_b200_engine *e)
{
    CU(cudaSetDevice(e->device));
    return 0;
}

extern "C" {

int latok_b200_abi_version(void) { return LATOK_B200_ABI_VERSION; }
const char *latok_b200_last_error(void) { return g_err; }

int latok_b200_device_count(int *count)
{
    if (!count) return fail(LATOK_B200_EINVAL, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
    *count = n;
    return LATOK_B200_OK;
}

static int build_table(latok_b200_engine *e)
{
    TableLayout &tl = e->tl;
    int o = 0;
    auto take = [&](int bytes) { int r = o; o += (bytes + 15) & ~15; return r; };
    tl.lutv = take(256 * 4);
    tl.ascii_feat = take(128 * 2);
    tl.class_feat = take(16 * 2);
    tl.stage1 = take(LATOK_TBL_STAGE1_LEN * (int)sizeof(latok_stage1_t));
    tl.stage2 = take(LATOK_TBL_STAGE2_LEN);
    tl.total = o;
    tl.stage1_len = LATOK_TBL_STAGE1_LEN;
    tl.stage2_len = LATOK_TBL_STAGE2_LEN;
    tl.low_limit = LATOK_TBL_LOW_LIMIT;
    static_assert(LATOK_TBL_NHIGH <= 1, "kernel supports one run above the two-stage table");
    static_assert(LATOK_TBL_SHIFT == 7, "kernel assumes 128-code-point blocks");
    tl.high_first = LATOK_HIGH_RUNS[0][0];
    tl.high_last = LATOK_HIGH_RUNS[0][1];
    tl.high_feat = LATOK_HIGH_RUNS[0][2];
    std::vector<uint8_t> blob((size_t)tl.total, 0);
    {
        uint32_t *lutv = reinterpret_cast<uint32_t *>(blob.data() + tl.lutv);
        for (int i = 0; i < 256; ++i) {
            uint32_t w = 0;
            for (int b = 0; b < 4; ++b) w |= ((((uint32_t)i >> b) & 1u) + 2u * (((uint32_t)i >> (4 + b)) & 1u)) << (8 * b);
            lutv[i] = w;
        }
    }
    memcpy(blob.data() + tl.ascii_feat, LATOK_ASCII_FEAT, sizeof LATOK_ASCII_FEAT);
    memcpy(blob.data() + tl.class_feat, LATOK_CLASS_FEAT, sizeof LATOK_CLASS_FEAT);
    memcpy(blob.data() + tl.stage1, LATOK_STAGE1, sizeof LATOK_STAGE1);
    memcpy(blob.data() + tl.stage2, LATOK_STAGE2, sizeof LATOK_STAGE2);
    if (int rc = e->d_table.ensure(blob.size())) return rc;
    CU(cudaMemcpy(e->d_table.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    return 0;
}

int latok_b200_create(int device, size_t max_batch_bytes, int64_t max_strings, latok_b200_engine **out)
{
    if (!out) return fail(LATOK_B200_EINVAL, "out is NULL");
    *out = nullptr;
    if (max_strings < 0) return fail(LATOK_B200_EINVAL, "max_strings must be >= 0");
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(LATOK_B200_ECUDA, "no CUDA device available (%s); latok_b200 has no CPU fallback",
                    ce != cudaSuccess ? cudaGetErrorString(ce) : "device count is 0");
    }
    if (device < 0 || device >= n) return fail(LATOK_B200_EINVAL, "device %d out of range [0,%d)", device, n);
    latok_b200_engine *e = new (std::nothrow) latok_b200_engine();
    if (!e) return fail(LATOK_B200_ENOMEM, "out of host memory");
    e->device = device;
    int rc = [&]() -> int {
        CU(cudaSetDevice(device));
        CU(cudaDeviceGetAttribute(&e->n_sm, cudaDevAttrMultiProcessorCount, device));
        for (cudaStream_t *st : {&e->stream, &e->aux, &e->s_in, &e->s_out}) CU(cudaStreamCreateWithFlags(st, cudaStreamNonBlocking));
        CU(cudaEventCreate(&e->ev_t0)); CU(cudaEventCreate(&e->ev_t1));
        CU(cudaEventCreate(&e->ev_b0)); CU(cudaEventCreate(&e->ev_b1));
        if (int r = build_table(e)) return r;
        e->rules = default_rules();
        for (Batch &b : e->set) {
            CU(cudaEventCreate(&b.ev_k0)); CU(cudaEventCreate(&b.ev_k1));
            for (cudaEvent_t *ev : {&b.ev_h2d, &b.ev_index, &b.ev_kdone}) CU(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
            if (int r = b.d_result.ensure(1, true)) return r;
            if (int r = b.h_result.ensure(1)) return r;
        }
        // max_batch_bytes / max_strings pre-size the first set (a second one is sized on first use, i.e. by a
        // pipelined caller or by back-to-back submits)
        Batch &b = e->set[0];
        if (max_batch_bytes) {
            if (int r = b.d_in.ensure(max_batch_bytes + 64)) return r;
            if (int r = b.d_splits.ensure(max_batch_bytes + 64)) return r;
            if (int r = b.d_spans.ensure(2 * (max_batch_bytes / 3 + 1024))) return r;
        }
        if (max_strings) {
            if (int r = b.d_off.ensure((size_t)max_strings + 1)) return r;
            if (int r = b.d_char_off.ensure((size_t)max_strings + 1)) return r;
            if (int r = b.d_tok_off.ensure((size_t)max_strings + 1)) return r;
        }
        return 0;
    }();
    if (rc) { latok_b200_destroy(e); return rc; }
    *out = e;
    return LATOK_B200_OK;
}

int latok_b200_destroy(latok_b200_engine *e)
{
    if (!e) return LATOK_B200_OK;
    cudaSetDevice(e->device);
    for (cudaStream_t st : {e->stream, e->aux, e->s_in, e->s_out}) if (st) cudaStreamSynchronize(st);
    e->d_table.release(); e->d_scratch.release(); e->d_scratch2.release(); e->d_scratch3.release();
    e->agg.release(); e->inc.release(); e->osum.release(); e->d_planes.release();
    e->d_tok_bytes.release(); e->d_blk_local.release(); e->d_group_tot.release(); e->d_group_pref.release(); e->d_starts.release();
    for (Batch &b : e->set) b.release();
    for (cudaEvent_t ev : {e->ev_t0, e->ev_t1, e->ev_b0, e->ev_b1}) if (ev) cudaEventDestroy(ev);
    for (cudaStream_t st : {e->stream, e->aux, e->s_in, e->s_out}) if (st) cudaStreamDestroy(st);
    delete e;
    return LATOK_B200_OK;
}

int latok_b200_set_pipeline_depth(latok_b200_engine *e, int depth)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (depth != 1 && depth != 2) return fail(LATOK_B200_EINVAL, "pipeline depth must be 1 or 2");
    e->nq = 0;                   // batches in flight are dropped (their device work still completes)
    e->depth = depth;
    return LATOK_B200_OK;
}

int latok_b200_set_rules(latok_b200_engine *e, const int8_t *split, int sr, int sc, const int8_t *mask, int mr,
                         int mc, const int8_t *sym, int yr, int yc)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (!split && !mask && !sym) { e->rules = default_rules(); return LATOK_B200_OK; }
    if (!split || !mask || !sym) return fail(LATOK_B200_EINVAL, "must specify split, mask and sym combo matrices");
    if (sr < 1 || mr < 0 || yr < 0 || sr > MAX_RULE_ROWS || mr > MAX_RULE_ROWS || yr > MAX_RULE_ROWS)
        return fail(LATOK_B200_EINVAL, "combo matrices must have between 1 and %d rows", MAX_RULE_ROWS);
    if (sc < 1 || (mr && mc < 1) || (yr && yc < 1)) return fail(LATOK_B200_EINVAL, "combo matrices must have >= 1 column");
    RuleSet r;
    memset(&r, 0, sizeof r);
    bool ok = true, has_space = false;
    for (int i = 0; i < sr; ++i) { r.split[i] = row_mask(split + i * sc, sc, ok); has_space |= r.split[i] == (1u << 5); }
    for (int i = 0; i < mr; ++i) r.mask[i] = row_mask(mask + i * mc, mc, ok);
    for (int i = 0; i < yr; ++i) r.sym[i] = row_mask(sym + i * yc, yc, ok);
    if (!ok) return fail(LATOK_B200_EINVAL, "combo matrix entries must be feature indices in [0,%d) or -1, with at least one index per row", NFEAT);
    if (!has_space)
        return fail(LATOK_B200_EINVAL, "the split combo matrix must contain the row [SPACE_IDX] (see latok_b200.h)");
    r.n_split = sr; r.n_mask = mr; r.n_sym = yr;
    const RuleSet d = default_rules();
    r.is_default = same_rows(r.split, sr, d.split, d.n_split) && same_rows(r.mask, mr, d.mask, d.n_mask) &&
                   same_rows(r.sym, yr, d.sym, d.n_sym);
    e->rules = r;
    return LATOK_B200_OK;
}

// narrows the int32 (start, end) pairs of the tokenize kernel to one uint32 (start | end << 16) per token
// (LATOK_B200_SPANS16: half the device -> host bytes when every string has fewer than 65 536 characters)
__global__ void narrow_spans_kernel(const int2 *spans, uint32_t *out, Result *res, long long cap)
{
    const long long n = min((long long)res->n_tokens, cap);
    bool over = false;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const int2 v = spans[k];
        over |= ((unsigned)v.x | (unsigned)v.y) > 0xFFFFu;
        out[k] = ((unsigned)v.x & 0xFFFFu) | ((unsigned)v.y << 16);
    }
    if (over) atomicOr(&res->error, 16u);
}

// characters in front of every 32-byte word of batch b (launch_char_prefix) on the compute stream
static int enqueue_char_prefix(latok_b200_engine *e, Batch &b)
{
    if (int r = e->d_blk_local.ensure((size_t)char_prefix_words(b.n_bytes))) return r;
    if (int r = e->d_group_tot.ensure((size_t)char_prefix_groups(b.n_bytes))) return r;
    if (int r = e->d_group_pref.ensure((size_t)char_prefix_groups(b.n_bytes))) return r;
    CU(launch_char_prefix(b.cur_in, b.n_bytes, e->d_blk_local.p, e->d_group_tot.p, e->d_group_pref.p, e->stream));
    e->launches += 2;
    return 0;
}

static int run_device(latok_b200_engine *e, Batch &b)
{
    // The tokenize kernel, in the geometry its plan picks for the batch.  It also gives the character counts and the
    // offsets check of a matrix-only batch.  The parse matrix follows it on the same stream.
    const bool feats = (b.what & LATOK_B200_FEATS) != 0;
    const Tok5Plan t5 = tokenize5_plan(b.n_bytes, b.n_strings, feats, e->tl, e->rules.is_default != 0, e->n_sm);
    if (int r = b.d_first.ensure((size_t)t5.nranges + 1)) return r;
    // the status word of every aggregate record carries the launch epoch, so records are zeroed only when (re)allocated
    // (agg / inc / osum / planes are shared by the two sets: tokenize kernels run one after the other on one stream)
    if ((size_t)t5.ntiles > e->agg.cap) { CU(cudaStreamSynchronize(e->stream)); if (int r = e->agg.ensure((size_t)t5.ntiles, true)) return r; }
    if ((size_t)t5.ntiles > e->inc.cap) { CU(cudaStreamSynchronize(e->stream)); if (int r = e->inc.ensure((size_t)t5.ntiles)) return r; }
    if (feats && (size_t)t5.nranges > e->osum.cap) { CU(cudaStreamSynchronize(e->stream)); if (int r = e->osum.ensure((size_t)t5.nranges, true)) return r; }
    if (feats && t5.plane_words > e->d_planes.cap) { CU(cudaStreamSynchronize(e->stream)); if (int r = e->d_planes.ensure(t5.plane_words)) return r; }
    if (int r = b.d_splits.ensure((size_t)b.n_bytes + 64)) return r;
    if (int r = b.d_char_off.ensure((size_t)b.n_strings + 1)) return r;
    if (int r = b.d_tok_off.ensure((size_t)b.n_strings + 1)) return r;
    if (b.d_spans.cap < 2048) { if (int r = b.d_spans.ensure(2 * ((size_t)b.n_bytes / 3 + 1024))) return r; }
    if (b.what & LATOK_B200_FEATS) { if (int r = b.d_feats.ensure((b.d_spans.cap / 2) * NFEAT)) return r; }
    if (b.what & LATOK_B200_MATRIX) { if (int r = b.d_matrix.ensure(((size_t)b.n_bytes + 64) * NFEAT)) return r; }
    if (b.what & LATOK_B200_SPANS16) { if (int r = b.d_spans16.ensure(b.d_spans.cap / 2)) return r; }

    e->epoch = (e->epoch + 1) & 0x3FFFFFFFu;
    if (e->epoch == 0) {  // wrapped: clear stale status words
        CU(cudaMemsetAsync(e->agg.p, 0, e->agg.cap * sizeof(AggRec), e->stream));
        e->epoch = 1;
    }
    Params p;
    memset(&p, 0, sizeof p);
    p.in = b.cur_in; p.n_bytes = b.n_bytes; p.offsets = b.cur_off; p.n_strings = b.n_strings;
    p.tile_first_str = b.d_first.p; p.ntiles = t5.ntiles; p.nranges = t5.nranges;
    p.splits = b.d_splits.p; p.char_off = b.d_char_off.p; p.spans = b.d_spans.p; p.tok_off = b.d_tok_off.p;
    p.feats = b.d_feats.p;
    p.cap_tokens = (long long)(b.d_spans.cap / 2);
    p.what = b.what & 7u;
    p.agg = e->agg.p; p.inc = e->inc.p; p.osum = e->osum.p; p.planes = e->d_planes.p; p.epoch = e->epoch;
    p.ticket = &b.d_result.p->ticket; p.ticket_base = 0;
    p.result = b.d_result.p;
    p.table_blob = e->d_table.p; p.tl = e->tl; p.rules = e->rules;

    // The string index of this batch is built on the aux stream, so that with back-to-back submits it overlaps the
    // tokenize kernel of the previous batch (the two sets alternate).
    if (b.inputs_on_stream) CU(cudaStreamWaitEvent(e->aux, b.ev_h2d, 0));    // host submit: the offsets arrive on the copy-in stream
    CU(cudaStreamWaitEvent(e->aux, b.ev_kdone, 0));            // this set's previous batch has been tokenized
    CU(cudaMemsetAsync(b.d_result.p, 0, sizeof(Result), e->aux));
    CU(launch_tile_index(b.cur_off, b.n_strings, b.n_bytes, b.d_first.p, t5.nranges, t5.range_bytes, b.d_result.p, e->aux));
    CU(cudaEventRecord(b.ev_index, e->aux));
    if (b.inputs_on_stream) CU(cudaStreamWaitEvent(e->stream, b.ev_h2d, 0));
    CU(cudaStreamWaitEvent(e->stream, b.ev_index, 0));
    CU(cudaEventRecord(b.ev_k0, e->stream));
    CU(launch_tokenize5(t5, p, e->stream));
    CU(cudaEventRecord(b.ev_k1, e->stream));
    e->launches += 2;
    if (b.what & LATOK_B200_MATRIX) {
        if (int r = enqueue_char_prefix(e, b)) return r;
        if (int r = e->d_starts.ensure((size_t)char_prefix_words(b.n_bytes))) return r;
        CU(launch_parse_matrix(b.cur_in, b.n_bytes, b.cur_off, b.n_strings, e->d_starts.p, e->d_blk_local.p, e->d_group_pref.p,
                               e->d_table.p, e->tl, b.d_matrix.p, b.d_result.p, e->n_sm, e->stream));
        e->launches += 2;
    }
    if (b.what & LATOK_B200_SPANS16) {
        narrow_spans_kernel<<<e->n_sm * 8, 256, 0, e->stream>>>(reinterpret_cast<const int2 *>(b.d_spans.p), b.d_spans16.p, b.d_result.p, p.cap_tokens);
        CU(cudaGetLastError());
        e->launches += 1;
    }
    CU(cudaMemcpyAsync(b.h_result.p, b.d_result.p, sizeof(Result), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(b.ev_kdone, e->stream));
    b.submitted = true;
    b.sized = false;
    return LATOK_B200_OK;
}

static int check_what(uint32_t &what)
{
    if (what & LATOK_B200_SPANS16) what |= LATOK_B200_SPANS;
    if (what == 0 || (what & ~31u)) return fail(LATOK_B200_EINVAL, "`what` must be a non-empty OR of LATOK_B200_SPLITS|SPANS|FEATS|MATRIX|SPANS16");
    return 0;
}

// the set the next submit uses: depth 1 = the batch in flight (if any) is dropped; depth 2 = at most two in flight
static int take_set(latok_b200_engine *e, Batch **out)
{
    if (e->depth == 1) e->nq = 0;
    if (e->nq >= e->depth) return fail(LATOK_B200_ESTATE, "%d batches are in flight: fetch and release the oldest one first", e->nq);
    const int s = e->last ^ 1;
    e->last = s;
    e->q[e->nq++] = s;
    *out = &e->set[s];
    return 0;
}
static void drop_last(latok_b200_engine *e) { if (e->nq) { --e->nq; e->last ^= 1; } }   // a submit that failed

int latok_b200_submit(latok_b200_engine *e, const uint8_t *utf8, const int64_t *offsets, int64_t n_strings, uint32_t what)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (n_strings < 0) return fail(LATOK_B200_EINVAL, "n_strings must be >= 0");
    if (!offsets) return fail(LATOK_B200_EINVAL, "must specify the offsets array (n_strings + 1 entries)");
    if (int r = check_what(what)) return r;
    if (offsets[0] != 0) return fail(LATOK_B200_EINVAL, "offsets[0] must be 0");
    const long long n_bytes = offsets[n_strings];
    if (n_bytes < 0) return fail(LATOK_B200_EINVAL, "offsets must be non-negative");
    if (n_bytes > 0 && !utf8) return fail(LATOK_B200_EINVAL, "must specify the UTF-8 buffer");
    if (int r = set_device(e)) return r;
    Batch *bp = nullptr;
    if (int r = take_set(e, &bp)) return r;
    Batch &b = *bp;
    b.submitted = false;
    int rc = [&]() -> int {
        // the device buffers of this set may still be read by its previous batch's kernels
        if ((size_t)n_bytes + 64 > b.d_in.cap || (size_t)n_strings + 1 > b.d_off.cap) CU(cudaEventSynchronize(b.ev_kdone));
        if (int r = b.d_in.ensure((size_t)n_bytes + 64)) return r;
        if (int r = b.d_off.ensure((size_t)n_strings + 1)) return r;
        // stage through pinned memory unless the caller's buffers already are pinned
        auto is_pinned = [](const void *ptr) {
            cudaPointerAttributes a;
            if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
            return a.type == cudaMemoryTypeHost;
        };
        const uint8_t *src_b = utf8;
        const long long *src_o = (const long long *)offsets;
        const bool stage_b = n_bytes > 0 && !is_pinned(utf8), stage_o = !is_pinned(offsets);
        if (stage_b || stage_o) CU(cudaEventSynchronize(b.ev_h2d));     // the staging buffers may still feed this set's previous copy
        if (stage_b) {
            if (int r = b.h_in.ensure((size_t)n_bytes)) return r;
            memcpy(b.h_in.p, utf8, (size_t)n_bytes);
            src_b = b.h_in.p;
        }
        if (stage_o) {
            if (int r = b.h_off.ensure((size_t)n_strings + 1)) return r;
            memcpy(b.h_off.p, offsets, sizeof(long long) * ((size_t)n_strings + 1));
            src_o = b.h_off.p;
        }
        CU(cudaStreamWaitEvent(e->s_in, b.ev_kdone, 0));               // ... and the device buffers its previous kernels
        if (n_bytes > 0) CU(cudaMemcpyAsync(b.d_in.p, src_b, (size_t)n_bytes, cudaMemcpyHostToDevice, e->s_in));
        CU(cudaMemcpyAsync(b.d_off.p, src_o, sizeof(long long) * ((size_t)n_strings + 1), cudaMemcpyHostToDevice, e->s_in));
        CU(cudaEventRecord(b.ev_h2d, e->s_in));
        b.cur_in = b.d_in.p; b.cur_off = b.d_off.p;
        b.n_strings = n_strings; b.n_bytes = n_bytes; b.what = what;
        b.inputs_on_stream = true;
        return run_device(e, b);
    }();
    if (rc) drop_last(e);
    return rc;
}

int latok_b200_submit_device(latok_b200_engine *e, const uint8_t *d_utf8, const int64_t *d_offsets, int64_t n_strings,
                             int64_t n_bytes, uint32_t what)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (n_strings < 0 || n_bytes < 0) return fail(LATOK_B200_EINVAL, "n_strings and n_bytes must be >= 0");
    if (!d_offsets || (n_bytes > 0 && !d_utf8)) return fail(LATOK_B200_EINVAL, "must specify device buffers");
    if (((uintptr_t)d_utf8 & 15u) != 0) return fail(LATOK_B200_EINVAL, "d_utf8 must be 16-byte aligned");
    if (int r = check_what(what)) return r;
    if (int r = set_device(e)) return r;
    Batch *bp = nullptr;
    if (int r = take_set(e, &bp)) return r;
    Batch &b = *bp;
    b.submitted = false;
    b.cur_in = d_utf8; b.cur_off = (const long long *)d_offsets;
    b.n_strings = n_strings; b.n_bytes = n_bytes; b.what = what;
    b.inputs_on_stream = false;
    const int rc = run_device(e, b);
    if (rc) drop_last(e);
    return rc;
}

static int size_batch(latok_b200_engine *e, Batch &b)
{
    if (!b.submitted) return fail(LATOK_B200_ESTATE, "no batch submitted");
    for (int attempt = 0; attempt < 4 && !b.sized; ++attempt) {
        CU(cudaEventSynchronize(b.ev_kdone));
        const Result res = *b.h_result.p;
        if (res.error & 2u) { b.submitted = false; return fail(LATOK_B200_EINVAL, "offsets must start at 0, be non-decreasing and end at the buffer length"); }
        if (res.error & 1u) { b.submitted = false; return fail(LATOK_B200_EINTERNAL, "device look-back watchdog tripped"); }
        if (res.error & 8u) {
            b.submitted = false;
            return fail(LATOK_B200_EINTERNAL, "device consistency check failed: tile %llu G_in %llu K_in %llu n_own %lld ntok %lld c_lo %lld c_hi %lld",
                        res.prof[8], res.prof[9], res.prof[10], (long long)res.prof[11], (long long)res.prof[12], (long long)res.prof[13], (long long)res.prof[14]);
        }
        if ((res.error & 4u) || (long long)res.n_tokens > (long long)(b.d_spans.cap / 2)) {
            // token buffers too small: grow to the exact count and run the batch again
            const size_t need = (size_t)res.n_tokens + 1024;
            if (int r = b.d_spans.ensure(2 * need)) return r;
            if (int r = run_device(e, b)) return r;
            continue;
        }
        if (res.error & 16u) { b.submitted = false; return fail(LATOK_B200_EINVAL, "LATOK_B200_SPANS16: a string of the batch has 65 536 or more characters"); }
        if (getenv("LATOK_B200_PRINT_PROF")) {
            fprintf(stderr, "[latok prof]");
            for (int i = 0; i < 16; ++i) fprintf(stderr, " %llu", res.prof[i]);
            fprintf(stderr, "\n");
        }
        b.n_chars = (long long)res.n_chars; b.n_tokens = (long long)res.n_tokens; b.walks = (long long)res.walks;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, b.ev_k0, b.ev_k1) == cudaSuccess) b.kernel_ms = ms; else cudaGetLastError();
        b.sized = true;
    }
    if (!b.sized) return fail(LATOK_B200_EINTERNAL, "token capacity did not converge");
    return LATOK_B200_OK;
}

#define FRONT(e, b)                                                                  \
    if (!(e)) return fail(LATOK_B200_EINVAL, "engine is NULL");                      \
    if (!(e)->front()) return fail(LATOK_B200_ESTATE, "no batch submitted");         \
    if (int r_ = set_device(e)) return r_;                                           \
    Batch &b = *(e)->front()

int latok_b200_sizes(latok_b200_engine *e, int64_t *n_chars, int64_t *n_tokens)
{
    FRONT(e, b);
    if (int r = size_batch(e, b)) return r;
    if (n_chars) *n_chars = b.n_chars;
    if (n_tokens) *n_tokens = b.n_tokens;
    return LATOK_B200_OK;
}

int latok_b200_fetch(latok_b200_engine *e, int64_t cap_chars, int64_t cap_tokens, int64_t cap_strings, int8_t *splits,
                     int64_t *char_offsets, void *spans, int64_t *tok_offsets, int8_t *tok_feats, int8_t *matrix)
{
    FRONT(e, b);
    if (int r = size_batch(e, b)) return r;
    const uint32_t w = b.what;
    if (splits && !(w & LATOK_B200_SPLITS)) return fail(LATOK_B200_ESTATE, "split mask was not requested at submit");
    if (spans && !(w & LATOK_B200_SPANS)) return fail(LATOK_B200_ESTATE, "spans were not requested at submit");
    if (tok_feats && !(w & LATOK_B200_FEATS)) return fail(LATOK_B200_ESTATE, "token features were not requested at submit");
    if (matrix && !(w & LATOK_B200_MATRIX)) return fail(LATOK_B200_ESTATE, "feature matrix was not requested at submit");
    if ((splits || matrix) && cap_chars < b.n_chars)
        return fail(LATOK_B200_EINVAL, "cap_chars = %lld, the batch has %lld characters", (long long)cap_chars, b.n_chars);
    if ((spans || tok_feats) && cap_tokens < b.n_tokens)
        return fail(LATOK_B200_EINVAL, "cap_tokens = %lld, the batch has %lld tokens", (long long)cap_tokens, b.n_tokens);
    if ((char_offsets || tok_offsets) && cap_strings < b.n_strings)
        return fail(LATOK_B200_EINVAL, "cap_strings = %lld, the batch has %lld strings", (long long)cap_strings, b.n_strings);
    const size_t C = (size_t)b.n_chars, T = (size_t)b.n_tokens, S1 = (size_t)b.n_strings + 1;
    cudaStream_t s = e->s_out;
    CU(cudaStreamWaitEvent(s, b.ev_kdone, 0));
    if (splits && C) CU(cudaMemcpyAsync(splits, b.d_splits.p, C, cudaMemcpyDeviceToHost, s));
    if (char_offsets) CU(cudaMemcpyAsync(char_offsets, b.d_char_off.p, S1 * sizeof(long long), cudaMemcpyDeviceToHost, s));
    if (spans && T) {
        if (w & LATOK_B200_SPANS16) CU(cudaMemcpyAsync(spans, b.d_spans16.p, T * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        else CU(cudaMemcpyAsync(spans, b.d_spans.p, T * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    }
    if (tok_offsets) CU(cudaMemcpyAsync(tok_offsets, b.d_tok_off.p, S1 * sizeof(long long), cudaMemcpyDeviceToHost, s));
    if (tok_feats && T) CU(cudaMemcpyAsync(tok_feats, b.d_feats.p, T * NFEAT, cudaMemcpyDeviceToHost, s));
    if (matrix && C) CU(cudaMemcpyAsync(matrix, b.d_matrix.p, C * NFEAT, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return LATOK_B200_OK;
}

int latok_b200_release(latok_b200_engine *e)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (!e->nq) return fail(LATOK_B200_ESTATE, "no batch in flight");
    e->q[0] = e->q[1];
    --e->nq;
    return LATOK_B200_OK;
}

int latok_b200_in_flight(latok_b200_engine *e, int *n)
{
    if (!e || !n) return fail(LATOK_B200_EINVAL, "engine or n is NULL");
    *n = e->nq;
    return LATOK_B200_OK;
}

// token byte ranges of batch b into d_out (int64 [T,2], device) on the compute stream, after the batch's kernels
static int enqueue_token_bytes(latok_b200_engine *e, Batch &b, long long *d_out)
{
    cudaStream_t s = e->stream;
    CU(cudaStreamWaitEvent(s, b.ev_kdone, 0));
    CU(cudaEventRecord(e->ev_b0, s));
    if (int r = enqueue_char_prefix(e, b)) return r;
    CU(launch_token_bytes(b.cur_in, b.n_bytes, b.cur_off, b.d_char_off.p, b.d_tok_off.p, b.n_strings, b.n_tokens, b.d_spans.p,
                          d_out, e->d_blk_local.p, e->d_group_pref.p, e->d_table.p, e->tl, e->n_sm, s));
    CU(cudaEventRecord(e->ev_b1, s));
    e->launches += 1;
    return 0;
}

int latok_b200_fetch_token_bytes(latok_b200_engine *e, int64_t cap_tokens, int64_t *byte_spans, int on_device)
{
    FRONT(e, b);
    if (int r = size_batch(e, b)) return r;
    if (!(b.what & LATOK_B200_SPANS)) return fail(LATOK_B200_ESTATE, "spans were not requested at submit");
    const size_t T = (size_t)b.n_tokens;
    if (T && !byte_spans) return fail(LATOK_B200_EINVAL, "must specify the byte_spans array (2 * n_tokens entries)");
    if (cap_tokens < b.n_tokens) return fail(LATOK_B200_EINVAL, "cap_tokens = %lld, the batch has %lld tokens", (long long)cap_tokens, b.n_tokens);
    if (!T) return LATOK_B200_OK;
    if (on_device && ((uintptr_t)byte_spans & 15u) != 0) return fail(LATOK_B200_EINVAL, "a device byte_spans array must be 16-byte aligned");
    long long *d_out = on_device ? (long long *)byte_spans : nullptr;
    if (!on_device) { if (int r = e->d_tok_bytes.ensure(2 * T)) return r; d_out = e->d_tok_bytes.p; }
    if (int r = enqueue_token_bytes(e, b, d_out)) return r;
    cudaStream_t s = e->stream;
    if (!on_device) CU(cudaMemcpyAsync(byte_spans, d_out, T * 2 * sizeof(long long), cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(b.ev_kdone, s));          // the set's inputs are in use until here
    CU(cudaStreamSynchronize(s));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev_b0, e->ev_b1) == cudaSuccess) e->last_token_bytes_ms = ms; else cudaGetLastError();
    return LATOK_B200_OK;
}

int latok_b200_token_bytes_ms(latok_b200_engine *e, float *ms)
{
    if (!e || !ms) return fail(LATOK_B200_EINVAL, "engine or ms is NULL");
    *ms = e->last_token_bytes_ms;
    return LATOK_B200_OK;
}

int latok_b200_device_results(latok_b200_engine *e, const int8_t **splits, const int64_t **char_offsets,
                              const int32_t **spans, const int64_t **tok_offsets, const int8_t **tok_feats,
                              const int8_t **matrix)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (!e->front() || !e->front()->submitted) return fail(LATOK_B200_ESTATE, "no batch submitted");
    Batch &b = *e->front();
    if (splits) *splits = b.d_splits.p;
    if (char_offsets) *char_offsets = (const int64_t *)b.d_char_off.p;
    if (spans) *spans = b.d_spans.p;
    if (tok_offsets) *tok_offsets = (const int64_t *)b.d_tok_off.p;
    if (tok_feats) *tok_feats = b.d_feats.p;
    if (matrix) *matrix = b.d_matrix.p;
    return LATOK_B200_OK;
}

int latok_b200_timer_begin(latok_b200_engine *e)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (int r = set_device(e)) return r;
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaEventRecord(e->ev_t0, e->stream));
    return LATOK_B200_OK;
}

int latok_b200_timer_end(latok_b200_engine *e, float *elapsed_ms)
{
    if (!e || !elapsed_ms) return fail(LATOK_B200_EINVAL, "engine or elapsed_ms is NULL");
    if (int r = set_device(e)) return r;
    CU(cudaEventRecord(e->ev_t1, e->stream));
    CU(cudaEventSynchronize(e->ev_t1));
    CU(cudaEventElapsedTime(elapsed_ms, e->ev_t0, e->ev_t1));
    return LATOK_B200_OK;
}

int latok_b200_launch_count(latok_b200_engine *e, int64_t *launches)
{
    if (!e || !launches) return fail(LATOK_B200_EINVAL, "engine or launches is NULL");
    *launches = e->launches;
    return LATOK_B200_OK;
}

int latok_b200_last_stats(latok_b200_engine *e, float *tokenize_kernel_ms, int64_t *lookahead_walks)
{
    FRONT(e, b);
    if (int r = size_batch(e, b)) return r;
    if (tokenize_kernel_ms) *tokenize_kernel_ms = b.kernel_ms;
    if (lookahead_walks) *lookahead_walks = b.walks;
    return LATOK_B200_OK;
}

int latok_b200_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) return fail(LATOK_B200_EINVAL, "ptr is NULL");
    CU(cudaMallocHost(ptr, bytes ? bytes : 1));
    return LATOK_B200_OK;
}

int latok_b200_host_free(void *ptr)
{
    if (ptr) CU(cudaFreeHost(ptr));
    return LATOK_B200_OK;
}

int latok_b200_gen_parse_matrix(latok_b200_engine *e, const uint8_t *utf8, int64_t n_bytes, int64_t *n_chars, int8_t *out)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (n_bytes < 0 || (n_bytes > 0 && !utf8)) return fail(LATOK_B200_EINVAL, "must specify string to generate the parse matrix for");
    const int64_t offs[2] = {0, n_bytes};
    if (int r = latok_b200_submit(e, utf8, offs, 1, LATOK_B200_MATRIX)) return r;
    int64_t C = 0;
    if (int r = latok_b200_sizes(e, &C, nullptr)) return r;
    if (n_chars) *n_chars = C;
    if (out) return latok_b200_fetch(e, C, 0, 1, nullptr, nullptr, nullptr, nullptr, nullptr, out);
    return LATOK_B200_OK;
}

int latok_b200_gen_block_mask(latok_b200_engine *e, const int8_t *a1, int64_t stride1, const int8_t *a2, int64_t stride2,
                              int64_t n, int8_t *out)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (n < 0) return fail(LATOK_B200_EINVAL, "must specify 1d numpy arrays of matching length");
    if (n == 0) return LATOK_B200_OK;
    if (!a1 || !a2 || !out) return fail(LATOK_B200_EINVAL, "must specify two aligning 1d numpy array args");
    if (int r = set_device(e)) return r;
    if (int r = e->d_scratch.ensure((size_t)n * 2)) return r;
    if (int r = e->d_scratch2.ensure((size_t)n)) return r;
    if (int r = e->d_scratch3.ensure((size_t)n)) return r;
    std::vector<int8_t> h((size_t)n * 2);
    for (int64_t i = 0; i < n; ++i) { h[(size_t)i] = a1[i * stride1]; h[(size_t)(n + i)] = a2[i * stride2]; }
    CU(cudaMemcpyAsync(e->d_scratch.p, h.data(), (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
    CU(launch_block_mask((const int8_t *)e->d_scratch.p, 1, (const int8_t *)e->d_scratch.p + n, 1, n,
                         (int8_t *)e->d_scratch2.p, e->d_scratch3.p, e->stream));
    e->launches += 1;
    CU(cudaMemcpyAsync(out, e->d_scratch2.p, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return LATOK_B200_OK;
}

int latok_b200_combine_matrix_rows(latok_b200_engine *e, const int8_t *m, int64_t m_rows, int64_t m_cols, int64_t stride_row,
                                   int64_t stride_col, const int8_t *idx, int idx_rows, int idx_cols, int8_t *out)
{
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (m_rows < 0 || m_cols < 0 || idx_rows < 0 || idx_cols < 0) return fail(LATOK_B200_EINVAL, "must specify 2d numpy array args");
    if (stride_row < 0 || stride_col < 0) return fail(LATOK_B200_EINVAL, "negative strides are not supported");
    if (m_cols == 0) return LATOK_B200_OK;
    if (!m || !out || (idx_rows && !idx)) return fail(LATOK_B200_EINVAL, "must specify 2d m and idxs matrices");
    if (int r = set_device(e)) return r;
    const size_t extent = m_rows ? (size_t)((m_rows - 1) * stride_row + (m_cols - 1) * stride_col + 1) : 0;
    const size_t n_idx = (size_t)idx_rows * (size_t)(idx_cols ? idx_cols : 1);
    if (int r = e->d_scratch.ensure(extent + 16)) return r;
    if (int r = e->d_scratch2.ensure((size_t)m_cols)) return r;
    if (int r = e->d_scratch3.ensure(n_idx + 16)) return r;
    if (extent) CU(cudaMemcpyAsync(e->d_scratch.p, m, extent, cudaMemcpyHostToDevice, e->stream));
    if (n_idx) CU(cudaMemcpyAsync(e->d_scratch3.p, idx, n_idx, cudaMemcpyHostToDevice, e->stream));
    CU(launch_combine_rows((const int8_t *)e->d_scratch.p, m_rows, m_cols, stride_row, stride_col,
                           (const int8_t *)e->d_scratch3.p, idx_rows, idx_cols, (int8_t *)e->d_scratch2.p, e->stream));
    e->launches += 1;
    CU(cudaMemcpyAsync(out, e->d_scratch2.p, (size_t)m_cols, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return LATOK_B200_OK;
}

// ---- token vocabulary (kernels: latok_vocab.cu) ---------------------------------------------------------------------
struct latok_b200_vocab {
    int device = 0;
    unsigned long long hmask = ~0ULL;
    long long cap = 0;                              // table slots, a power of two; the load limit is cap / 2 keys
    long long n_keys = 0, key_bytes = 0;
    DevBuf<VocabSlot> table;
    DevBuf<unsigned long long> first_occ;           // [cap]
    DevBuf<uint8_t> arena;                          // key bytes in id order
    DevBuf<long long> key_off;                      // [n_keys + 1]
    DevBuf<long long> counts;                       // [n_keys]
    DevBuf<uint32_t> slot;                          // per token of the largest batch: its slot
    DevBuf<int32_t> rank;                           // per token: first-occurrence flags, then new ids, then the ids
    DevBuf<uint8_t> scan_tmp, imp_bytes;
    DevBuf<longlong2> imp_rng;
    DevBuf<long long> imp_w;                        // a merge from another device: its counts, then its key offsets
    DevBuf<VocabStatus> st;
    PinBuf<VocabStatus> h_st;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_ms = 0.f;
};

static VocabParams vocab_params(latok_b200_vocab *v)
{
    VocabParams p;
    memset(&p, 0, sizeof p);
    p.table = v->table.p; p.mask = (unsigned long long)v->cap - 1; p.hmask = v->hmask;
    p.arena = v->arena.p; p.key_off = v->key_off.p; p.n_keys = v->n_keys;
    p.first_occ = v->first_occ.p; p.slot = v->slot.p; p.rank = v->rank.p;
    p.counts = reinterpret_cast<unsigned long long *>(v->counts.p); p.st = v->st.p;
    p.limit = (unsigned long long)(v->cap / 2 > v->n_keys ? v->cap / 2 - v->n_keys : 0);
    return p;
}

// an empty table of `cap` slots that holds the committed keys: drops the claims of a batch that did not commit
static int vocab_rebuild(latok_b200_vocab *v, long long cap, int n_sm, cudaStream_t s)
{
    if (cap > (1LL << 31)) return fail(LATOK_B200_ENOMEM, "a vocabulary table holds at most 2^31 slots");
    if (cap != v->cap) {
        CU(cudaStreamSynchronize(s));
        if (int r = v->table.ensure((size_t)cap)) return r;
        if (int r = v->first_occ.ensure((size_t)cap)) return r;
        v->cap = cap;
    }
    CU(cudaMemsetAsync(v->table.p, 0, (size_t)cap * sizeof(VocabSlot), s));
    CU(cudaMemsetAsync(v->st.p, 0, sizeof(VocabStatus), s));
    CU(launch_vocab(VOCAB_REHASH, vocab_params(v), 0, n_sm, s));
    return 0;
}

// claims the keys text[rng[k].x, rng[k].y) (k < n) that the vocabulary lacks: *n_new keys of *new_bytes bytes, claimed
// but not committed.  A batch that passes the load limit grows the table 4x and runs again.
static int vocab_insert(latok_b200_vocab *v, const uint8_t *text, const longlong2 *rng, long long n, int n_sm, cudaStream_t s,
                        long long *n_new, long long *new_bytes)
{
    if (int r = v->slot.ensure((size_t)n)) return r;
    if (int r = v->rank.ensure((size_t)n + 1)) return r;
    for (int attempt = 0; attempt < 24; ++attempt) {
        VocabParams p = vocab_params(v);
        p.text = text; p.rng = rng; p.n = n;
        CU(cudaMemsetAsync(v->first_occ.p, 0xFF, (size_t)v->cap * sizeof(unsigned long long), s));
        CU(cudaMemsetAsync(v->st.p, 0, sizeof(VocabStatus), s));
        CU(launch_vocab(VOCAB_INSERT, p, 0, n_sm, s));
        CU(launch_vocab(VOCAB_FLAG, p, 0, n_sm, s));
        CU(cudaEventRecord(v->ev[1], s));
        CU(cudaMemcpyAsync(v->h_st.p, v->st.p, sizeof(VocabStatus), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        const VocabStatus st = *v->h_st.p;
        if (!st.overflow) { *n_new = (long long)st.n_new; *new_bytes = (long long)st.new_bytes; return 0; }
        if (int r = vocab_rebuild(v, v->cap * 4, n_sm, s)) return r;
    }
    return fail(LATOK_B200_EINTERNAL, "vocabulary insert did not converge");
}

// gives the claimed keys of vocab_insert the ids n_keys .. n_keys + n_new - 1 in token order and copies them into the arena
static int vocab_commit(latok_b200_vocab *v, const uint8_t *text, const longlong2 *rng, long long n, long long n_new,
                        long long new_bytes, int n_sm, cudaStream_t s)
{
    if (v->n_keys + n_new > INT32_MAX) {
        if (int r = vocab_rebuild(v, v->cap, n_sm, s)) return r;
        CU(cudaStreamSynchronize(s));
        return fail(LATOK_B200_EINVAL, "a vocabulary holds at most 2^31 - 1 keys");
    }
    CU(cudaEventRecord(v->ev[2], s));
    if (!n_new) return 0;
    if (int r = grow_keep(v->arena, (size_t)(v->key_bytes + new_bytes), (size_t)v->key_bytes, s)) return r;
    if (int r = grow_keep(v->key_off, (size_t)(v->n_keys + n_new + 1), (size_t)v->n_keys + 1, s)) return r;
    if (int r = grow_keep(v->counts, (size_t)(v->n_keys + n_new), (size_t)v->n_keys, s)) return r;
    CU(cudaMemsetAsync(v->counts.p + v->n_keys, 0, (size_t)n_new * sizeof(long long), s));
    VocabParams p = vocab_params(v);
    p.text = text; p.rng = rng; p.n = n;
    size_t need = 0, need1 = 0;
    CU(vocab_scan(0, nullptr, &need, p, n_new, v->key_bytes, s));
    CU(vocab_scan(1, nullptr, &need1, p, n_new, v->key_bytes, s));
    if (need1 > need) need = need1;
    if (need > v->scan_tmp.cap) { CU(cudaStreamSynchronize(s)); if (int r = v->scan_tmp.ensure(need)) return r; }
    CU(vocab_scan(0, v->scan_tmp.p, &need, p, n_new, v->key_bytes, s));
    CU(launch_vocab(VOCAB_LENS, p, n_new, n_sm, s));
    CU(vocab_scan(1, v->scan_tmp.p, &need, p, n_new, v->key_bytes, s));
    CU(launch_vocab(VOCAB_COMMIT, p, n_new, n_sm, s));
    v->n_keys += n_new;
    v->key_bytes += new_bytes;
    return 0;
}

// One batch into v (encode, import, merge): the keys text[rng[k].x, rng[k].y) (k < n, on v's device) are inserted and
// committed, then, with `count` or ids, the count kernel writes the id of every key into ids and adds 1 per key, or
// weight[k] with weights, to its count.  strict: every key must be new (import); otherwise nothing is committed and
// the call is EINVAL.  Records v->ev[1] (insert done) and v->ev[2] (commit started).
static int vocab_add(latok_b200_engine *e, latok_b200_vocab *v, const uint8_t *text, const longlong2 *rng, long long n,
                     bool strict, bool count, const long long *weight, int32_t *ids)
{
    cudaStream_t s = e->stream;
    long long n_new = 0, new_bytes = 0;
    if (int r = vocab_insert(v, text, rng, n, e->n_sm, s, &n_new, &new_bytes)) return r;
    if (strict && n_new != n) {
        if (int r = vocab_rebuild(v, v->cap, e->n_sm, s)) return r;
        CU(cudaStreamSynchronize(s));
        return fail(LATOK_B200_EINVAL, "duplicate keys: %lld of the %lld keys are new to the vocabulary", n_new, n);
    }
    if (int r = vocab_commit(v, text, rng, n, n_new, new_bytes, e->n_sm, s)) return r;
    e->launches += 5;
    if (!count && !ids) return 0;
    VocabParams p = vocab_params(v);
    if (!count) p.counts = nullptr;
    p.weight = weight; p.ids = ids;
    p.text = text; p.rng = rng; p.n = n;
    CU(launch_vocab(VOCAB_COUNT, p, 0, e->n_sm, s));
    e->launches += 1;
    return 0;
}

static float elapsed(cudaEvent_t a, cudaEvent_t b)
{
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); ms = 0.f; }
    return ms;
}

int latok_b200_vocab_create(latok_b200_engine *e, int64_t expected_keys, latok_b200_vocab **out)
{
    if (!out) return fail(LATOK_B200_EINVAL, "out is NULL");
    *out = nullptr;
    if (!e) return fail(LATOK_B200_EINVAL, "engine is NULL");
    if (expected_keys < 0 || expected_keys > INT32_MAX) return fail(LATOK_B200_EINVAL, "expected_keys must be in [0, 2^31 - 1]");
    if (int r = set_device(e)) return r;
    latok_b200_vocab *v = new (std::nothrow) latok_b200_vocab();
    if (!v) return fail(LATOK_B200_ENOMEM, "out of host memory");
    v->device = e->device;
    // test seam: keep only the low n bits of the hash, so that tests can force collisions and long probe chains
    if (const char *hb = getenv("LATOK_B200_VOCAB_HASH_BITS")) {
        const int bits = atoi(hb);
        if (bits >= 1 && bits < 64) v->hmask = (1ULL << bits) - 1;
    }
    long long cap = 64;
    while (cap < 2 * expected_keys) cap <<= 1;
    const int rc = [&]() -> int {
        for (cudaEvent_t &ev : v->ev) CU(cudaEventCreate(&ev));
        if (int r = v->st.ensure(1)) return r;
        if (int r = v->h_st.ensure(1)) return r;
        if (int r = v->key_off.ensure(1, true)) return r;
        if (int r = v->table.ensure((size_t)cap)) return r;
        if (int r = v->first_occ.ensure((size_t)cap)) return r;
        v->cap = cap;
        CU(cudaMemset(v->table.p, 0, (size_t)cap * sizeof(VocabSlot)));
        CU(cudaDeviceSynchronize());
        return 0;
    }();
    if (rc) { latok_b200_vocab_destroy(v); return rc; }
    *out = v;
    return LATOK_B200_OK;
}

int latok_b200_vocab_destroy(latok_b200_vocab *v)
{
    if (!v) return LATOK_B200_OK;
    cudaSetDevice(v->device);
    v->table.release(); v->first_occ.release(); v->arena.release(); v->key_off.release(); v->counts.release();
    v->slot.release(); v->rank.release(); v->scan_tmp.release(); v->imp_bytes.release(); v->imp_rng.release();
    v->imp_w.release();
    v->st.release(); v->h_st.release();
    for (cudaEvent_t ev : v->ev) if (ev) cudaEventDestroy(ev);
    delete v;
    return LATOK_B200_OK;
}

int latok_b200_vocab_encode(latok_b200_engine *e, latok_b200_vocab *v, int add, int32_t unk_id, int64_t cap_tokens,
                            int32_t *ids, int on_device)
{
    if (!v) return fail(LATOK_B200_EINVAL, "vocabulary is NULL");
    FRONT(e, b);
    if (v->device != e->device) return fail(LATOK_B200_EINVAL, "the vocabulary is on device %d, the engine on device %d", v->device, e->device);
    if (int r = size_batch(e, b)) return r;
    if (!(b.what & LATOK_B200_SPANS)) return fail(LATOK_B200_ESTATE, "spans were not requested at submit");
    const long long T = b.n_tokens;
    if (cap_tokens < T) return fail(LATOK_B200_EINVAL, "cap_tokens = %lld, the batch has %lld tokens", (long long)cap_tokens, T);
    if (ids && on_device && ((uintptr_t)ids & 3u) != 0) return fail(LATOK_B200_EINVAL, "a device ids array must be 4-byte aligned");
    v->last_ms = 0.f;
    if (!T || (!add && !ids)) return LATOK_B200_OK;
    if (int r = e->d_tok_bytes.ensure(2 * (size_t)T)) return r;
    if (int r = v->rank.ensure((size_t)T + 1)) return r;
    cudaStream_t s = e->stream;
    CU(cudaStreamWaitEvent(s, b.ev_kdone, 0));
    CU(cudaEventRecord(v->ev[0], s));
    if (int r = enqueue_token_bytes(e, b, e->d_tok_bytes.p)) return r;
    const longlong2 *rng = reinterpret_cast<const longlong2 *>(e->d_tok_bytes.p);
    VocabParams p;
    if (add) {
        p.ids = ids ? (on_device ? ids : v->rank.p) : nullptr;
        if (int r = vocab_add(e, v, b.cur_in, rng, T, false, true, nullptr, p.ids)) return r;
        CU(cudaEventRecord(v->ev[3], s));
    } else {
        p = vocab_params(v);
        p.ids = on_device ? ids : v->rank.p;
        p.unk = unk_id;
        p.text = b.cur_in; p.rng = rng; p.n = T;
        CU(launch_vocab(VOCAB_LOOKUP, p, 0, e->n_sm, s));
        CU(cudaEventRecord(v->ev[1], s));
        e->launches += 1;
    }
    if (ids && !on_device) CU(cudaMemcpyAsync(ids, p.ids, (size_t)T * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(b.ev_kdone, s));          // the set's inputs are in use until here
    CU(cudaStreamSynchronize(s));
    v->last_ms = elapsed(v->ev[0], v->ev[1]) + (add ? elapsed(v->ev[2], v->ev[3]) : 0.f);
    return LATOK_B200_OK;
}

int latok_b200_vocab_size(latok_b200_vocab *v, int64_t *n_keys, int64_t *key_bytes, int64_t *table_slots)
{
    if (!v) return fail(LATOK_B200_EINVAL, "vocabulary is NULL");
    if (n_keys) *n_keys = v->n_keys;
    if (key_bytes) *key_bytes = v->key_bytes;
    if (table_slots) *table_slots = v->cap;
    return LATOK_B200_OK;
}

int latok_b200_vocab_export(latok_b200_vocab *v, int64_t cap_keys, int64_t cap_bytes, uint8_t *bytes, int64_t *offsets,
                            int64_t *counts)
{
    if (!v) return fail(LATOK_B200_EINVAL, "vocabulary is NULL");
    if ((offsets || counts) && cap_keys < v->n_keys)
        return fail(LATOK_B200_EINVAL, "cap_keys = %lld, the vocabulary has %lld keys", (long long)cap_keys, v->n_keys);
    if (bytes && cap_bytes < v->key_bytes)
        return fail(LATOK_B200_EINVAL, "cap_bytes = %lld, the keys have %lld bytes", (long long)cap_bytes, v->key_bytes);
    CU(cudaSetDevice(v->device));
    if (bytes && v->key_bytes) CU(cudaMemcpy(bytes, v->arena.p, (size_t)v->key_bytes, cudaMemcpyDeviceToHost));
    if (offsets) CU(cudaMemcpy(offsets, v->key_off.p, ((size_t)v->n_keys + 1) * sizeof(long long), cudaMemcpyDeviceToHost));
    if (counts && v->n_keys) CU(cudaMemcpy(counts, v->counts.p, (size_t)v->n_keys * sizeof(long long), cudaMemcpyDeviceToHost));
    return LATOK_B200_OK;
}

int latok_b200_vocab_import(latok_b200_engine *e, latok_b200_vocab *v, const uint8_t *bytes, const int64_t *offsets,
                            int64_t n_keys, const int64_t *counts)
{
    if (!e || !v) return fail(LATOK_B200_EINVAL, "engine or vocabulary is NULL");
    if (v->device != e->device) return fail(LATOK_B200_EINVAL, "the vocabulary is on device %d, the engine on device %d", v->device, e->device);
    if (n_keys < 0) return fail(LATOK_B200_EINVAL, "n_keys must be >= 0");
    if (n_keys == 0) return LATOK_B200_OK;
    if (!offsets || !bytes) return fail(LATOK_B200_EINVAL, "must specify the key bytes and offsets (n_keys + 1 entries)");
    if (offsets[0] != 0) return fail(LATOK_B200_EINVAL, "offsets[0] must be 0");
    for (int64_t i = 0; i < n_keys; ++i)
        if (offsets[i + 1] <= offsets[i]) return fail(LATOK_B200_EINVAL, "key %lld is empty (offsets must increase)", (long long)i);
    if (v->n_keys + n_keys > INT32_MAX) return fail(LATOK_B200_EINVAL, "a vocabulary holds at most 2^31 - 1 keys");
    if (int r = set_device(e)) return r;
    cudaStream_t s = e->stream;
    const long long nb = offsets[n_keys];
    std::vector<longlong2> rng((size_t)n_keys);
    for (int64_t i = 0; i < n_keys; ++i) rng[(size_t)i] = make_longlong2(offsets[i], offsets[i + 1]);
    CU(cudaStreamSynchronize(s));
    if (int r = v->imp_bytes.ensure((size_t)nb)) return r;
    if (int r = v->imp_rng.ensure((size_t)n_keys)) return r;
    CU(cudaMemcpyAsync(v->imp_bytes.p, bytes, (size_t)nb, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(v->imp_rng.p, rng.data(), (size_t)n_keys * sizeof(longlong2), cudaMemcpyHostToDevice, s));
    CU(cudaEventRecord(v->ev[0], s));
    const long long first = v->n_keys;
    if (int r = vocab_add(e, v, v->imp_bytes.p, v->imp_rng.p, n_keys, true, false, nullptr, nullptr)) return r;
    if (counts) CU(cudaMemcpyAsync(v->counts.p + first, counts, (size_t)n_keys * sizeof(long long), cudaMemcpyHostToDevice, s));
    CU(cudaEventRecord(v->ev[3], s));
    CU(cudaStreamSynchronize(s));
    v->last_ms = elapsed(v->ev[0], v->ev[1]) + elapsed(v->ev[2], v->ev[3]);
    return LATOK_B200_OK;
}

int latok_b200_vocab_merge(latok_b200_engine *e, latok_b200_vocab *dst, const latok_b200_vocab *src, int32_t *map, int on_device)
{
    if (!e || !dst || !src) return fail(LATOK_B200_EINVAL, "engine or vocabulary is NULL");
    if (dst->device != e->device) return fail(LATOK_B200_EINVAL, "the vocabulary is on device %d, the engine on device %d", dst->device, e->device);
    if (src == dst) return fail(LATOK_B200_EINVAL, "a vocabulary cannot be merged into itself");
    if (map && on_device && ((uintptr_t)map & 3u) != 0) return fail(LATOK_B200_EINVAL, "a device map must be 4-byte aligned");
    dst->last_ms = 0.f;
    const long long n = src->n_keys;
    if (!n) return LATOK_B200_OK;
    if (int r = set_device(e)) return r;
    cudaStream_t s = e->stream;
    CU(cudaStreamSynchronize(s));
    if (int r = dst->imp_rng.ensure((size_t)n)) return r;
    CU(cudaEventRecord(dst->ev[0], s));
    // the source's keys, offsets and counts: read in place on the same device, else copied into the staging buffers
    // (imp_w = counts [n], then key_off [n + 1]) on dst's stream.  cudaMemcpyPeerAsync needs no peer access; the
    // source is stable while the copies run because every vocabulary call ends synchronised.
    const uint8_t *text = src->arena.p;
    const long long *key_off = src->key_off.p, *weight = src->counts.p;
    if (src->device != dst->device) {
        if (int r = dst->imp_bytes.ensure((size_t)src->key_bytes)) return r;
        if (int r = dst->imp_w.ensure(2 * (size_t)n + 1)) return r;
        CU(cudaMemcpyPeerAsync(dst->imp_bytes.p, dst->device, src->arena.p, src->device, (size_t)src->key_bytes, s));
        CU(cudaMemcpyPeerAsync(dst->imp_w.p, dst->device, src->counts.p, src->device, (size_t)n * sizeof(long long), s));
        CU(cudaMemcpyPeerAsync(dst->imp_w.p + n, dst->device, src->key_off.p, src->device, ((size_t)n + 1) * sizeof(long long), s));
        text = dst->imp_bytes.p; weight = dst->imp_w.p; key_off = dst->imp_w.p + n;
    }
    CU(launch_vocab_ranges(key_off, n, dst->imp_rng.p, e->n_sm, s));
    e->launches += 1;
    int32_t *ids = map ? (on_device ? map : nullptr) : nullptr;
    if (map && !on_device) {
        if (int r = dst->rank.ensure((size_t)n + 1)) return r;
        ids = dst->rank.p;
    }
    if (int r = vocab_add(e, dst, text, dst->imp_rng.p, n, false, true, weight, ids)) return r;
    CU(cudaEventRecord(dst->ev[3], s));
    if (map && !on_device) CU(cudaMemcpyAsync(map, ids, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    dst->last_ms = elapsed(dst->ev[0], dst->ev[1]) + elapsed(dst->ev[2], dst->ev[3]);
    return LATOK_B200_OK;
}

int latok_b200_vocab_clear(latok_b200_vocab *v)
{
    if (!v) return fail(LATOK_B200_EINVAL, "vocabulary is NULL");
    CU(cudaSetDevice(v->device));
    CU(cudaMemsetAsync(v->table.p, 0, (size_t)v->cap * sizeof(VocabSlot), 0));
    CU(cudaStreamSynchronize(0));
    v->n_keys = 0;
    v->key_bytes = 0;
    v->last_ms = 0.f;
    return LATOK_B200_OK;
}

int latok_b200_vocab_last_ms(latok_b200_vocab *v, float *ms)
{
    if (!v || !ms) return fail(LATOK_B200_EINVAL, "vocabulary or ms is NULL");
    *ms = v->last_ms;
    return LATOK_B200_OK;
}

}  // extern "C"
