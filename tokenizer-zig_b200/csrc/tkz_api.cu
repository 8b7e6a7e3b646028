// tkz_api.cu -- device layer of the C ABI (include/tokzig_b200.h): context, device arenas, model upload, and the
// batch-encode pipelines that replace the caller loop over Tokenizer.encode (src/lib.zig:109-160):
//
//   [K0 normalise-compact]  only when the normalizer drops bytes (struct BertNormalizer, normalizer.zig:47-73)
//   encode_slices           any model with a pre-tokenizer: pass A tokenizes 1 KiB slices, pass B writes (tkz_slices.cuh)
//   encode_words            per-occurrence: K1 pre-token spans (pretokenizer.zig:49-241), K3 bpe / K4 wordpiece per
//                           pre-token (bpe.zig:173-263 / wordpiece.zig:141-222), scans to CSR offsets, K5 emit
//   shared epilogue         output arrays, padding + template tokens, stage times, result (encoding.zig:246-294, 363-463)
//
// There is no CPU fallback: without a usable CUDA device every entry point fails with TKZ_ERR_CUDA.
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <array>
#include <chrono>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/tokzig_b200.h"
#include "tkz_bpe.cuh"
#include "tkz_bpe_block.cuh"
#include "tkz_bpe_grid.cuh"
#include "tkz_common.cuh"
#include "tkz_decode.cuh"
#include "tkz_emit.cuh"
#include "tkz_fast.cuh"
#include "tkz_overflow.cuh"
#include "tkz_slices.cuh"
#include "tkz_scan.cuh"
#include "tkz_split.cuh"
#include "tkz_wordpiece.cuh"

using namespace tkz;

namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};
struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct tkz_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    std::string err;
    bool has_model = false;
    DevModel dm{}, dm_post{};
    // model tables
    DevBuf t_lut, t_lut_post, t_char_ascii, t_char_tab, t_merges, t_merge_win, t_wp_tab, t_wp_pool;
    // arenas (grow-only; replace src/arena.zig)
    DevBuf a_text, a_doc_off, a_norm_text, a_norm_doc_off, a_chunk, a_tiles, a_word_start, a_word_end, a_word_doc, a_doc_word_off,
        a_word_ntok, a_pool_id, a_pool_s, a_pool_e, a_pool_rk, a_scan_tmp, a_ctrl;
    // output arrays, double-buffered so that the D2H copy of one chunk overlaps the kernels of the next (tkz_encode_batch); a
    // third set stages the untruncated tokens that TKZ_HF_OVERFLOW cuts into rows (tkz_overflow.cuh)
    struct OutSet { DevBuf doc_tok_off, ids, off, attn, type, special, off16, ids16, spans, wide, wid, row_tok_off, doc_row_off; } outs[3];
    int out_sel = 0;
    OutSet& O() { return outs[out_sel]; }
    DevBuf in_text[2], in_doc_off[2];
    HostBuf h_doc_stage[2];
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    uint64_t chunk_bytes = 64ull << 20;
    // slice pipeline arenas (tkz_slices.cuh)
    DevBuf a_long_start, a_long_end, a_long_ntok, a_long_slice, a_long_ins, a_tile_ntok, a_tile_ntok_inline, a_tile_tok_off, a_tile_long,
        a_doc_tok_local, a_doc_tok_start, a_doc_real, a_upool, a_tile_doc_lo, a_g_first, a_g_win, a_g_flag, a_big,
        a_slice_nword, a_doc_word_local, a_doc_word_base, a_long_k,        // word ids (TKZ_OUT_WORD_IDS)
        a_row_real, a_row_doc;                                             // overflowing windows (TKZ_HF_OVERFLOW)
    bool use_dedup = true;                // TKZ_NO_DEDUP=1: per-occurrence pipeline even with a pre-tokenizer (A/B switch of the parity tests)
    DevBuf a_wtable, a_lscratch, a_tok_id;
    bool has_iso = false;                 // the class table isolates some byte (punctuation split)
    ClassRanges cr{}, cr_post{};          // byte classes as ranges (raw bytes / bytes already normalised by K0)
    bool narrow_records = true;           // TKZ_TOK_RECORD=wide: u32 ids in the token stream even for 16-bit vocabularies (A/B switch)
    // chunks of ONE host-buffer call share the word table and the record pool of the slice pipeline: the first chunk starts from an
    // empty table, the later ones find the call's frequent words already tokenized (every call starts cold)
    bool call_keep = false;               // inside a chunked host-buffer call
    bool kept_valid = false;              // the table of the previous chunk can be reused
    uint64_t call_bytes = 0;              // text bytes of the whole call (sizes the shared table)
    uint32_t kept_tcap = 0, kept_upool_count = 0; uint64_t kept_upool_cap = 0, call_uniq = 0;
    bool force_lut = false;               // TKZ_CLASSIFY=lut: per-byte look-up even when the class table fits ranges (A/B switch)
    DevBuf a_huge_w, a_huge_base, a_huge_done, a_grid_state, a_grid_words;   // bpe_grid_kernel (tkz_bpe_grid.cuh)
    bool use_grid = true;                 // TKZ_NO_GRID=1: huge words stay with one block each (A/B switch of the parity tests)
    uint32_t grid_min_len = 12289;        // shortest word (bytes) that goes to bpe_grid_kernel (TKZ_GRID_MIN_LEN)
    bool grid_used = false;               // the last encode ran bpe_grid_kernel
    bool retried = false;                 // the last encode re-ran the slice pipeline with worst-case capacities
    int grid_blocks = 0;                  // co-resident blocks of bpe_grid_kernel (0: cooperative launch not available)
    uint64_t tw_uniq_hist = 0;            // most unique words seen in one batch: sizes the next batch's word table
    uint64_t tw_upool_hist = 0;           // most token records used by one batch
    double tw_tok_per_byte = 0.0;         // densest batch so far: sizes the token stream
    HostBuf h_ctrl, h_doc_tok_off, h_ids, h_off, h_attn, h_type, h_special, h_off16, h_ids16, h_spans, h_wide, h_wid, h_row_tok_off, h_doc_row_off;
    DevBuf a_fast_heap, a_word_aux;       // FastTokenizer mode (tkz_fast.cuh)
    bool ids16_ok = false;                // every id the model can emit is below 65536 (TKZ_OUT_IDS_U16)
    uint32_t max_id = 0;                  // largest id the model can emit (word ids need it below 2^22: TW_REC_WORD)
    // decode direction (tkz_decode.cuh)
    bool has_decode = false;
    DecodeTables dt{};
    DevBuf t_dec_bytes, t_dec_off, t_dec_special, a_dec_ids, a_dec_seq_off, a_dec_len, a_dec_raw, a_dec_out, a_dec_olen, a_dec_boff;
    HostBuf h_dec_bytes, h_dec_off;
    unsigned long long* h_ctrl_dev = nullptr;   // device alias of h_ctrl (mapped pinned memory): scalars are read back by a tiny
                                                // kernel, not by a D2H memcpy that would queue behind the result copies
    uint64_t arena_bytes = 0;
    tkz_stats stats{};
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // stage boundaries of the last encode
};

namespace {

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                          \
            return e__ == cudaErrorMemoryAllocation ? TKZ_ERR_OOM : TKZ_ERR_CUDA;                    \
        }                                                                                            \
    } while (0)

int ensure(tkz_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return TKZ_OK;
    if (b.p) {
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->s_h2d) CK(cudaStreamSynchronize(ctx->s_h2d));
        if (ctx->s_d2h) CK(cudaStreamSynchronize(ctx->s_d2h));
        CK(cudaFree(b.p)); ctx->arena_bytes -= b.cap; b.p = nullptr; b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;      // head-room so steady-state batches of similar size do not re-allocate
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { want = bytes; e = cudaMalloc(&b.p, want); }
    if (e != cudaSuccess) { ctx->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); b.p = nullptr; return TKZ_ERR_OOM; }
    b.cap = want; ctx->arena_bytes += want;
    return TKZ_OK;
}
int ensure_host(tkz_ctx* ctx, HostBuf& b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return TKZ_OK;
    if (b.p) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFreeHost(b.p)); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaHostAlloc(&b.p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { ctx->err = std::string("cudaHostAlloc: ") + cudaGetErrorString(e); b.p = nullptr; return TKZ_ERR_OOM; }
    b.cap = want;
    return TKZ_OK;
}
void release(DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
void release_host(HostBuf& b) { if (b.p) cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }

#define TRY(x) do { int rc__ = (x); if (rc__ != TKZ_OK) return rc__; } while (0)

// every entry point runs on its context's device and gives the caller's current device back on every return path
struct DeviceGuard {
    int prev = -1; bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(ctx) DeviceGuard guard__((ctx)->device); if (!guard__.ok) { (ctx)->err = "cudaSetDevice failed"; return TKZ_ERR_CUDA; }

int upload(tkz_ctx* ctx, DevBuf& b, const void* src, size_t bytes) {
    TRY(ensure(ctx, b, bytes));
    if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return TKZ_OK;
}

uint32_t pow2_at_least(uint64_t n) { uint32_t c = 2; while (c < n) c <<= 1; return c; }

__global__ void ctrl_reset_kernel(unsigned long long* ctrl) {
    // ctrl[0] = error word, ctrl[1] = work counter (u32 view), ctrl[2..4] = read-back scalars,
    // [11..12], [17], [20..21] block-kernel work counters, [13..15] long-word length classes, [18..19] huge-word list (count, bytes)
    // slice pipeline: [5] entry count, [6] n_uniq | n_uncached << 32, [7] n_long, [8] abort, [9] upool | lscratch << 32,
    //                [10] n_words, [16] big-copy list, [22] tokens of the long words, [23] wide-offset list
    // per-occurrence pipeline: high half of [9] big-copy list
    ctrl[0] = TKZ_ERRW_NONE;
    for (int i = 1; i < 32; i++) ctrl[i] = 0;
}
// scalars -> mapped host memory, in stream order (replaces small D2H memcpys: those share the copy engine's queue with the
// multi-megabyte result copies of the previous chunk and would stall the kernels of this one behind them)
// chunk-relative CSR offsets -> call-relative (host path: a chunk's doc_tok_off is shifted on the device before it is copied out)
__global__ void add_base_u64_kernel(unsigned long long* __restrict__ p, uint64_t n, unsigned long long base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] += base;
}
__global__ void set_u32_kernel(unsigned int* p, unsigned int v) { *p = v; }
__global__ void publish_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint32_t n) {
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
}
int readback(tkz_ctx* ctx, unsigned long long* h_dst, const void* d_src, size_t bytes) {
    unsigned long long* hbase = (unsigned long long*)ctx->h_ctrl.p;
    uint32_t* dst = (uint32_t*)(ctx->h_ctrl_dev + (h_dst - hbase));
    publish_kernel<<<1, 32, 0, ctx->stream>>>((const uint32_t*)d_src, dst, (uint32_t)(bytes / 4));
    return TKZ_OK;
}
// word-length classes of the BPE kernels: [0] 65..2048 bytes, [1] > 2048, [2] > 12288 (needs global state arrays)
constexpr uint32_t BB_WARP_MAX = 64, BB_MINI_MAX = 512, BB_TINY_MAX = 1024, BB_SMALL_MAX = 2048, BB_MID_MAX = 4096, BB_BIG_CAP = 12288;
__global__ void len_class_count_kernel(const uint32_t* word_start, const uint32_t* word_end, uint32_t n_fixed, const unsigned int* n_dev,
                                       unsigned long long* counts) {
    const uint32_t n = n_dev ? *n_dev : n_fixed;
    unsigned int c0 = 0, c1 = 0, c2 = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t len = word_end[i] - word_start[i];
        c0 += (len > BB_WARP_MAX && len <= BB_SMALL_MAX); c1 += (len > BB_SMALL_MAX); c2 += (len > BB_BIG_CAP);
    }
    for (int d = 16; d > 0; d >>= 1) { c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, d); c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, d); c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, d); }
    if ((threadIdx.x & 31) == 0) { if (c0) atomicAdd(counts, (unsigned long long)c0); if (c1) atomicAdd(counts + 1, (unsigned long long)c1); if (c2) atomicAdd(counts + 2, (unsigned long long)c2); }
}
__global__ void gather_scalars_kernel(unsigned long long* ctrl, const uint32_t* word_tok_off, uint32_t n_words,
                                      const unsigned long long* doc_tok_off, uint32_t n_docs, const uint32_t* word_doc) {
    ctrl[2] = word_tok_off[n_words];
    ctrl[3] = doc_tok_off[n_docs];
    const unsigned long long ew = ctrl[0];
    ctrl[4] = (ew != TKZ_ERRW_NONE && n_words) ? word_doc[(uint32_t)(ew >> 8)] : 0;
}

// pass A's shared memory (above the 48 KB default) for every class mode and record kind of a model
template <int MODEL, int REC>
void slice_words_smem_rec() {
    const int sm = (int)sizeof(BlockShared);
    cudaFuncSetAttribute(slice_words_kernel<MODEL, 0, REC>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm);
    cudaFuncSetAttribute(slice_words_kernel<MODEL, 1, REC>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm);
    cudaFuncSetAttribute(slice_words_kernel<MODEL, 2, REC>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm);
    cudaFuncSetAttribute(slice_words_kernel<MODEL, 3, REC>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm);
}
template <int MODEL>
void slice_words_smem() {
    slice_words_smem_rec<MODEL, TW_REC_ID32>();
    slice_words_smem_rec<MODEL, TW_REC_WIDE>();
    slice_words_smem_rec<MODEL, TW_REC_ID16>();
    slice_words_smem_rec<MODEL, TW_REC4>();
    slice_words_smem_rec<MODEL, TW_REC_WORD>();
}

}  // namespace

// ------------------------------------------------------------------------------------------------ context
extern "C" int tkz_ctx_create(int device, void* stream, uint64_t arena_hint_bytes, tkz_ctx** out) {
    if (!out) return TKZ_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                         " (tokzig_b200 has no CPU fallback)";
        return TKZ_ERR_CUDA;
    }
    if (device < 0 || device >= n) { g_create_error = "invalid device ordinal"; return TKZ_ERR_INVALID_ARG; }
    DeviceGuard guard__(device);
    if (!guard__.ok) { g_create_error = "cudaSetDevice failed"; return TKZ_ERR_CUDA; }
    tkz_ctx* ctx = new tkz_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
    else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { g_create_error = std::string("cudaStreamCreate: ") + cudaGetErrorString(e); delete ctx; return TKZ_ERR_CUDA; }
        ctx->own_stream = true;
    }
    cudaFuncSetAttribute(bpe_block_kernel<1024, 12288>, cudaFuncAttributeMaxDynamicSharedMemorySize, 12288 * 15);
    cudaFuncSetAttribute(bpe_block_kernel<512, 4096, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4096 * 15);
    slice_words_smem<TKZ_MODEL_BPE>();
    slice_words_smem<TKZ_MODEL_WORDPIECE>();
    e = cudaFuncSetAttribute(bpe_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BPE_SMEM_BYTES);
    if (e != cudaSuccess) {
        g_create_error = std::string("kernel image not usable on this device (built for sm_100a): ") + cudaGetErrorString(e);
        if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
        delete ctx; return TKZ_ERR_CUDA;
    }
    if (ensure(ctx, ctx->a_ctrl, 64 * sizeof(unsigned long long)) != TKZ_OK ||
        cudaHostAlloc(&ctx->h_ctrl.p, 64 * sizeof(unsigned long long), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&ctx->h_ctrl_dev, ctx->h_ctrl.p, 0) != cudaSuccess) {
        g_create_error = ctx->err.empty() ? "cudaHostAlloc (mapped control block) failed" : ctx->err;
        if (ctx->own_stream) cudaStreamDestroy(ctx->stream); delete ctx; return TKZ_ERR_OOM;
    }
    ctx->h_ctrl.cap = 64 * sizeof(unsigned long long);
    (void)arena_hint_bytes;
    if (const char* e = getenv("TKZ_NO_DEDUP")) ctx->use_dedup = !(e[0] == '1');     // A/B switch for the parity tests
    if (const char* e = getenv("TKZ_CLASSIFY")) ctx->force_lut = (e[0] == 'l');
    if (const char* e = getenv("TKZ_TOK_RECORD")) ctx->narrow_records = !(e[0] == 'w');
    if (const char* e = getenv("TKZ_NO_GRID")) ctx->use_grid = !(e[0] == '1');
    if (const char* e = getenv("TKZ_GRID_MIN_LEN")) { const long long v = atoll(e); if (v > (long long)BB_WARP_MAX) ctx->grid_min_len = (uint32_t)v; }
    {
        int coop = 0, per_sm = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
        if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bpe_grid_kernel, BG_NT, 0) == cudaSuccess && per_sm > 0)
            ctx->grid_blocks = ctx->sm_count * per_sm;
    }
    if (const char* e = getenv("TKZ_CHUNK_BYTES")) { const long long v = atoll(e); if (v > 0) ctx->chunk_bytes = (uint64_t)v; }
    cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking);
    for (int i = 0; i < 2; i++) { cudaEventCreateWithFlags(&ctx->ev_h2d[i], cudaEventDisableTiming); cudaEventCreateWithFlags(&ctx->ev_d2h[i], cudaEventDisableTiming); }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    {
        unsigned long long pw[TW_MAX_MED]; pw[0] = 1;
        for (int i = 1; i < (int)TW_MAX_MED; i++) pw[i] = pw[i - 1] * TKZ_MED_HASH_MUL;
        cudaMemcpyToSymbol(c_med_pw, pw, sizeof pw);
    }
    *out = ctx;
    return TKZ_OK;
}

extern "C" void tkz_ctx_destroy(tkz_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard guard__(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf* bufs[] = {&ctx->t_lut, &ctx->t_lut_post, &ctx->t_char_ascii, &ctx->t_char_tab, &ctx->t_merges, &ctx->t_merge_win, &ctx->t_wp_tab, &ctx->t_wp_pool,
                      &ctx->a_text, &ctx->a_doc_off, &ctx->a_norm_text, &ctx->a_norm_doc_off, &ctx->a_chunk, &ctx->a_tiles, &ctx->a_word_start,
                      &ctx->a_word_end, &ctx->a_word_doc, &ctx->a_doc_word_off, &ctx->a_word_ntok, &ctx->a_pool_id, &ctx->a_pool_s, &ctx->a_pool_e,
                      &ctx->a_pool_rk, &ctx->a_scan_tmp, &ctx->in_text[0], &ctx->in_text[1], &ctx->in_doc_off[0],
                      &ctx->in_doc_off[1], &ctx->a_ctrl, &ctx->a_long_start, &ctx->a_long_end, &ctx->a_long_ntok, &ctx->a_long_slice, &ctx->a_long_ins,
                      &ctx->a_tile_ntok, &ctx->a_tile_ntok_inline, &ctx->a_tile_tok_off, &ctx->a_tile_long, &ctx->a_doc_tok_local,
                      &ctx->a_doc_tok_start, &ctx->a_doc_real, &ctx->a_upool, &ctx->a_tile_doc_lo, &ctx->a_g_first, &ctx->a_g_win, &ctx->a_g_flag, &ctx->a_big,
                      &ctx->a_slice_nword, &ctx->a_doc_word_local, &ctx->a_doc_word_base, &ctx->a_long_k, &ctx->a_row_real, &ctx->a_row_doc,
                      &ctx->a_wtable, &ctx->a_lscratch, &ctx->a_tok_id, &ctx->a_fast_heap, &ctx->a_word_aux,
                      &ctx->a_huge_w, &ctx->a_huge_base, &ctx->a_huge_done, &ctx->a_grid_state, &ctx->a_grid_words,
                      &ctx->t_dec_bytes, &ctx->t_dec_off, &ctx->t_dec_special, &ctx->a_dec_ids, &ctx->a_dec_seq_off, &ctx->a_dec_len, &ctx->a_dec_raw,
                      &ctx->a_dec_out, &ctx->a_dec_olen, &ctx->a_dec_boff};
    for (auto& os : ctx->outs) for (DevBuf* b : {&os.doc_tok_off, &os.ids, &os.off, &os.attn, &os.type, &os.special, &os.off16, &os.ids16, &os.spans, &os.wide, &os.wid, &os.row_tok_off, &os.doc_row_off}) release(*b);
    for (DevBuf* b : bufs) release(*b);
    HostBuf* hb[] = {&ctx->h_ctrl, &ctx->h_doc_tok_off, &ctx->h_ids, &ctx->h_off, &ctx->h_attn, &ctx->h_type, &ctx->h_special, &ctx->h_off16, &ctx->h_ids16, &ctx->h_spans, &ctx->h_wide, &ctx->h_wid,
                     &ctx->h_row_tok_off, &ctx->h_doc_row_off, &ctx->h_doc_stage[0], &ctx->h_doc_stage[1], &ctx->h_dec_bytes, &ctx->h_dec_off};
    for (HostBuf* b : hb) release_host(*b);
    if (ctx->s_h2d) cudaStreamDestroy(ctx->s_h2d);
    if (ctx->s_d2h) cudaStreamDestroy(ctx->s_d2h);
    for (int i = 0; i < 2; i++) { if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]); if (ctx->ev_d2h[i]) cudaEventDestroy(ctx->ev_d2h[i]); }
    for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* tkz_last_error(tkz_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int tkz_ctx_numa_node(tkz_ctx* ctx) {
    if (!ctx) return -1;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, ctx->device) != cudaSuccess) return -1;
    for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c - 'A' + 'a');
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

extern "C" int tkz_ctx_get_stats(tkz_ctx* ctx, tkz_stats* out) {
    if (!ctx || !out) return TKZ_ERR_INVALID_ARG;
    *out = ctx->stats; out->arena_bytes = ctx->arena_bytes;
    out->model_flags = ((ctx->has_model && ctx->dm.windowed_ok) ? 1u : 0u) | (ctx->grid_used ? 2u : 0u) | (ctx->retried ? 4u : 0u);
    return TKZ_OK;
}

// ------------------------------------------------------------------------------------------------ model upload
extern "C" int tkz_model_upload(tkz_ctx* ctx, const tkz_model_desc* d) {
    if (!ctx || !d) return TKZ_ERR_INVALID_ARG;
    ON_DEVICE(ctx);
    if (d->model_kind != TKZ_MODEL_BPE && d->model_kind != TKZ_MODEL_WORDPIECE) { ctx->err = "unknown model_kind"; return TKZ_ERR_INVALID_ARG; }
    if (d->vocab_n && (!d->vocab_bytes || !d->vocab_off || !d->vocab_ids)) { ctx->err = "vocab arrays missing"; return TKZ_ERR_INVALID_ARG; }
    DevModel m{};
    m.kind = d->model_kind;
    m.has_pretok = d->class_lut != nullptr;
    // ---- byte pipeline LUTs: [0,256) normalised byte, [256,512) class of the raw byte, [512,768) dropped flag
    std::vector<uint8_t> lut(768, 0), lut_post(768, 0);
    bool identity = true, has_drop = false;
    for (int b = 0; b < 256; b++) {
        uint16_t nb = d->norm_lut ? d->norm_lut[b] : (uint16_t)b;
        const bool drop = nb == TKZ_NORM_DROP;
        if (!drop && nb > 0xFF) { ctx->err = "norm_lut entry out of range"; return TKZ_ERR_INVALID_ARG; }
        if (drop) { has_drop = true; nb = 0; }
        if (nb != b || drop) identity = false;
        lut[b] = (uint8_t)nb;
        lut[512 + b] = drop ? 1 : 0;
        uint8_t c = d->class_lut ? d->class_lut[nb] : (uint8_t)TKZ_CLS_WORD;
        if (c > 2) { ctx->err = "class_lut entry out of range"; return TKZ_ERR_INVALID_ARG; }
        lut[256 + b] = drop ? (uint8_t)TKZ_CLS_DELIM : c;
        lut_post[b] = (uint8_t)b;
        lut_post[256 + b] = d->class_lut ? d->class_lut[b] : (uint8_t)TKZ_CLS_WORD;
    }
    m.norm_identity = identity; m.norm_has_drop = has_drop;
    // byte classes as ranges (tkz_slices.cuh, four bytes per instruction) when the tables allow it: the byte map is the
    // identity or exactly A-Z -> a-z, bytes >= 0x80 are WORD, and DELIM / ISOLATE are a few runs of byte values each
    auto make_ranges = [](const uint8_t* nrm, const uint8_t* cls, bool drops) -> ClassRanges {
        ClassRanges r{};
        if (drops) return r;
        bool ident = true, lower = true;
        for (int b = 0; b < 256; b++) {
            if (nrm[b] != b) ident = false;
            if (nrm[b] != ((b >= 'A' && b <= 'Z') ? b + 32 : b)) lower = false;
        }
        if (!ident && !lower) return r;
        for (int b = 128; b < 256; b++) if (cls[b] != TKZ_CLS_WORD) return r;
        for (int c = TKZ_CLS_DELIM; c <= TKZ_CLS_ISOLATE; c++) {
            int n = 0;
            for (int b = 0; b < 128;) {
                if (cls[b] != c) { b++; continue; }
                int e = b; while (e + 1 < 128 && cls[e + 1] == c) e++;
                if (n == TW_MAX_RANGES) return r;
                const uint32_t lo = (uint32_t)(0x80 - b) * 0x01010101u, hi = (uint32_t)(0x7F - e) * 0x01010101u;
                if (c == TKZ_CLS_DELIM) { r.d_lo[n] = lo; r.d_hi[n] = hi; } else { r.i_lo[n] = lo; r.i_hi[n] = hi; }
                n++; b = e + 1;
            }
            if (c == TKZ_CLS_DELIM) r.n_delim = n; else r.n_iso = n;
        }
        r.norm_lower = (lower && !ident) ? 1 : 0;
        r.usable = tw_ranges_supported(r.n_delim, r.n_iso) ? 1 : 0;
        return r;
    };
    ctx->has_iso = false;
    for (int b = 0; b < 256; b++) if (lut[256 + b] == TKZ_CLS_ISOLATE || lut_post[256 + b] == TKZ_CLS_ISOLATE) ctx->has_iso = true;
    ctx->cr = make_ranges(lut.data(), lut.data() + 256, has_drop);
    ctx->cr_post = make_ranges(lut_post.data(), lut_post.data() + 256, false);
    TRY(upload(ctx, ctx->t_lut, lut.data(), lut.size()));
    TRY(upload(ctx, ctx->t_lut_post, lut_post.data(), lut_post.size()));
    m.lut = (const uint8_t*)ctx->t_lut.p;
    m.has_unk = d->has_unk; m.unk_id = d->unk_id;

    if (d->model_kind == TKZ_MODEL_BPE) {
        // single-codepoint keys (bpe.zig:192: only the bytes of one UTF-8 sequence are ever looked up)
        std::vector<uint32_t> ascii(128, TKZ_NONE);
        std::vector<std::pair<uint32_t, uint32_t>> multi;
        for (uint32_t i = 0; i < d->vocab_n; i++) {
            const uint64_t a = d->vocab_off[i], len = d->vocab_off[i + 1] - a;
            if (len < 1 || len > 4) continue;
            const uint8_t* k = d->vocab_bytes + a;
            if ((uint64_t)utf8_seq_len(k[0]) != len) continue;
            if (len == 1) ascii[k[0]] = d->vocab_ids[i];
            else { uint32_t key = 0; for (uint64_t j = 0; j < len; j++) key |= (uint32_t)k[j] << (8 * j); multi.push_back({key, d->vocab_ids[i]}); }
        }
        const uint32_t ccap = pow2_at_least(multi.size() * 2 + 2);
        std::vector<CharEnt> ctab(ccap, CharEnt{0, 0});
        for (auto& kv : multi) {
            uint32_t s = char_hash32(kv.first) & (ccap - 1);
            while (ctab[s].key != 0 && ctab[s].key != kv.first) s = (s + 1) & (ccap - 1);
            ctab[s].key = kv.first; ctab[s].id = kv.second;            // put: later entry overwrites
        }
        TRY(upload(ctx, ctx->t_char_ascii, ascii.data(), ascii.size() * 4));
        TRY(upload(ctx, ctx->t_char_tab, ctab.data(), ctab.size() * sizeof(CharEnt)));
        m.char_ascii = (const uint32_t*)ctx->t_char_ascii.p; m.char_tab = (const CharEnt*)ctx->t_char_tab.p; m.char_mask = ccap - 1;
        // merges (bpe.zig:40): put semantics, later entry for the same pair overwrites (config.zig:269)
        if (d->merges_n && (!d->merge_first || !d->merge_second || !d->merge_rank || !d->merge_new)) { ctx->err = "merge arrays missing"; return TKZ_ERR_INVALID_ARG; }
        const uint32_t mcap = pow2_at_least((uint64_t)d->merges_n * 2 + 2);
        std::vector<MergeEnt> mtab(mcap, MergeEnt{0, 0, TKZ_NONE, 0});
        uint32_t live = 0;
        for (uint32_t i = 0; i < d->merges_n; i++) {
            const uint32_t a = d->merge_first[i], b = d->merge_second[i], r = d->merge_rank[i];
            if (r == TKZ_DIRTY) { ctx->err = "merge rank 0xFFFFFFFE is reserved"; return TKZ_ERR_INVALID_ARG; }
            uint32_t s = pair_hash32(a, b) & (mcap - 1);
            while (mtab[s].rank != TKZ_NONE && !(mtab[s].first == a && mtab[s].second == b)) s = (s + 1) & (mcap - 1);
            if (mtab[s].rank == TKZ_NONE) {
                if (r == TKZ_NONE) continue;      // rank maxInt(u32) can never win the strict `<` of bpe.zig:225: same as absent
                live++;
            } else if (r == TKZ_NONE) {
                // overwritten by an unselectable rank: keep the slot occupied (probe chains) but make it never match a rank
                // by storing the reserved value; handled as "no rank" by giving it the largest selectable rank is NOT exact,
                // so re-build without the pair instead.
                ctx->err = "merge rank 0xFFFFFFFF overwriting an earlier rank is not supported"; return TKZ_ERR_INVALID_ARG;
            }
            mtab[s] = MergeEnt{a, b, r, d->merge_new[i]};
        }
        TRY(upload(ctx, ctx->t_merges, mtab.data(), mtab.size() * sizeof(MergeEnt)));
        m.merges = (const MergeEnt*)ctx->t_merges.p; m.merge_mask = mcap - 1; m.n_merges = live;
        // ---- is the table "proper"?  (every producer of a symbol has a lower rank than every merge that consumes it, ranks
        // are unique).  Then the round order of bpe.zig:214-253 equals strict rank order and merges can be scheduled by
        // windowed local minima (tkz_bpe_block.cuh); otherwise long words keep the literal round kernel.
        {
            std::vector<uint32_t> order;                       // live slots sorted by rank
            for (uint32_t sl = 0; sl < mcap; sl++) if (mtab[sl].rank != TKZ_NONE) order.push_back(sl);
            std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return mtab[x].rank < mtab[y].rank; });
            bool proper = true;
            for (size_t i = 1; i < order.size() && proper; i++) if (mtab[order[i]].rank == mtab[order[i - 1]].rank) proper = false;
            // (ranks / ids in the reserved range of TKZ_BOUNDARY, TKZ_DIRTY, BG_PENDING keep the literal kernel)
            for (uint32_t sl : order) if (mtab[sl].rank >= TKZ_BOUNDARY || mtab[sl].new_id >= BG_PENDING) proper = false;
            std::unordered_map<uint32_t, uint32_t> max_prod, min_cons, nsym;    // per symbol id
            for (uint32_t sl : order) {
                const MergeEnt& e = mtab[sl];
                auto it = max_prod.find(e.new_id);
                if (it == max_prod.end() || it->second < e.rank) max_prod[e.new_id] = e.rank;
                for (uint32_t x : {e.first, e.second}) { auto c = min_cons.find(x); if (c == min_cons.end() || c->second > e.rank) min_cons[x] = e.rank; }
            }
            for (auto& kv : max_prod) { auto c = min_cons.find(kv.first); if (c != min_cons.end() && c->second <= kv.second) { proper = false; break; } }
            std::vector<uint16_t> win(mcap, 0);
            if (proper) {
                auto ns = [&](uint32_t id) -> uint32_t { auto it = nsym.find(id); return it == nsym.end() ? 1u : it->second; };
                for (uint32_t sl : order) {                    // rank order: operands are final before they are consumed
                    const MergeEnt& e = mtab[sl];
                    const uint32_t v = ns(e.first) + ns(e.second);
                    auto it = nsym.find(e.new_id);
                    if (it == nsym.end() || it->second < v) nsym[e.new_id] = v;
                }
                // Threats to an occurrence (a, b) of rank r: merges that consume a from the left or b from the right BEFORE round
                // r, i.e. entries (X, a) / (b, Z) with a rank below r (X, Z are then built by merges of even lower rank).  Window
                // of the entry: wl = max nsym(X) over (X, a) with rank < r, wr = max nsym(Z) over (b, Z) with rank < r.  Early
                // merges involve short symbols, so the pairs that merge in the first, populous steps get windows of 1-3 symbols
                // (a rank-blind window would be as wide as the longest token that ever joins the symbol).
                std::unordered_map<uint32_t, uint32_t> WL, WR;  // running max while the entries are visited in rank order
                for (uint32_t sl : order) {                    // ascending rank: WL / WR hold exactly the entries of lower rank
                    const MergeEnt& e = mtab[sl];
                    auto get = [](std::unordered_map<uint32_t, uint32_t>& mp, uint32_t k) { auto it = mp.find(k); return it == mp.end() ? 0u : it->second; };
                    uint32_t wl = get(WL, e.first), wr = get(WR, e.second);     // threats to `first` from its left, to `second` from its right
                    // (A, A): the window is laid around the whole RUN of A and must also see an A that could still appear next
                    // to the run (it would change which A pairs with which): such an A is built from at most nsym(A) symbols
                    if (e.first == e.second) { wl = std::max(wl, ns(e.first)); wr = std::max(wr, ns(e.first)); }
                    if (wl > 250 || wr > 250) { proper = false; break; }
                    win[sl] = (uint16_t)(wl | (wr << 8));
                    uint32_t& l = WL[e.second]; l = std::max(l, ns(e.first)); uint32_t& r = WR[e.first]; r = std::max(r, ns(e.second));
                }
                if (getenv("TKZ_GRID_DEBUG") && !order.empty()) {
                    double sl_ = 0, sr_ = 0; uint32_t ml = 0, mr = 0;
                    for (uint32_t sl : order) { sl_ += win[sl] & 0xFF; sr_ += win[sl] >> 8; ml = std::max<uint32_t>(ml, win[sl] & 0xFF); mr = std::max<uint32_t>(mr, win[sl] >> 8); }
                    fprintf(stderr, "[tkz upload] %zu merges, windows: mean left %.2f right %.2f, max left %u right %u\n", order.size(), sl_ / order.size(), sr_ / order.size(), ml, mr);
                }
            }
            TRY(upload(ctx, ctx->t_merge_win, win.data(), win.size() * 2));
            m.merge_win = (const uint16_t*)ctx->t_merge_win.p;
            m.windowed_ok = proper ? 1 : 0;
            if (const char* e = getenv("TKZ_NO_WINDOWED")) if (e[0] == '1') m.windowed_ok = 0;
        }
    } else {
        if (d->prefix_len > TKZ_MAX_PREFIX) { ctx->err = "continuing_subword_prefix longer than 64 bytes"; return TKZ_ERR_INVALID_ARG; }
        m.prefix_len = d->prefix_len;
        uint64_t st = TKZ_FNV_OFFSET;
        for (uint32_t i = 0; i < d->prefix_len; i++) { m.prefix[i] = d->prefix[i]; st = fnv1a_step(st, d->prefix[i]); }
        m.prefix_state = st;
        m.max_chars = d->max_input_chars_per_word;
        const uint32_t wcap = pow2_at_least((uint64_t)d->vocab_n * 2 + 2);
        std::vector<WpEnt> wtab(wcap, WpEnt{0, 0, 0, 0, 0});
        uint32_t max_first = 0, max_cont = 0;
        const uint64_t pool_bytes = d->vocab_n ? d->vocab_off[d->vocab_n] : 0;
        if (pool_bytes >= 0xFFFFFFFFull) { ctx->err = "vocabulary larger than 4 GiB"; return TKZ_ERR_INVALID_ARG; }
        for (uint32_t i = 0; i < d->vocab_n; i++) {
            const uint64_t a = d->vocab_off[i], len = d->vocab_off[i + 1] - a;
            const uint8_t* k = d->vocab_bytes + a;
            uint64_t h = TKZ_FNV_OFFSET;
            for (uint64_t j = 0; j < len; j++) h = fnv1a_step(h, k[j]);
            uint32_t s = wp_slot(h) & (wcap - 1);
            while (wtab[s].used && !(wtab[s].hash == h && wtab[s].len == len && memcmp(d->vocab_bytes + wtab[s].str_off, k, len) == 0)) s = (s + 1) & (wcap - 1);
            wtab[s] = WpEnt{h, d->vocab_ids[i], (uint32_t)a, (uint32_t)len, 1u};       // put: later entry overwrites
            if (len > max_first) max_first = (uint32_t)len;
            if (len >= d->prefix_len && (d->prefix_len == 0 || memcmp(k, d->prefix, d->prefix_len) == 0)) {
                const uint32_t c = (uint32_t)(len - d->prefix_len);
                if (c > max_cont) max_cont = c;
            }
        }
        TRY(upload(ctx, ctx->t_wp_tab, wtab.data(), wtab.size() * sizeof(WpEnt)));
        TRY(upload(ctx, ctx->t_wp_pool, d->vocab_bytes, (size_t)pool_bytes));
        m.wp_tab = (const WpEnt*)ctx->t_wp_tab.p; m.wp_mask = wcap - 1; m.wp_pool = (const uint8_t*)ctx->t_wp_pool.p;
        m.max_key_first = max_first; m.max_key_cont = max_cont;
    }
    {
        uint32_t max_id = d->has_unk ? d->unk_id : 0u;
        for (uint32_t i = 0; i < d->vocab_n; i++) max_id = std::max(max_id, d->vocab_ids[i]);
        if (d->model_kind == TKZ_MODEL_BPE) for (uint32_t i = 0; i < d->merges_n; i++) max_id = std::max(max_id, d->merge_new[i]);
        ctx->ids16_ok = max_id < 65536u;
        ctx->max_id = max_id;
    }
    CK(cudaStreamSynchronize(ctx->stream));      // host staging vectors die at return
    ctx->dm = m;
    ctx->dm_post = m;
    ctx->dm_post.lut = (const uint8_t*)ctx->t_lut_post.p;
    ctx->dm_post.norm_identity = 1; ctx->dm_post.norm_has_drop = 0;
    ctx->has_model = true;
    return TKZ_OK;
}

// ------------------------------------------------------------------------------------------------ encode
namespace {

// BPE over a word list: warp kernel (literal rounds) for short words or improper tables, block kernels with the windowed
// schedule for long words of proper tables.  cls = {#65..2048, #>2048, #>12288} from len_class_count_kernel.
int launch_bpe(tkz_ctx* ctx, const DevModel& m, const uint8_t* d_text, const uint32_t* word_start, const uint32_t* word_end, uint32_t nw,
               uint32_t* word_ntok, unsigned long long* ctrl, int ctr_slot, int sentinel, const unsigned long long* cls, uint64_t N,
               uint64_t& launches) {
    cudaStream_t st = ctx->stream;
    const bool windowed = m.windowed_ok && (cls[0] || cls[1]);
    TRY(ensure(ctx, ctx->a_pool_rk, N * 4));
    BpeArgs a{d_text, word_start, word_end, nw, (uint32_t*)ctx->a_pool_id.p, (uint32_t*)ctx->a_pool_s.p, (uint32_t*)ctx->a_pool_e.p,
              (uint32_t*)ctx->a_pool_rk.p, word_ntok, (unsigned int*)(ctrl + ctr_slot), ctrl, sentinel, windowed ? BB_WARP_MAX : 0xFFFFFFFFu};
    uint64_t blocks = ((uint64_t)nw + BPE_WARPS - 1) / BPE_WARPS;
    const uint64_t cap = (uint64_t)ctx->sm_count * 3; if (blocks > cap) blocks = cap;
    bpe_warp_kernel<<<(unsigned)blocks, BPE_WARPS * 32, BPE_SMEM_BYTES, st>>>(m, a); launches++;
    if (!windowed) return TKZ_OK;
    if (cls[2]) { TRY(ensure(ctx, ctx->a_g_first, N * 4)); TRY(ensure(ctx, ctx->a_g_win, N * 2)); TRY(ensure(ctx, ctx->a_g_flag, N)); }
    BlockBpeArgs b{};
    b.text = d_text; b.word_start = word_start; b.word_end = word_end; b.n_words = nw;
    b.pool_id = (uint32_t*)ctx->a_pool_id.p; b.pool_s = (uint32_t*)ctx->a_pool_s.p; b.pool_e = (uint32_t*)ctx->a_pool_e.p; b.pool_rk = (uint32_t*)ctx->a_pool_rk.p;
    b.g_first = (uint32_t*)ctx->a_g_first.p; b.g_win = (uint16_t*)ctx->a_g_win.p; b.g_flag = (uint8_t*)ctx->a_g_flag.p;
    b.word_ntok = word_ntok; b.errw = ctrl; b.sentinel_errors = sentinel;
    const uint32_t grid_min = ctx->grid_min_len;
    if ((grid_min > BB_BIG_CAP ? cls[2] != 0 : (cls[0] || cls[1])) && ctx->use_grid && ctx->grid_blocks > 0) {
        // words above the shared-memory capacity: all of them together on one cooperative grid (tkz_bpe_grid.cuh); a word
        // it leaves alone (malformed UTF-8) and everything when its state does not fit falls through to the block kernel
        const uint32_t hcap = grid_min == BB_BIG_CAP + 1 ? (uint32_t)cls[2] : nw;
        unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
        TRY(ensure(ctx, ctx->a_huge_w, ((size_t)hcap + 2) * 4));
        TRY(ensure(ctx, ctx->a_huge_base, ((size_t)hcap + 2) * 4));
        TRY(ensure(ctx, ctx->a_huge_done, (size_t)nw + 16));
        CK(cudaMemsetAsync(ctx->a_huge_done.p, 0, (size_t)nw, st));
        huge_list_kernel<<<1, 1024, 0, st>>>(word_start, word_end, nw, grid_min, hcap, (uint32_t*)ctx->a_huge_w.p, (uint32_t*)ctx->a_huge_base.p, ctrl + 18);
        launches++;
        TRY(readback(ctx, hctrl + 40, ctrl + 18, 16));
        CK(cudaStreamSynchronize(st));
        const uint64_t n_huge = hctrl[40], M = hctrl[41];
        auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t per4 = al((size_t)M * 4 + 16), per2 = al((size_t)M * 2 + 16);
        const size_t state_bytes = 11 * per4 + 2 * per2;                    // (id, s, e, rk, wid) x 2 + hn, win x 2
        const size_t words_bytes = 4 * al(((size_t)n_huge + 2) * 4) + al((size_t)n_huge + 16) + al((size_t)ctx->grid_blocks * 33 * 4 + 64) + 256 + 5120;
        bool ok = n_huge > 0 && n_huge <= hcap && M < 0xFFFFF000ull;
        if (ok && (ensure(ctx, ctx->a_grid_state, state_bytes) != TKZ_OK || ensure(ctx, ctx->a_grid_words, words_bytes) != TKZ_OK)) {
            ok = false; ctx->err.clear(); cudaGetLastError();                // no room for the grid state: one block per word
        }
        if (ok) {
            GridBpeArgs ga{};
            ga.text = d_text; ga.word_start = word_start; ga.word_end = word_end;
            ga.sparse_walk = BG_SPARSE_WALK;
            if (const char* e = getenv("TKZ_GRID_SPARSE_WALK")) ga.sparse_walk = (uint32_t)atoll(e);
            ga.hw = (const uint32_t*)ctx->a_huge_w.p; ga.hbase = (const uint32_t*)ctx->a_huge_base.p; ga.n_huge = (uint32_t)n_huge; ga.M = (uint32_t)M;
            uint8_t* p = (uint8_t*)ctx->a_grid_state.p;
            auto take = [&](size_t bytes) { uint8_t* r = p; p += bytes; return r; };
            for (int k = 0; k < 2; k++) {
                ga.id[k] = (uint32_t*)take(per4); ga.s[k] = (uint32_t*)take(per4); ga.e[k] = (uint32_t*)take(per4);
                ga.rk[k] = (uint32_t*)take(per4); ga.wid[k] = (uint32_t*)take(per4); ga.win[k] = (uint16_t*)take(per2);
            }
            ga.hn = (uint32_t*)take(per4);
            p = (uint8_t*)ctx->a_grid_words.p;
            const size_t pw = al(((size_t)n_huge + 2) * 4);
            ga.wmin[0] = (uint32_t*)take(pw); ga.wmin[1] = (uint32_t*)take(pw); ga.wstart = (uint32_t*)take(pw); take(pw);
            ga.wbad = take(al((size_t)n_huge + 16));
            ga.blk = (uint32_t*)take(al((size_t)ctx->grid_blocks * 33 * 4 + 64));
            ga.gs = (uint32_t*)take(256);
            ga.dbg = (uint32_t*)take(5120);
            ga.pool_id = (uint32_t*)ctx->a_pool_id.p; ga.pool_s = (uint32_t*)ctx->a_pool_s.p; ga.pool_e = (uint32_t*)ctx->a_pool_e.p;
            ga.word_ntok = word_ntok; ga.done = (uint8_t*)ctx->a_huge_done.p;
            DevModel mm = m;
            void* args[] = {(void*)&mm, (void*)&ga};
            // (a refused cooperative launch -- e.g. not all blocks can be co-resident on a partitioned device -- is not an
            // error: the block kernel below then takes every word, as with TKZ_NO_GRID=1)
            const cudaError_t le = cudaLaunchCooperativeKernel((void*)bpe_grid_kernel, dim3((unsigned)ctx->grid_blocks), dim3(BG_NT), args, 0, st);
            if (le != cudaSuccess) { cudaGetLastError(); ok = false; }
            else launches++;
            if (ok && getenv("TKZ_GRID_DEBUG")) {
                uint32_t gsh[32];
                cudaStreamSynchronize(st);
                cudaMemcpy(gsh, ga.gs, sizeof gsh, cudaMemcpyDeviceToHost);
                const unsigned long long* g64 = (const unsigned long long*)(gsh + 8);
                fprintf(stderr, "[tkz grid] words %u bytes %u symbols %u dense steps %u run-scans %u sparse steps %u (%u phases)  ms: heads %.2f compact+ranks %.2f sparse %.2f\n", ga.n_huge, ga.M,
                        gsh[7], gsh[5], gsh[6], gsh[20], gsh[21], g64[1] * 1e-6, g64[2] * 1e-6, g64[0] * 1e-6);
                if (getenv("TKZ_GRID_DEBUG")[0] == '2') {
                    uint32_t d[1280];
                    cudaMemcpy(d, ga.dbg, sizeof d, cudaMemcpyDeviceToHost);
                    for (uint32_t k = 0; k < gsh[5] && k < 256; k++)
                        fprintf(stderr, "[tkz grid]   step %3u  n %10u  heads %9u  ranked pairs after %9u  H %7.3f ms  K %7.3f ms\n", k, d[4 * k], d[4 * k + 1], d[1024 + k], d[4 * k + 2] * 1e-6, d[4 * k + 3] * 1e-6);
                }
            }
            if (ok) { b.skip = (const uint8_t*)ctx->a_huge_done.p; ctx->grid_used = true; }
        }
    }
    // One class per shared-memory footprint (15 B per symbol of capacity): an SM holds ~14 k symbols of state whatever the
    // class, so a word in a class far above its length wastes the SM (c2a: 73 % of the words above 2048 bytes are below
    // 4096; 59 % of those up to 1024 are below 512).
    if (cls[0]) {
        // 65..512 bytes: one warp per word, 28 words in flight per SM; ..1024: two warps, 14 words; ..2048: eight warps, 6 words
        b.min_len = BB_WARP_MAX + 1; b.max_len = BB_MINI_MAX; b.work_counter = (unsigned int*)(ctrl + 20);
        uint64_t g = cls[0]; uint64_t gc = (uint64_t)ctx->sm_count * 28; if (g > gc) g = gc;
        bpe_block_kernel<32, BB_MINI_MAX, 28><<<(unsigned)g, 32, BB_MINI_MAX * 15, st>>>(m, b); launches++;
        b.min_len = BB_MINI_MAX + 1; b.max_len = BB_TINY_MAX; b.work_counter = (unsigned int*)(ctrl + 17);
        g = cls[0]; gc = (uint64_t)ctx->sm_count * 14; if (g > gc) g = gc;
        bpe_block_kernel<64, BB_TINY_MAX, 14><<<(unsigned)g, 64, BB_TINY_MAX * 15, st>>>(m, b); launches++;
        b.min_len = BB_TINY_MAX + 1; b.max_len = BB_SMALL_MAX; b.work_counter = (unsigned int*)(ctrl + 11);
        g = cls[0]; gc = (uint64_t)ctx->sm_count * 6; if (g > gc) g = gc;
        bpe_block_kernel<256, BB_SMALL_MAX, 6><<<(unsigned)g, 256, BB_SMALL_MAX * 15, st>>>(m, b); launches++;
    }
    if (cls[1]) {
        // 2049..4096 bytes: sixteen warps, 3 words in flight per SM; longer: 32 warps, one word per SM (global state above 12288)
        b.min_len = BB_SMALL_MAX + 1; b.max_len = BB_MID_MAX; b.work_counter = (unsigned int*)(ctrl + 21);
        uint64_t g = cls[1]; uint64_t gc = (uint64_t)ctx->sm_count * 3; if (g > gc) g = gc;
        bpe_block_kernel<512, BB_MID_MAX, 3><<<(unsigned)g, 512, BB_MID_MAX * 15, st>>>(m, b); launches++;
        b.min_len = BB_MID_MAX + 1; b.max_len = 0xFFFFFFFFu; b.work_counter = (unsigned int*)(ctrl + 12);
        g = cls[1]; gc = (uint64_t)ctx->sm_count; if (g > gc) g = gc;
        bpe_block_kernel<1024, BB_BIG_CAP><<<(unsigned)g, 1024, BB_BIG_CAP * 15, st>>>(m, b); launches++;
    }
    return TKZ_OK;
}

// ---- epilogue of both device pipelines: everything after each document's token count is known

// (hf_compat fields from tkz_encode_params.hf_flags / tpl_*, validated in encode_device_impl)
EmitParams emit_params(const tkz_encode_params& P) {
    EmitParams ep{P.has_truncation, P.max_length, P.has_padding, P.pad_length, P.pad_id, P.pad_type_id, P.pad_left, P.outputs};
    if (P.hf_flags) {
        ep.hf_flags = P.hf_flags; ep.n_pre = P.tpl_n_prefix; ep.n_suf = P.tpl_n_suffix; ep.seq_type = P.tpl_seq_type;
        for (uint32_t i = 0; i < TKZ_TPL_MAX; i++) {
            ep.pre_id[i] = P.tpl_prefix_id[i]; ep.pre_type[i] = P.tpl_prefix_type[i]; ep.suf_id[i] = P.tpl_suffix_id[i]; ep.suf_type[i] = P.tpl_suffix_type[i];
        }
    }
    return ep;
}
bool has_frame(const EmitParams& ep) { return (ep.hf_flags & 1u) && ep.n_pre + ep.n_suf; }   // hf_compat: the template's special tokens

// the output arrays of T slots that ep.outputs asks for, and the wide-offset side list, in the context's current output set
int alloc_outputs(tkz_ctx* ctx, const EmitParams& ep, uint64_t T, uint32_t wide_cap, EmitOut& eo) {
    auto& O = ctx->O();
    const uint32_t o = ep.outputs;
    if (o & TKZ_OUT_IDS_U16) TRY(ensure(ctx, O.ids16, (T + 4) * 2)); else TRY(ensure(ctx, O.ids, (T + 4) * 4));
    if (o & TKZ_OUT_OFFSETS) TRY(ensure(ctx, O.off, (T + 4) * 8));
    if (o & TKZ_OUT_ATTENTION) TRY(ensure(ctx, O.attn, (T + 4) * 4));
    if (o & TKZ_OUT_TYPE_IDS) TRY(ensure(ctx, O.type, (T + 4) * 4));
    if (o & TKZ_OUT_SPECIAL) TRY(ensure(ctx, O.special, (T + 4) * 4));
    if (o & TKZ_OUT_OFFSETS_PACKED) TRY(ensure(ctx, O.off16, (T + 4) * 2));
    if (o & TKZ_OUT_SPAN_TOKENS) TRY(ensure(ctx, O.spans, (T + 4) * 16));
    if (o & TKZ_OUT_WORD_IDS) TRY(ensure(ctx, O.wid, (T + 4) * 4));
    if (wide_cap) TRY(ensure(ctx, O.wide, (size_t)wide_cap * 16));
    eo = EmitOut{(uint32_t*)O.ids.p, (uint32_t*)O.off.p, (uint32_t*)O.attn.p, (uint32_t*)O.type.p, (uint32_t*)O.special.p, (uint16_t*)O.off16.p,
                 (uint16_t*)O.ids16.p, (uint4*)O.spans.p, (uint4*)O.wide.p, (unsigned int*)((unsigned long long*)ctx->a_ctrl.p + 23), wide_cap,
                 (uint32_t*)O.wid.p};
    return TKZ_OK;
}

// before the real tokens are written.  Mostly padding (pad to 512 around a few dozen tokens): every array is filled with its
// padding value at streaming-store speed and the real tokens overwrite it; else pad_epilogue writes each document's gaps.
// Returns whether the arrays were filled.
bool pad_prologue(tkz_ctx* ctx, const EmitParams& ep, const EmitOut& eo, uint32_t nd, uint64_t T, uint64_t T_real, uint64_t& launches) {
    if (!ep.has_pad || !nd || T < 2 * T_real) return false;
    const unsigned fg = (unsigned)ctx->sm_count * 8;
    auto fill = [&](void* p, uint64_t bytes, uint4 v) { fill16_kernel<<<fg, 256, 0, ctx->stream>>>((uint4*)p, bytes, v); launches++; };
    auto rep = [](uint32_t x) { return make_uint4(x, x, x, x); };
    const uint32_t o = ep.outputs;
    if (o & TKZ_OUT_IDS_U16) fill(eo.ids16, T * 2, rep(ep.pad_id | (ep.pad_id << 16))); else fill(eo.ids, T * 4, rep(ep.pad_id));
    if (o & TKZ_OUT_OFFSETS) fill(eo.offsets, T * 8, rep(0u));
    if (o & TKZ_OUT_ATTENTION) fill(eo.attention, T * 4, rep(0u));
    if (o & TKZ_OUT_TYPE_IDS) fill(eo.type_ids, T * 4, rep(ep.pad_type_id));
    if (o & TKZ_OUT_SPECIAL) fill(eo.special, T * 4, rep(1u));
    if (o & TKZ_OUT_OFFSETS_PACKED) fill(eo.offsets16, T * 2, rep(0u));
    if (o & TKZ_OUT_SPAN_TOKENS) fill(eo.spans, T * 16, make_uint4(ep.pad_id, 0u, 0u, 0x0400u));
    if (o & TKZ_OUT_WORD_IDS) fill(eo.word_ids, T * 4, rep(TKZ_NONE));
    return true;
}

// after the real tokens are written: the template's special tokens, and the padding slots unless pad_prologue filled them
// (doc_real: real tokens per document)
void pad_epilogue(tkz_ctx* ctx, const EmitParams& ep, const EmitOut& eo, uint32_t nd, const uint32_t* doc_real, const unsigned long long* doc_tok_off,
                  bool filled, uint64_t& launches) {
    if (!nd) return;
    const bool wid = (ep.outputs & TKZ_OUT_WORD_IDS) != 0;
    if (ep.has_pad && !filled) {
        const unsigned g = (unsigned)(((uint64_t)nd * 32 + 255) / 256);
        if (wid) emit_pad_real_kernel<true><<<g, 256, 0, ctx->stream>>>(ep, eo, nd, doc_real, doc_tok_off);
        else emit_pad_real_kernel<false><<<g, 256, 0, ctx->stream>>>(ep, eo, nd, doc_real, doc_tok_off);
        launches++;
    } else if (has_frame(ep)) {
        if (wid) emit_frame_kernel<true><<<(nd + 255) / 256, 256, 0, ctx->stream>>>(ep, eo, nd, doc_real, doc_tok_off);
        else emit_frame_kernel<false><<<(nd + 255) / 256, 256, 0, ctx->stream>>>(ep, eo, nd, doc_real, doc_tok_off);
        launches++;
    }
}

// the nine per-token arrays of a result in TKZ_OUT_* bit order (ids, offsets, attention, type ids, special, packed offsets,
// ids16, span tokens, word ids), nullptr where not delivered
constexpr uint32_t N_RESULT_ARRAYS = 9;
using ResultArrays = std::array<const void*, N_RESULT_ARRAYS>;
void set_result(tkz_batch_result* out, uint64_t n_docs, uint64_t T, uint64_t T_real, const uint64_t* doc_tok_off, const ResultArrays& a,
                uint64_t n_wide, const void* wide) {
    out->n_docs = n_docs; out->n_tokens = T; out->n_real_tokens = T_real;
    out->doc_tok_off = doc_tok_off;
    out->ids = (const uint32_t*)a[0]; out->offsets = (const uint32_t*)a[1]; out->attention_mask = (const uint32_t*)a[2];
    out->type_ids = (const uint32_t*)a[3]; out->special_tokens_mask = (const uint32_t*)a[4]; out->offsets_packed = (const uint16_t*)a[5];
    out->ids16 = (const uint16_t*)a[6]; out->span_tokens = (const uint32_t*)a[7]; out->word_ids = (const uint32_t*)a[8];
    out->n_wide = n_wide; out->wide_tokens = n_wide ? (const uint32_t*)wide : nullptr;
}

// device-resident result of an encode, its launch count and its stage times (events ev[0..4])
void finish(tkz_ctx* ctx, const EmitParams& ep, const EmitOut& eo, const unsigned long long* doc_tok_off, uint64_t n_docs, uint64_t T, uint64_t T_real,
            uint64_t n_wide, uint64_t launches, tkz_batch_result* out) {
    ctx->stats.kernel_launches = launches;
    cudaEventElapsedTime(&ctx->stats.ms_split, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->stats.ms_model, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->stats.ms_scan, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&ctx->stats.ms_emit, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&ctx->stats.ms_total, ctx->ev[0], ctx->ev[4]);
    const uint32_t o = ep.outputs;
    ResultArrays a = {eo.ids, eo.offsets, eo.attention, eo.type_ids, eo.special, eo.offsets16, eo.ids16, eo.spans, eo.word_ids};
    for (uint32_t i = 0; i < N_RESULT_ARRAYS; i++) if (!(o & (1u << i))) a[i] = nullptr;
    if (o & TKZ_OUT_IDS_U16) a[0] = nullptr;                          // exactly one of ids / ids16
    set_result(out, n_docs, T, T_real, (const uint64_t*)doc_tok_off, a, n_wide, eo.wide);
}

// a failed word: its document to err_doc, the message and the return code of the error word's code
int report_error(tkz_ctx* ctx, unsigned long long errw, uint64_t err_doc, uint64_t launches, tkz_batch_result* out) {
    out->err_doc = (int64_t)err_doc;
    const uint32_t code = (uint32_t)(errw & 0xFF);
    ctx->err = code == TKZ_ECODE_UTF8 ? "invalid UTF-8 in a BPE pre-token (reference behaviour undefined)" : "MissingUnkToken";
    ctx->stats.kernel_launches = launches;
    return code == TKZ_ECODE_UTF8 ? TKZ_ERR_INVALID_UTF8 : TKZ_ERR_MISSING_UNK;
}

// The slice pipeline (tkz_slices.cuh).  Capacities that depend on the text (token stream, record pool, word table) are
// estimated from the batch and from what earlier batches of the context needed; when pass A runs out of one of them the
// call returns TKZ_RETRY_WORST and the caller runs it again with worst-case capacities (tokens <= bytes), never truncated.
#define TKZ_RETRY_WORST 2
template <int MODEL, int REC>
void launch_slice_words_rec(const DevModel& m, const SliceArgs& ta, int cls, uint32_t blocks, cudaStream_t st) {
    const size_t sm = sizeof(BlockShared);
    if (cls == 0) slice_words_kernel<MODEL, 0, REC><<<blocks, TW_THREADS, sm, st>>>(m, ta);
    else if (cls == 1) slice_words_kernel<MODEL, 1, REC><<<blocks, TW_THREADS, sm, st>>>(m, ta);
    else if (cls == 2) slice_words_kernel<MODEL, 2, REC><<<blocks, TW_THREADS, sm, st>>>(m, ta);
    else slice_words_kernel<MODEL, 3, REC><<<blocks, TW_THREADS, sm, st>>>(m, ta);
}
template <int MODEL>
void launch_slice_words(const DevModel& m, const SliceArgs& ta, int cls, int rec, uint32_t blocks, cudaStream_t st) {
    if (rec == TW_REC_ID32) launch_slice_words_rec<MODEL, TW_REC_ID32>(m, ta, cls, blocks, st);
    else if (rec == TW_REC_WORD) launch_slice_words_rec<MODEL, TW_REC_WORD>(m, ta, cls, blocks, st);
    else if (rec == TW_REC_WIDE) launch_slice_words_rec<MODEL, TW_REC_WIDE>(m, ta, cls, blocks, st);
    else if (rec == TW_REC_ID16) launch_slice_words_rec<MODEL, TW_REC_ID16>(m, ta, cls, blocks, st);
    else launch_slice_words_rec<MODEL, TW_REC4>(m, ta, cls, blocks, st);
}
// the output forms with offsets read TW_REC_WIDE or TW_REC4 records, the ids-only forms TW_REC_ID32 or TW_REC_ID16; calls
// with word ids TW_REC_WORD records, always per document (never PLAIN) and through the generic form
template <bool PLAIN>
void launch_slice_emit(const SliceEmitArgs& ea, const EmitParams& ep, const EmitOut& eo, int rec, uint32_t blocks, cudaStream_t st) {
    const uint32_t o = ep.outputs;
    const bool narrow = rec == TW_REC4 || rec == TW_REC_ID16;
#define TKZ_SLICE_EMIT(OUTS, REC) slice_emit_kernel<PLAIN, OUTS, REC><<<blocks, TW_THREADS, 0, st>>>(ea, ep, eo)
    if (rec == TW_REC_WORD) { if (!PLAIN) slice_emit_kernel<false, 0u, TW_REC_WORD><<<blocks, TW_THREADS, 0, st>>>(ea, ep, eo); }
    else if (o == TKZ_OUT_IDS) { if (narrow) TKZ_SLICE_EMIT(1u, TW_REC_ID16); else TKZ_SLICE_EMIT(1u, TW_REC_ID32); }
    else if (o == (TKZ_OUT_IDS | TKZ_OUT_OFFSETS | TKZ_OUT_ATTENTION)) { if (narrow) TKZ_SLICE_EMIT(7u, TW_REC4); else TKZ_SLICE_EMIT(7u, TW_REC_WIDE); }
    else if (o == (TKZ_OUT_IDS | TKZ_OUT_OFFSETS_PACKED)) { if (narrow) TKZ_SLICE_EMIT(33u, TW_REC4); else TKZ_SLICE_EMIT(33u, TW_REC_WIDE); }
    else if (o == (TKZ_OUT_IDS | TKZ_OUT_IDS_U16 | TKZ_OUT_OFFSETS_PACKED)) { if (narrow) TKZ_SLICE_EMIT(97u, TW_REC4); else TKZ_SLICE_EMIT(97u, TW_REC_WIDE); }
    else if (o == (TKZ_OUT_IDS | TKZ_OUT_IDS_U16)) { if (narrow) TKZ_SLICE_EMIT(65u, TW_REC_ID16); else TKZ_SLICE_EMIT(65u, TW_REC_ID32); }
    else if (rec == TW_REC_ID32) TKZ_SLICE_EMIT(0u, TW_REC_ID32);
    else if (rec == TW_REC_WIDE) TKZ_SLICE_EMIT(0u, TW_REC_WIDE);
    else if (rec == TW_REC_ID16) TKZ_SLICE_EMIT(0u, TW_REC_ID16);
    else TKZ_SLICE_EMIT(0u, TW_REC4);
#undef TKZ_SLICE_EMIT
}

int encode_slices(tkz_ctx* ctx, const DevModel& m, const ClassRanges& cr, const uint8_t* d_text, const uint64_t* d_doc_off, uint32_t nd, uint64_t N,
                  tkz_encode_params P, bool worst, tkz_batch_result* out, uint64_t& launches) {
    cudaStream_t st = ctx->stream;
    unsigned long long* ctrl = (unsigned long long*)ctx->a_ctrl.p;
    unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
    const uint64_t n_docs = nd;
    const uint32_t n_slices = (uint32_t)(N / TW_SLICE + 1);
    const bool want_wid = (P.outputs & TKZ_OUT_WORD_IDS) != 0;
    // (hf_compat and word ids: per-document destinations and offsets / word bases)
    const bool plain = !P.has_truncation && !P.has_padding && !P.hf_flags && !want_wid;
    // ---- capacities: from the text size and from what earlier batches of this context needed
    const bool keep = ctx->call_keep && ctx->kept_valid && !worst;           // reuse the table + pool of this call's previous chunk
    const uint64_t Nsz = ctx->call_keep ? std::max<uint64_t>(N, ctx->call_bytes) : N;
    uint64_t want = Nsz / 32; if (want < (1u << 16)) want = 1u << 16; if (want > (1u << 22)) want = 1u << 22;
    if (want < ctx->tw_uniq_hist * 4) want = ctx->tw_uniq_hist * 4;          // load factor <= 1/4
    if (want > (1u << 26)) want = 1u << 26;
    const uint32_t tcap = keep ? ctx->kept_tcap : pow2_at_least(want);
    uint32_t tbits = 0; while ((1u << tbits) < tcap) tbits++;
    const uint32_t mcap = tcap >= (1u << 17) ? tcap / 8 : (1u << 14);
    const uint32_t m32cap = tcap >= (1u << 16) ? tcap / 4 : (1u << 14);        // 64-byte slots for words of 16..31 bytes
    uint64_t upool_cap = worst ? N + (1u << 16) : Nsz / 8 + (1u << 20);
    if (upool_cap < ctx->tw_upool_hist * 2) upool_cap = ctx->tw_upool_hist * 2;
    if (upool_cap > 0xFFFFFF00ull) upool_cap = 0xFFFFFF00ull;
    if (keep) upool_cap = ctx->kept_upool_cap;
    // persistent grid: every warp keeps a private chunk of the token stream and a private model scratch
    const uint32_t grid = (uint32_t)std::min<uint64_t>(((uint64_t)n_slices + TW_WARPS - 1) / TW_WARPS, (uint64_t)ctx->sm_count * TW_BLOCKS_PER_SM);
    const uint64_t warps = (uint64_t)grid * TW_WARPS;
    // token stream: a warp claims TW_TOK_CHUNK tokens at a time and starts a slice only with TW_SLICE_TOK_MAX of them left
    double tpb = worst ? 1.0 : (ctx->tw_tok_per_byte > 0.0 ? std::min(1.0, ctx->tw_tok_per_byte * 1.25) : 0.5);
    uint64_t tok_cap = (uint64_t)((double)N * tpb) + 4096;
    tok_cap = tok_cap + tok_cap / 8 + (tok_cap * TW_SLICE_TOK_MAX) / (TW_TOK_CHUNK - TW_SLICE_TOK_MAX) + warps * TW_TOK_CHUNK;
    if (tok_cap > 0xFFFFF000ull) tok_cap = 0xFFFFF000ull;
    const uint32_t long_cap = (uint32_t)(N / 256 + 16);                        // a long word has more than 255 bytes: always enough
    const bool want_of = (P.outputs & (TKZ_OUT_OFFSETS | TKZ_OUT_OFFSETS_PACKED)) != 0;
    // token stream records: 16-bit ids when every id of the model fits, with the two offset bytes beside them in 4 bytes --
    // unless the offsets are document-relative (hf_compat), which needs the word's position in the slice as well
    const bool narrow = ctx->narrow_records && ctx->ids16_ok && !(want_of && (P.hf_flags & TKZ_HF_DOC_OFFSETS));
    // (word ids: the word's index in its slice beside the id, with or without offsets)
    const int rec = want_wid ? TW_REC_WORD : want_of ? (narrow ? TW_REC4 : TW_REC_WIDE) : (narrow ? TW_REC_ID16 : TW_REC_ID32);
    const size_t rec_bytes = (rec == TW_REC_WIDE || rec == TW_REC_WORD) ? 8 : (rec == TW_REC_ID16 ? 2 : 4);
    TRY(ensure(ctx, ctx->a_wtable, ((size_t)tcap + mcap) * sizeof(WordSlot) + (size_t)m32cap * sizeof(WordSlot32)));
    TRY(ensure(ctx, ctx->a_upool, (size_t)upool_cap * 8));
    TRY(ensure(ctx, ctx->a_lscratch, (size_t)warps * 4 * 256 * 4));
    TRY(ensure(ctx, ctx->a_tok_id, (size_t)tok_cap * rec_bytes + 16));     // (pass B copies whole 16-byte units around each run)
    TRY(ensure(ctx, ctx->a_tile_tok_off, ((size_t)n_slices + 2) * 4));
    TRY(ensure(ctx, ctx->a_tile_ntok_inline, ((size_t)n_slices + 2) * 4));
    TRY(ensure(ctx, ctx->a_tile_ntok, ((size_t)n_slices + 2) * 4));
    TRY(ensure(ctx, ctx->a_tile_long, ((size_t)n_slices + 2) * 4));
    TRY(ensure(ctx, ctx->a_tile_doc_lo, ((size_t)n_slices + 2) * 4));
    TRY(ensure(ctx, ctx->a_doc_tok_local, (n_docs + 2) * 4));
    TRY(ensure(ctx, ctx->a_long_start, (size_t)long_cap * 4));
    TRY(ensure(ctx, ctx->a_long_end, (size_t)long_cap * 4));
    TRY(ensure(ctx, ctx->a_long_slice, (size_t)long_cap * 4));
    TRY(ensure(ctx, ctx->a_long_ins, (size_t)long_cap * 4));
    if (want_wid) {
        TRY(ensure(ctx, ctx->a_slice_nword, ((size_t)n_slices + 2) * 4));
        TRY(ensure(ctx, ctx->a_doc_word_local, (n_docs + 2) * 4));
        TRY(ensure(ctx, ctx->a_doc_word_base, (n_docs + 2) * 4));
        TRY(ensure(ctx, ctx->a_long_k, (size_t)long_cap * 4));
    }
    TRY(ensure(ctx, ctx->O().doc_tok_off, (n_docs + 1) * 8));
    TRY(ensure(ctx, ctx->a_scan_tmp, (scan_tmp_elems(n_slices) + scan_tmp_elems(n_docs)) * 8));
    if (!keep) CK(cudaMemsetAsync(ctx->a_wtable.p, 0, ((size_t)tcap + mcap) * sizeof(WordSlot) + (size_t)m32cap * sizeof(WordSlot32), st));
    else { set_u32_kernel<<<1, 1, 0, st>>>((unsigned int*)(ctrl + 9), ctx->kept_upool_count); launches++; }   // (ctrl was reset: the pool goes on where it was)
    tile_doc_index_kernel<<<(n_slices + 1 + 255) / 256, 256, 0, st>>>(d_doc_off, nd, n_slices, TW_SLICE, (uint32_t*)ctx->a_tile_doc_lo.p); launches++;
    SliceArgs ta{};
    ta.text = d_text; ta.n = N; ta.doc_off = d_doc_off; ta.n_docs = nd; ta.n_slices = n_slices; ta.slice_doc_lo = (const uint32_t*)ctx->a_tile_doc_lo.p;
    ta.table = (WordSlot*)ctx->a_wtable.p; ta.table_shift = 32 - tbits; ta.med_base = tcap; ta.med_mask = mcap - 1;
    ta.table32 = (WordSlot32*)((WordSlot*)ctx->a_wtable.p + tcap + mcap); ta.table32_mask = m32cap - 1;
    ta.upool = (unsigned long long*)ctx->a_upool.p; ta.upool_cap = (uint32_t)upool_cap; ta.upool_count = (unsigned int*)(ctrl + 9);
    ta.lscratch = (uint32_t*)ctx->a_lscratch.p;
    ta.tok = ctx->a_tok_id.p;
    ta.tok_cap = (uint32_t)tok_cap; ta.tok_count = (unsigned int*)(ctrl + 5);
    ta.slice_tok_off = (uint32_t*)ctx->a_tile_tok_off.p; ta.slice_ntok_inline = (uint32_t*)ctx->a_tile_ntok_inline.p;
    ta.slice_ntok = (uint32_t*)ctx->a_tile_ntok.p; ta.slice_long = (uint32_t*)ctx->a_tile_long.p;
    ta.doc_tok_local = (uint32_t*)ctx->a_doc_tok_local.p;
    ta.long_start = (uint32_t*)ctx->a_long_start.p; ta.long_end = (uint32_t*)ctx->a_long_end.p; ta.long_slice = (uint32_t*)ctx->a_long_slice.p;
    ta.long_ins = (uint32_t*)ctx->a_long_ins.p; ta.n_long = (unsigned int*)(ctrl + 7); ta.long_cap = long_cap;
    ta.abort_flag = (unsigned int*)(ctrl + 8); ta.errw = ctrl;
    ta.n_words = ctrl + 10; ta.n_uniq = (unsigned int*)(ctrl + 6); ta.n_uncached = (unsigned int*)(ctrl + 6) + 1;
    ta.cr = cr;
    ta.n_bulk = N >= (uint64_t)(TW_SLICE + TW_POST) ? (uint32_t)std::min<uint64_t>(n_slices, (N - (TW_SLICE + TW_POST)) / TW_SLICE + 1) : 0u;
    ta.has_iso = ctx->has_iso ? 1 : 0;
    if (want_wid) { ta.slice_nword = (uint32_t*)ctx->a_slice_nword.p; ta.doc_word_local = (uint32_t*)ctx->a_doc_word_local.p; ta.long_k = (uint32_t*)ctx->a_long_k.p; }
    const int cls = (cr.usable && !ctx->force_lut) ? (cr.norm_lower ? 1 : 0) : (m.norm_identity ? 2 : 3);
    if (m.kind == TKZ_MODEL_BPE) launch_slice_words<TKZ_MODEL_BPE>(m, ta, cls, rec, grid, st);
    else launch_slice_words<TKZ_MODEL_WORDPIECE>(m, ta, cls, rec, grid, st);
    launches++;
    if (m.kind == TKZ_MODEL_BPE) { len_class_count_kernel<<<128, 256, 0, st>>>(ta.long_start, ta.long_end, 0, ta.n_long, ctrl + 13); launches++; }
    TRY(readback(ctx, hctrl, ctrl, 16 * 8));
    CK(cudaEventRecord(ctx->ev[1], st));
    CK(cudaStreamSynchronize(st));
    const uint32_t n_uniq = (uint32_t)hctrl[6], n_unc = (uint32_t)(hctrl[6] >> 32), n_long = (uint32_t)hctrl[7];
    if (ctx->call_keep) { ctx->call_uniq += n_uniq; ctx->tw_uniq_hist = std::max<uint64_t>(ctx->tw_uniq_hist, ctx->call_uniq); }
    ctx->tw_uniq_hist = std::max<uint64_t>(ctx->tw_uniq_hist, n_uniq);
    ctx->tw_upool_hist = std::max<uint64_t>(ctx->tw_upool_hist, (uint32_t)hctrl[9]);
    ctx->kept_valid = false;
    if ((uint32_t)hctrl[8] != 0) {
        ctx->call_keep = false;                              // (the retry and the rest of the call work with tables of their own)
        if (worst) { ctx->err = "internal: slice pipeline ran out of a worst-case capacity"; return TKZ_ERR_CUDA; }
        ctx->tw_tok_per_byte = 1.0;                         // later batches of this context get the worst-case token stream at once
        return TKZ_RETRY_WORST;
    }
    ctx->stats.n_unique_words = n_uniq + n_unc; ctx->stats.n_long_words = n_long;
    ctx->stats.path = 2;
    if (ctx->call_keep && !worst) { ctx->kept_valid = true; ctx->kept_tcap = tcap; ctx->kept_upool_cap = upool_cap; ctx->kept_upool_count = (uint32_t)hctrl[9]; }

    // ---- the few pre-tokens longer than TW_MAX_INLINE bytes: per-occurrence word-list kernels, counts folded back in
    TRY(ensure(ctx, ctx->a_long_ntok, ((size_t)n_long + 2) * 4));
    if (n_long) {
        TRY(ensure(ctx, ctx->a_pool_id, N * 4));
        TRY(ensure(ctx, ctx->a_pool_s, N * 4));
        TRY(ensure(ctx, ctx->a_pool_e, N * 4));
        if (m.kind == TKZ_MODEL_BPE) {
            TRY(launch_bpe(ctx, m, d_text, ta.long_start, ta.long_end, n_long, (uint32_t*)ctx->a_long_ntok.p, ctrl, 1, 1, hctrl + 13, N, launches));
        } else {
            WpArgs a{d_text, ta.long_start, ta.long_end, n_long, (uint32_t*)ctx->a_pool_id.p, (uint32_t*)ctx->a_pool_s.p, (uint32_t*)ctx->a_pool_e.p,
                     (uint32_t*)ctx->a_long_ntok.p, (unsigned int*)(ctrl + 1), ctrl, 1};
            uint64_t blocks = ((uint64_t)n_long + WP_WARPS - 1) / WP_WARPS;
            const uint64_t cap = (uint64_t)ctx->sm_count * 8; if (blocks > cap) blocks = cap;
            wordpiece_warp_kernel<<<(unsigned)blocks, WP_WARPS * 32, 0, st>>>(m, a); launches++;
        }
        long_fix_kernel<<<(n_long + 255) / 256, 256, 0, st>>>(ta.long_start, ta.long_slice, (const uint32_t*)ctx->a_long_ntok.p, n_long, ta.slice_doc_lo,
                                                               d_doc_off, ta.slice_ntok, ta.doc_tok_local, ctrl + 22); launches++;
    }
    CK(cudaEventRecord(ctx->ev[2], st));

    // ---- tokens per tile -> token base per tile; CSR offsets
    EmitParams ep = emit_params(P);
    launches += exclusive_scan<uint32_t>(ta.slice_ntok, n_slices, ta.slice_ntok, (unsigned long long*)ctx->a_scan_tmp.p, st);
    // word ids: words per slice -> global index of each slice's first word (in place)
    if (want_wid) launches += exclusive_scan<uint32_t>(ta.slice_nword, n_slices, ta.slice_nword, (unsigned long long*)ctx->a_scan_tmp.p, st);
    unsigned long long* doc_tok_off = (unsigned long long*)ctx->O().doc_tok_off.p;
    if (!plain) {
        TRY(ensure(ctx, ctx->a_doc_tok_start, (n_docs + 2) * 4));
        TRY(ensure(ctx, ctx->a_doc_real, (n_docs + 2) * 4));
        doc_finish2_kernel<<<(nd + 1 + 255) / 256, 256, 0, st>>>(d_doc_off, nd, ta.slice_ntok, ta.doc_tok_local, ep, (uint32_t*)ctx->a_doc_tok_start.p,
                                                                  (uint32_t*)ctx->a_doc_real.p, doc_tok_off, ta.slice_nword, ta.doc_word_local,
                                                                  want_wid ? (uint32_t*)ctx->a_doc_word_base.p : nullptr); launches++;
        launches += exclusive_scan<unsigned long long>(doc_tok_off, n_docs, doc_tok_off, (unsigned long long*)ctx->a_scan_tmp.p, st);
        TRY(readback(ctx, hctrl + 3, doc_tok_off + n_docs, 8));
    }
    TRY(readback(ctx, hctrl + 32, ta.slice_ntok + n_slices, 4));
    TRY(readback(ctx, hctrl, ctrl, 8));
    if (n_long) TRY(readback(ctx, hctrl + 22, ctrl + 22, 8));
    CK(cudaStreamSynchronize(st));
    const uint64_t T_real = (uint32_t)hctrl[32], T = plain ? T_real : hctrl[3];
    // one-u16 offsets: only the tokens of pre-tokens of 256 bytes or more can fail to fit; they go to a side list sized for all
    // of them -- unless they are many (skewed corpora with MiB-long words): then the call delivers 32-bit pairs
    uint32_t wide_cap = 0;
    if ((P.outputs & TKZ_OUT_OFFSETS_PACKED) && n_long) {
        const uint64_t lt = hctrl[22];
        if (lt > T_real / 8 + 4096 || lt > (4u << 20)) { P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS; ep.outputs = P.outputs; }
        else wide_cap = (uint32_t)lt;
    }
    auto fail = [&]() -> int {        // (the error word holds a byte position)
        err_doc_kernel<<<1, 1, 0, st>>>(ctrl, d_doc_off, nd); launches++;
        readback(ctx, hctrl + 4, ctrl + 4, 8);
        cudaStreamSynchronize(st);
        return report_error(ctx, hctrl[0], hctrl[4], launches, out);
    };
    if (hctrl[0] != TKZ_ERRW_NONE && n_long == 0) return fail();   // (errors of long words surface in pass B)
    CK(cudaEventRecord(ctx->ev[3], st));

    // ---- pass B
    EmitOut eo;
    TRY(alloc_outputs(ctx, ep, T, wide_cap, eo));
    const uint32_t big_cap = (uint32_t)(N / EMIT_BIG + 16);
    TRY(ensure(ctx, ctx->a_big, (size_t)big_cap * (sizeof(uint4) + 2 * sizeof(uint32_t))));
    SliceEmitArgs ea{};
    ea.doc_off = d_doc_off; ea.n_docs = nd; ea.n_slices = n_slices; ea.slice_doc_lo = ta.slice_doc_lo;
    ea.tok = ta.tok;
    ea.slice_tok_off = ta.slice_tok_off; ea.slice_ntok_inline = ta.slice_ntok_inline; ea.slice_long = ta.slice_long; ea.slice_tokbase = ta.slice_ntok;
    ea.long_start = ta.long_start; ea.long_ins = ta.long_ins; ea.long_ntok = (const uint32_t*)ctx->a_long_ntok.p;
    ea.pool_id = (const uint32_t*)ctx->a_pool_id.p; ea.pool_s = (const uint32_t*)ctx->a_pool_s.p; ea.pool_e = (const uint32_t*)ctx->a_pool_e.p;
    ea.doc_tok_local = ta.doc_tok_local; ea.doc_tok_start = (const uint32_t*)ctx->a_doc_tok_start.p;
    ea.doc_tok_off = doc_tok_off; ea.errw = ctrl; ea.err_code = m.kind == TKZ_MODEL_BPE ? TKZ_ECODE_UTF8 : TKZ_ECODE_UNK;
    ea.big = BigList{(uint4*)ctx->a_big.p, (unsigned int*)(ctrl + 16), big_cap, (uint32_t*)((uint4*)ctx->a_big.p + big_cap),
                     (uint32_t*)((uint4*)ctx->a_big.p + big_cap) + big_cap};
    if (want_wid) { ea.slice_wordbase = ta.slice_nword; ea.doc_word_base = (const uint32_t*)ctx->a_doc_word_base.p; ea.long_k = ta.long_k; }
    const bool filled = pad_prologue(ctx, ep, eo, nd, T, T_real, launches);
    const uint32_t egrid = (uint32_t)std::min<uint64_t>(((uint64_t)n_slices + TW_WARPS - 1) / TW_WARPS, (uint64_t)ctx->sm_count * 16);
    if (plain) launch_slice_emit<true>(ea, ep, eo, rec, egrid, st);
    else launch_slice_emit<false>(ea, ep, eo, rec, egrid, st);
    launches++;
    if (n_long) {
        if (want_wid) emit_big_kernel<true><<<ctx->sm_count * 4, 256, 0, st>>>(ep, eo, ea.big, ea.pool_id, ea.pool_s, ea.pool_e);
        else emit_big_kernel<false><<<ctx->sm_count * 4, 256, 0, st>>>(ep, eo, ea.big, ea.pool_id, ea.pool_s, ea.pool_e);
        launches++;
    }
    pad_epilogue(ctx, ep, eo, nd, (const uint32_t*)ctx->a_doc_real.p, doc_tok_off, filled, launches);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[4], st));
    TRY(readback(ctx, hctrl, ctrl, 11 * 8));
    if (wide_cap) TRY(readback(ctx, hctrl + 23, ctrl + 23, 8));
    CK(cudaStreamSynchronize(st));
    if (hctrl[0] != TKZ_ERRW_NONE) return fail();
    if (wide_cap && (uint32_t)hctrl[23] > wide_cap) { ctx->err = "internal: more wide offsets than tokens of long pre-tokens"; return TKZ_ERR_CUDA; }
    ctx->stats.n_words = hctrl[10];
    if (N) ctx->tw_tok_per_byte = std::max(ctx->tw_tok_per_byte, (double)T_real / (double)N);
    finish(ctx, ep, eo, doc_tok_off, n_docs, T, T_real, wide_cap ? (uint32_t)hctrl[23] : 0, launches, out);
    return TKZ_OK;
}

// The per-occurrence pipeline: models without a pre-tokenizer (every document is one pre-token), the FastTokenizer mode and
// TKZ_NO_DEDUP=1.  K1 pre-token spans, K3 / K4 one warp (or block) per pre-token, scans to CSR offsets, K5 emit.
int encode_words(tkz_ctx* ctx, const DevModel& m, const uint8_t* d_text, const uint64_t* d_doc_off, uint32_t nd, uint64_t N,
                 tkz_encode_params P, tkz_batch_result* out, uint64_t& launches) {
    cudaStream_t st = ctx->stream;
    unsigned long long* ctrl = (unsigned long long*)ctx->a_ctrl.p;
    unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
    const uint64_t n_docs = nd;
    // a pre-token can have any length: offsets are delivered as 32-bit pairs
    if (P.outputs & TKZ_OUT_OFFSETS_PACKED) P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS;

    // ---- K1: pre-token spans
    uint64_t W = 0;
    TRY(ensure(ctx, ctx->a_doc_word_off, (n_docs + 1) * 4));
    uint32_t* doc_word_off = (uint32_t*)ctx->a_doc_word_off.p;
    if (m.has_pretok) {
        const uint64_t n_tiles = N / SPLIT_TILE + 1;
        TRY(ensure(ctx, ctx->a_tiles, (n_tiles + 1) * 8));
        TRY(ensure(ctx, ctx->a_scan_tmp, scan_tmp_elems(n_tiles) * 8));
        unsigned long long* tiles = (unsigned long long*)ctx->a_tiles.p;
        split_count_kernel<<<(unsigned)n_tiles, SPLIT_THREADS, 0, st>>>(m, d_text, N, d_doc_off, nd, tiles); launches++;
        launches += exclusive_scan<unsigned long long>(tiles, n_tiles, tiles, (unsigned long long*)ctx->a_scan_tmp.p, st);
        TRY(readback(ctx, hctrl + 8, tiles + n_tiles, 8));
        CK(cudaStreamSynchronize(st));
        const unsigned long long tot = hctrl[8];
        W = tot >> 32;
        if ((tot & 0xFFFFFFFFull) != W) { ctx->err = "internal: word start/end counts differ"; return TKZ_ERR_CUDA; }
        TRY(ensure(ctx, ctx->a_word_start, (W + 1) * 4));
        TRY(ensure(ctx, ctx->a_word_end, (W + 1) * 4));
        TRY(ensure(ctx, ctx->a_word_doc, (W + 1) * 4));
        split_write_kernel<<<(unsigned)n_tiles, SPLIT_THREADS, 0, st>>>(m, d_text, N, d_doc_off, nd, tiles, (uint32_t*)ctx->a_word_start.p,
                                                                        (uint32_t*)ctx->a_word_end.p, (uint32_t*)ctx->a_word_doc.p, doc_word_off); launches++;
    } else {
        W = n_docs;
        TRY(ensure(ctx, ctx->a_word_start, (W + 1) * 4));
        TRY(ensure(ctx, ctx->a_word_end, (W + 1) * 4));
        TRY(ensure(ctx, ctx->a_word_doc, (W + 1) * 4));
        words_from_docs_kernel<<<(unsigned)((n_docs + 1 + 255) / 256), 256, 0, st>>>(d_doc_off, nd, (uint32_t*)ctx->a_word_start.p,
                                                                                     (uint32_t*)ctx->a_word_end.p, (uint32_t*)ctx->a_word_doc.p, doc_word_off); launches++;
    }
    const uint32_t nw = (uint32_t)W;
    uint32_t* word_start = (uint32_t*)ctx->a_word_start.p;
    uint32_t* word_end = (uint32_t*)ctx->a_word_end.p;
    uint32_t* word_doc = (uint32_t*)ctx->a_word_doc.p;

    CK(cudaEventRecord(ctx->ev[1], st));
    // ---- K3 / K4: model, one warp per pre-token
    TRY(ensure(ctx, ctx->a_word_ntok, (W + 2) * 4));
    TRY(ensure(ctx, ctx->a_pool_id, N * 4));
    TRY(ensure(ctx, ctx->a_pool_s, N * 4));
    TRY(ensure(ctx, ctx->a_pool_e, N * 4));
    uint32_t* word_ntok = (uint32_t*)ctx->a_word_ntok.p;
    unsigned int* work_counter = (unsigned int*)(ctrl + 1);
    if (nw && P.fast) {
        // FastTokenizer mode: one thread per pre-token replays tokenizeFast (tkz_fast.cuh)
        TRY(ensure(ctx, ctx->a_pool_rk, N * 4));
        TRY(ensure(ctx, ctx->a_fast_heap, N * 16 + 64));
        TRY(ensure(ctx, ctx->a_word_aux, (W + 2) * 4));
        FastArgs fa{d_text, word_start, word_end, word_doc, doc_word_off, nw, P.fast_max_sequence_length, P.fast_max_tokens,
                    (uint32_t*)ctx->a_pool_id.p, (uint32_t*)ctx->a_pool_s.p, (uint32_t*)ctx->a_pool_e.p, (uint32_t*)ctx->a_pool_rk.p,
                    (unsigned long long*)ctx->a_fast_heap.p, word_ntok, (uint32_t*)ctx->a_word_aux.p, ctrl};
        if (m.kind == TKZ_MODEL_BPE) { fast_bpe_kernel<<<(nw + 127) / 128, 128, 0, st>>>(m, fa); launches++; }
        else {
            fast_wp_kernel<<<(nw + 127) / 128, 128, 0, st>>>(m, fa); launches++;
            if (nd) { fast_wp_fix_kernel<<<(unsigned)(((uint64_t)nd * 32 + 255) / 256), 256, 0, st>>>(fa, nd); launches++; }
        }
    } else if (nw) {
        if (m.kind == TKZ_MODEL_BPE) {
            len_class_count_kernel<<<128, 256, 0, st>>>(word_start, word_end, nw, nullptr, ctrl + 13); launches++;
            TRY(readback(ctx, hctrl + 24, ctrl + 13, 3 * 8));
            CK(cudaStreamSynchronize(st));
            TRY(launch_bpe(ctx, m, d_text, word_start, word_end, nw, word_ntok, ctrl, 1, 0, hctrl + 24, N, launches));
        } else {
            WpArgs a{d_text, word_start, word_end, nw, (uint32_t*)ctx->a_pool_id.p, (uint32_t*)ctx->a_pool_s.p, (uint32_t*)ctx->a_pool_e.p,
                     word_ntok, work_counter, ctrl, 0};
            uint64_t blocks = (W + WP_WARPS - 1) / WP_WARPS;
            const uint64_t cap = (uint64_t)ctx->sm_count * 8;
            if (blocks > cap) blocks = cap;
            wordpiece_warp_kernel<<<(unsigned)blocks, WP_WARPS * 32, 0, st>>>(m, a); launches++;
        }
    }

    CK(cudaEventRecord(ctx->ev[2], st));
    // ---- scans: tokens per word -> per document -> CSR
    TRY(ensure(ctx, ctx->a_scan_tmp, (scan_tmp_elems(W) + scan_tmp_elems(n_docs)) * 8));
    launches += exclusive_scan<uint32_t>(word_ntok, W, word_ntok, (unsigned long long*)ctx->a_scan_tmp.p, st);
    const uint32_t* word_tok_off = word_ntok;
    TRY(ensure(ctx, ctx->O().doc_tok_off, (n_docs + 1) * 8));
    unsigned long long* doc_tok_off = (unsigned long long*)ctx->O().doc_tok_off.p;
    const EmitParams ep = emit_params(P);
    uint32_t* doc_real = nullptr;                           // (only the padding / template kernels read it)
    if (ep.has_pad || has_frame(ep)) { TRY(ensure(ctx, ctx->a_doc_real, (n_docs + 2) * 4)); doc_real = (uint32_t*)ctx->a_doc_real.p; }
    if (nd) { doc_len_kernel<<<(nd + 255) / 256, 256, 0, st>>>(ep, word_tok_off, doc_word_off, nd, doc_tok_off, doc_real); launches++; }
    launches += exclusive_scan<unsigned long long>(doc_tok_off, n_docs, doc_tok_off, (unsigned long long*)ctx->a_scan_tmp.p, st);
    gather_scalars_kernel<<<1, 1, 0, st>>>(ctrl, word_tok_off, nw, doc_tok_off, nd, word_doc); launches++;
    TRY(readback(ctx, hctrl, ctrl, 5 * 8));
    CK(cudaStreamSynchronize(st));
    const uint64_t T_real = hctrl[2], T = hctrl[3];
    ctx->stats.n_words = W; ctx->stats.n_unique_words = W; ctx->stats.n_long_words = 0;
    if (hctrl[0] != TKZ_ERRW_NONE) return report_error(ctx, hctrl[0], hctrl[4], launches, out);   // (the error word holds a word index)

    CK(cudaEventRecord(ctx->ev[3], st));
    // ---- K5: emit
    EmitOut eo;
    TRY(alloc_outputs(ctx, ep, T, 0, eo));
    const bool filled = pad_prologue(ctx, ep, eo, nd, T, T_real, launches);
    if (nw) {
        const uint32_t big_cap = (uint32_t)(N / EMIT_BIG + 16);
        TRY(ensure(ctx, ctx->a_big, (size_t)big_cap * (sizeof(uint4) + 2 * sizeof(uint32_t))));
        BigList bl{(uint4*)ctx->a_big.p, (unsigned int*)(ctrl + 9) + 1, big_cap, (uint32_t*)((uint4*)ctx->a_big.p + big_cap),
                   (uint32_t*)((uint4*)ctx->a_big.p + big_cap) + big_cap};
        const uint32_t *pid = (const uint32_t*)ctx->a_pool_id.p, *ps = (const uint32_t*)ctx->a_pool_s.p, *pe = (const uint32_t*)ctx->a_pool_e.p;
        if (ep.outputs & TKZ_OUT_WORD_IDS) {
            emit_words_kernel<true><<<(nw + 255) / 256, 256, 0, st>>>(ep, eo, nw, word_start, word_doc, word_tok_off, doc_word_off, doc_tok_off, pid, ps, pe, bl, d_doc_off);
            emit_big_kernel<true><<<ctx->sm_count * 4, 256, 0, st>>>(ep, eo, bl, pid, ps, pe);
        } else {
            emit_words_kernel<false><<<(nw + 255) / 256, 256, 0, st>>>(ep, eo, nw, word_start, word_doc, word_tok_off, doc_word_off, doc_tok_off, pid, ps, pe, bl, d_doc_off);
            emit_big_kernel<false><<<ctx->sm_count * 4, 256, 0, st>>>(ep, eo, bl, pid, ps, pe);
        }
        launches += 2;
    }
    pad_epilogue(ctx, ep, eo, nd, doc_real, doc_tok_off, filled, launches);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[4], st));
    CK(cudaStreamSynchronize(st));
    finish(ctx, ep, eo, doc_tok_off, n_docs, T, T_real, 0, launches, out);
    return TKZ_OK;
}

// TKZ_HF_OVERFLOW (tkz_overflow.cuh): what a pipeline left in the staging output set (*out: every document's real tokens, no
// truncation, padding or template) becomes rows of the call's output set, one per window.  P = the call's parameters.
int encode_overflow(tkz_ctx* ctx, const tkz_encode_params& P, uint64_t launches, tkz_batch_result* out) {
    cudaStream_t st = ctx->stream;
    unsigned long long* ctrl = (unsigned long long*)ctx->a_ctrl.p;
    unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
    const tkz_batch_result stage = *out;
    const uint32_t nd = (uint32_t)stage.n_docs;
    const unsigned long long* stage_off = (const unsigned long long*)stage.doc_tok_off;
    const EmitParams ep = emit_params(P);
    const uint64_t L = P.max_length - ((P.hf_flags & TKZ_HF_TEMPLATE) ? P.tpl_n_prefix + P.tpl_n_suffix : 0u), step = L - P.stride;
    auto& O = ctx->O();
    // ---- rows per document -> doc_row_off
    TRY(ensure(ctx, O.doc_row_off, ((size_t)nd + 2) * 8));
    TRY(ensure(ctx, ctx->a_scan_tmp, scan_tmp_elems(nd) * 8));
    unsigned long long* doc_row_off = (unsigned long long*)O.doc_row_off.p;
    if (nd) { ovf_doc_rows_kernel<<<(nd + 255) / 256, 256, 0, st>>>(stage_off, nd, L, step, doc_row_off, ctrl + 24); launches++; }
    launches += exclusive_scan<unsigned long long>(doc_row_off, nd, doc_row_off, (unsigned long long*)ctx->a_scan_tmp.p, st);
    TRY(readback(ctx, hctrl + 48, doc_row_off + nd, 8));
    TRY(readback(ctx, hctrl + 49, ctrl + 24, 8));
    CK(cudaStreamSynchronize(st));
    const uint64_t R = hctrl[48], rows_real = hctrl[49];
    // (the epilogue kernels index documents -- rows here -- with a u32)
    if (R >= (1ull << 32)) { ctx->err = "overflowing windows: 2^32 rows or more in one call"; return TKZ_ERR_INVALID_ARG; }
    const uint32_t nr = (uint32_t)R;
    // ---- each row's document, window length and slots -> row_tok_off
    TRY(ensure(ctx, O.row_tok_off, (R + 2) * 8));
    TRY(ensure(ctx, ctx->a_row_real, (R + 2) * 4));
    TRY(ensure(ctx, ctx->a_row_doc, (R + 2) * 4));
    TRY(ensure(ctx, ctx->a_scan_tmp, scan_tmp_elems(R) * 8));
    unsigned long long* row_tok_off = (unsigned long long*)O.row_tok_off.p;
    const uint32_t* row_real = (const uint32_t*)ctx->a_row_real.p;
    const uint32_t* row_doc = (const uint32_t*)ctx->a_row_doc.p;
    if (nr) {
        ovf_row_len_kernel<<<(nr + 255) / 256, 256, 0, st>>>(ep, stage_off, doc_row_off, nd, nr, L, step, row_tok_off, (uint32_t*)row_real, (uint32_t*)row_doc);
        launches++;
    }
    launches += exclusive_scan<unsigned long long>(row_tok_off, R, row_tok_off, (unsigned long long*)ctx->a_scan_tmp.p, st);
    TRY(readback(ctx, hctrl + 50, row_tok_off + R, 8));
    CK(cudaStreamSynchronize(st));
    const uint64_t T = hctrl[50];
    // ---- the rows: windows, then the template's special tokens and the padding of the shared epilogue
    TRY(ensure(ctx, O.doc_tok_off, ((size_t)nd + 1) * 8));
    EmitOut eo;
    TRY(alloc_outputs(ctx, ep, T, 0, eo));
    const bool filled = pad_prologue(ctx, ep, eo, nr, T, rows_real, launches);
    const OvfStage src{stage.ids, stage.ids16, (const uint2*)stage.offsets, stage.word_ids};
    if (nr) {
        const unsigned g = (unsigned)(((uint64_t)nr * 32 + 255) / 256);
        if (ep.outputs & TKZ_OUT_WORD_IDS) ovf_copy_kernel<true><<<g, 256, 0, st>>>(ep, eo, src, nr, step, stage_off, doc_row_off, row_tok_off, row_real, row_doc);
        else ovf_copy_kernel<false><<<g, 256, 0, st>>>(ep, eo, src, nr, step, stage_off, doc_row_off, row_tok_off, row_real, row_doc);
        launches++;
    }
    unsigned long long* doc_tok_off = (unsigned long long*)O.doc_tok_off.p;
    ovf_doc_off_kernel<<<(nd + 1 + 255) / 256, 256, 0, st>>>(doc_row_off, row_tok_off, nd, doc_tok_off); launches++;
    pad_epilogue(ctx, ep, eo, nr, row_real, row_tok_off, filled, launches);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[4], st));
    CK(cudaStreamSynchronize(st));
    finish(ctx, ep, eo, doc_tok_off, nd, T, stage.n_real_tokens, 0, launches, out);
    out->n_rows = R; out->row_tok_off = (const uint64_t*)row_tok_off; out->doc_row_off = (const uint64_t*)doc_row_off;
    return TKZ_OK;
}

int encode_device_impl(tkz_ctx* ctx, const uint8_t* d_text, const uint64_t* d_doc_off, uint64_t n_docs, uint64_t N,
                       const tkz_encode_params* params, tkz_batch_result* out) {
    memset(out, 0, sizeof *out);
    out->err_doc = -1;
    if (!ctx->has_model) { ctx->err = "no model uploaded"; return TKZ_ERR_INVALID_ARG; }
    ctx->grid_used = false; ctx->retried = false;
    if (N >= 0xFFFFF000ull) { ctx->err = "batch text must be < 4 GiB (u32 offsets, types.zig:4-6): split the batch"; return TKZ_ERR_INVALID_ARG; }
    if (n_docs >= 0xFFFFFFF0ull) { ctx->err = "too many documents in one batch"; return TKZ_ERR_INVALID_ARG; }
    ON_DEVICE(ctx);
    cudaStream_t st = ctx->stream;
    uint64_t launches = 0;
    tkz_encode_params P{};
    if (params) P = *params;
    if (P.outputs == 0) P.outputs = TKZ_OUT_ALL;
    P.outputs |= TKZ_OUT_IDS;
    if (P.fast) {
        // FastTokenizer.encode: no truncation / padding parameters; the token buffer of the arena caps every document
        if (P.fast_max_sequence_length == 0) P.fast_max_sequence_length = 8192;        // ArenaConfig defaults (arena.zig:140-145)
        if (P.fast_max_tokens == 0) P.fast_max_tokens = 512;
        if (P.fast_max_sequence_length < 4 || P.fast_max_sequence_length > 65535) { ctx->err = "fast_max_sequence_length must be 4 .. 65535 (16-bit symbol indices, arena.zig:17-42)"; return TKZ_ERR_INVALID_ARG; }
        P.has_truncation = 1; P.max_length = P.fast_max_tokens; P.has_padding = 0;
    }
    // (before the template's ids are checked against the u16 form: a vocabulary with larger ids ignores it)
    if ((P.outputs & TKZ_OUT_IDS_U16) && (!ctx->ids16_ok || (P.has_padding && P.pad_id > 0xFFFFu))) P.outputs &= ~TKZ_OUT_IDS_U16;
    if (P.hf_flags) {
        // hf_compat (beyond the reference, opt-in)
        if (P.hf_flags & ~(uint32_t)(TKZ_HF_TEMPLATE | TKZ_HF_DOC_OFFSETS | TKZ_HF_OVERFLOW)) { ctx->err = "unknown hf_flags bit"; return TKZ_ERR_INVALID_ARG; }
        if (P.fast) { ctx->err = "hf_flags cannot be combined with the FastTokenizer mode"; return TKZ_ERR_INVALID_ARG; }
        if (P.tpl_n_prefix > TKZ_TPL_MAX || P.tpl_n_suffix > TKZ_TPL_MAX) { ctx->err = "at most TKZ_TPL_MAX special tokens on either side of the sequence"; return TKZ_ERR_INVALID_ARG; }
        if (!(P.hf_flags & TKZ_HF_TEMPLATE)) { P.tpl_n_prefix = P.tpl_n_suffix = 0; P.tpl_seq_type = 0; }
        if (P.outputs & TKZ_OUT_IDS_U16)
            for (uint32_t i = 0; i < TKZ_TPL_MAX; i++)
                if ((i < P.tpl_n_prefix && P.tpl_prefix_id[i] > 0xFFFFu) || (i < P.tpl_n_suffix && P.tpl_suffix_id[i] > 0xFFFFu)) { ctx->err = "template id above 65535 with TKZ_OUT_IDS_U16"; return TKZ_ERR_INVALID_ARG; }
        // document-relative offsets do not fit the one-u16-per-token form
        if ((P.hf_flags & TKZ_HF_DOC_OFFSETS) && (P.outputs & TKZ_OUT_OFFSETS_PACKED)) P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS;
        if (P.hf_flags & TKZ_HF_OVERFLOW) {
            const uint64_t added = (P.hf_flags & TKZ_HF_TEMPLATE) ? P.tpl_n_prefix + P.tpl_n_suffix : 0u;
            if (!P.has_truncation) { ctx->err = "overflowing windows need truncation"; return TKZ_ERR_INVALID_ARG; }
            if (P.max_length <= added || P.stride >= P.max_length - added) { ctx->err = "overflowing windows need stride < max_length minus the template's tokens"; return TKZ_ERR_INVALID_ARG; }
            if (P.outputs & TKZ_OUT_SPAN_TOKENS) { ctx->err = "overflowing windows do not carry span tokens"; return TKZ_ERR_INVALID_ARG; }
            // (the windows are copied with their 32-bit offsets)
            if (P.outputs & TKZ_OUT_OFFSETS_PACKED) P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS;
        }
    }
    if (P.outputs & TKZ_OUT_WORD_IDS) {
        if (P.fast) { ctx->err = "word ids cannot be combined with the FastTokenizer mode"; return TKZ_ERR_INVALID_ARG; }
        // (the slice pipeline's token records keep the word's index in the slice above a 22-bit id)
        if (ctx->max_id >= (1u << 22)) { ctx->err = "word ids need every id of the model below 2^22"; return TKZ_ERR_INVALID_ARG; }
    }
    // overflowing windows: the pipelines encode into the staging set with no truncation, padding or template tokens, and ask
    // only for the arrays that differ per token (the document-offset shift stays theirs)
    const bool overflow = (P.hf_flags & TKZ_HF_OVERFLOW) != 0;
    tkz_encode_params S = P;
    if (overflow) {
        S.has_truncation = 0; S.has_padding = 0; S.hf_flags = P.hf_flags & TKZ_HF_DOC_OFFSETS;
        S.outputs = TKZ_OUT_IDS | (P.outputs & (TKZ_OUT_IDS_U16 | TKZ_OUT_OFFSETS | TKZ_OUT_WORD_IDS));
    }
    const uint32_t nd = (uint32_t)n_docs;
    DevModel m = ctx->dm;

    // misaligned text: stage into the arena (the split scan uses 16-byte vector loads)
    if (((uintptr_t)d_text & 15u) != 0 && N) {
        TRY(ensure(ctx, ctx->a_text, N));
        CK(cudaMemcpyAsync(ctx->a_text.p, d_text, N, cudaMemcpyDeviceToDevice, st));
        d_text = (const uint8_t*)ctx->a_text.p;
    }
    unsigned long long* ctrl = (unsigned long long*)ctx->a_ctrl.p;
    unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
    CK(cudaEventRecord(ctx->ev[0], st));
    ctrl_reset_kernel<<<1, 1, 0, st>>>(ctrl); launches++;

    // ---- K0: normalizer that drops bytes
    if (m.norm_has_drop) {
        const uint64_t n_chunks = N / NORM_CHUNK + 1;
        TRY(ensure(ctx, ctx->a_chunk, (n_chunks + 1) * 4));
        TRY(ensure(ctx, ctx->a_scan_tmp, scan_tmp_elems(n_chunks) * 8));
        TRY(ensure(ctx, ctx->a_norm_text, N));
        TRY(ensure(ctx, ctx->a_norm_doc_off, (n_docs + 1) * 8));
        uint32_t* chunk = (uint32_t*)ctx->a_chunk.p;
        norm_count_kernel<<<(unsigned)n_chunks, 256, 0, st>>>(m, d_text, N, chunk); launches++;
        launches += exclusive_scan<uint32_t>(chunk, n_chunks, chunk, (unsigned long long*)ctx->a_scan_tmp.p, st);
        norm_write_kernel<<<(unsigned)n_chunks, 256, 0, st>>>(m, d_text, N, chunk, (uint8_t*)ctx->a_norm_text.p); launches++;
        norm_docoff_kernel<<<(unsigned)((n_docs + 1 + 255) / 256), 256, 0, st>>>(m, d_text, N, chunk, d_doc_off, nd, (uint64_t*)ctx->a_norm_doc_off.p); launches++;
        TRY(readback(ctx, hctrl + 8, chunk + n_chunks, 4));
        CK(cudaStreamSynchronize(st));
        N = *(uint32_t*)(hctrl + 8);
        d_text = (const uint8_t*)ctx->a_norm_text.p;
        d_doc_off = (const uint64_t*)ctx->a_norm_doc_off.p;
        m = ctx->dm_post;
    }

    // ---- slice pipeline (tkz_slices.cuh) whenever there is a pre-tokenizer; TKZ_NO_DEDUP=1 keeps the per-occurrence
    //      pipeline for A/B tests
    ctx->stats.path = 0;
    const int out_sel = ctx->out_sel;
    if (overflow) ctx->out_sel = 2;
    int rc;
    if (m.has_pretok && ctx->use_dedup && !P.fast) {
        const ClassRanges& cr = ctx->dm.norm_has_drop ? ctx->cr_post : ctx->cr;      // (K0 ran: the text is already normalised)
        rc = encode_slices(ctx, m, cr, d_text, d_doc_off, nd, N, S, false, out, launches);
        if (rc == TKZ_RETRY_WORST) {
            ctx->retried = true;
            ctrl_reset_kernel<<<1, 1, 0, st>>>(ctrl); launches++;
            rc = encode_slices(ctx, m, cr, d_text, d_doc_off, nd, N, S, true, out, launches);
        }
    } else rc = encode_words(ctx, m, d_text, d_doc_off, nd, N, S, out, launches);
    ctx->out_sel = out_sel;
    if (rc != TKZ_OK || !overflow) return rc;
    return encode_overflow(ctx, P, launches, out);
}

}  // namespace

extern "C" int tkz_encode_batch_device(tkz_ctx* ctx, const void* d_text, const void* d_doc_off, uint64_t n_docs, uint64_t text_bytes,
                                       const tkz_encode_params* params, tkz_batch_result* out) {
    if (!ctx || !out || !d_doc_off || (text_bytes && !d_text)) return TKZ_ERR_INVALID_ARG;
    return encode_device_impl(ctx, (const uint8_t*)d_text, (const uint64_t*)d_doc_off, n_docs, text_bytes, params, out);
}

namespace {

// grows a pinned host result array keeping its first `keep` bytes
int ensure_host_keep(tkz_ctx* ctx, HostBuf& b, size_t bytes, size_t keep) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return TKZ_OK;
    CK(cudaStreamSynchronize(ctx->s_d2h));
    void* np = nullptr;
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaHostAlloc(&np, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { ctx->err = std::string("cudaHostAlloc: ") + cudaGetErrorString(e); return TKZ_ERR_OOM; }
    if (b.p) { if (keep) memcpy(np, b.p, keep); cudaFreeHost(b.p); }
    b.p = np; b.cap = want;
    return TKZ_OK;
}

// wide-offset records {slot lo, slot hi, start, end}: add a base to the slots of [first, first + n) and sort the whole list by slot
struct WideRec { uint32_t lo, hi, s, e; };
void wide_finish(WideRec* w, uint64_t n_total, const std::vector<std::array<uint64_t, 3>>& parts) {
    for (const auto& pt : parts)
        for (uint64_t k = pt[0]; k < pt[0] + pt[1]; k++) { const uint64_t v = (((uint64_t)w[k].hi << 32) | w[k].lo) + pt[2]; w[k].lo = (uint32_t)v; w[k].hi = (uint32_t)(v >> 32); }
    std::sort(w, w + n_total, [](const WideRec& a, const WideRec& b) { return a.hi != b.hi ? a.hi < b.hi : a.lo < b.lo; });
}

// the per-token arrays of a device result (ResultArrays order), the pinned host arrays they are copied to, bytes per slot
struct ResultCopy { const void* dev; HostBuf* host; size_t elem; };
// (word ids are relative to their document: chunks of the host path copy them as they are)
std::array<ResultCopy, N_RESULT_ARRAYS> result_copies(tkz_ctx* ctx, const tkz_batch_result& r) {
    return {{{r.ids, &ctx->h_ids, 4}, {r.offsets, &ctx->h_off, 8}, {r.attention_mask, &ctx->h_attn, 4}, {r.type_ids, &ctx->h_type, 4},
             {r.special_tokens_mask, &ctx->h_special, 4}, {r.offsets_packed, &ctx->h_off16, 2}, {r.ids16, &ctx->h_ids16, 2},
             {r.span_tokens, &ctx->h_spans, 16}, {r.word_ids, &ctx->h_wid, 4}}};
}

// one shot: H2D everything, encode, D2H everything (small batches)
int encode_host_single(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs, uint64_t N,
                       const tkz_encode_params* params, tkz_batch_result* out) {
    ctx->out_sel = 0;
    TRY(ensure(ctx, ctx->a_text, N));
    TRY(ensure(ctx, ctx->a_doc_off, (n_docs + 1) * 8));
    if (N) CK(cudaMemcpyAsync(ctx->a_text.p, text, N, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->a_doc_off.p, doc_off, (n_docs + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    tkz_batch_result dev{};
    int rc = encode_device_impl(ctx, (const uint8_t*)ctx->a_text.p, (const uint64_t*)ctx->a_doc_off.p, n_docs, N, params, &dev);
    *out = dev;
    set_result(out, dev.n_docs, dev.n_tokens, dev.n_real_tokens, nullptr, {}, 0, nullptr);    // (no device pointer leaves)
    out->row_tok_off = out->doc_row_off = nullptr;
    if (rc != TKZ_OK) return rc;
    const uint64_t T = dev.n_tokens;
    cudaStream_t st = ctx->stream;
    TRY(ensure_host(ctx, ctx->h_doc_tok_off, (n_docs + 1) * 8));
    CK(cudaMemcpyAsync(ctx->h_doc_tok_off.p, dev.doc_tok_off, (n_docs + 1) * 8, cudaMemcpyDeviceToHost, st));
    const auto cp = result_copies(ctx, dev);
    ResultArrays host{};
    for (uint32_t i = 0; i < N_RESULT_ARRAYS; i++) {
        if (!cp[i].dev) continue;
        TRY(ensure_host(ctx, *cp[i].host, T * cp[i].elem));
        if (T) CK(cudaMemcpyAsync(cp[i].host->p, cp[i].dev, T * cp[i].elem, cudaMemcpyDeviceToHost, st));
        host[i] = cp[i].host->p;
    }
    if (dev.n_wide) {
        TRY(ensure_host(ctx, ctx->h_wide, dev.n_wide * 16));
        CK(cudaMemcpyAsync(ctx->h_wide.p, dev.wide_tokens, dev.n_wide * 16, cudaMemcpyDeviceToHost, st));
    }
    if (dev.n_rows) {
        TRY(ensure_host(ctx, ctx->h_row_tok_off, (dev.n_rows + 1) * 8));
        TRY(ensure_host(ctx, ctx->h_doc_row_off, (n_docs + 1) * 8));
        CK(cudaMemcpyAsync(ctx->h_row_tok_off.p, dev.row_tok_off, (dev.n_rows + 1) * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(ctx->h_doc_row_off.p, dev.doc_row_off, (n_docs + 1) * 8, cudaMemcpyDeviceToHost, st));
        out->row_tok_off = (const uint64_t*)ctx->h_row_tok_off.p; out->doc_row_off = (const uint64_t*)ctx->h_doc_row_off.p;
    }
    CK(cudaStreamSynchronize(st));
    if (dev.n_wide) wide_finish((WideRec*)ctx->h_wide.p, dev.n_wide, {});
    set_result(out, dev.n_docs, T, dev.n_real_tokens, (const uint64_t*)ctx->h_doc_tok_off.p, host, dev.n_wide, ctx->h_wide.p);
    ctx->stats.ms_call_kernels = ctx->stats.ms_total;
    return TKZ_OK;
}

// chunked: documents are cut into ~chunk_bytes pieces; the H2D copy of chunk i+1 and the D2H copy of chunk i-1 run on
// their own streams while the kernels of chunk i run (PCIe is full duplex).  Input and output device buffers are
// double-buffered; results land in one set of pinned host arrays at their final positions.
int encode_host_chunked(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs, uint64_t N,
                        const tkz_encode_params* params_in, tkz_batch_result* out) {
    memset(out, 0, sizeof *out);
    out->err_doc = -1;
    // chunk boundaries (document indices) are decided as the call goes: a chunk of `target` bytes ends at the last document
    // boundary not beyond it (at least one document).  The target starts at chunk_bytes; when the kernels of a chunk take longer
    // than its transfers would (long-word corpora: the block / grid kernels want many words in flight) it doubles, up to 8x
    std::vector<uint64_t> cb; cb.push_back(0);
    auto next_boundary = [&](uint64_t d0, uint64_t target_bytes) -> uint64_t {
        const uint64_t target = doc_off[d0] + target_bytes;
        uint64_t lo = d0 + 1, hi = n_docs;                       // last boundary with doc_off <= target, at least one document
        while (lo < hi) { const uint64_t mid = lo + (hi - lo + 1) / 2; if (doc_off[mid] <= target) lo = mid; else hi = mid - 1; }
        return lo;
    };
    uint64_t chunk_target = ctx->chunk_bytes;
    const uint64_t chunk_max = std::min<uint64_t>(ctx->chunk_bytes * 8, 1ull << 30);
    struct KeepGuard { tkz_ctx* c; ~KeepGuard() { c->call_keep = false; c->kept_valid = false; c->call_bytes = 0; } } keep_guard{ctx};
    ctx->call_keep = true; ctx->kept_valid = false; ctx->call_bytes = N; ctx->call_uniq = 0;
    cb.push_back(next_boundary(0, chunk_target));
    tkz_encode_params P{};
    if (params_in) P = *params_in;
    if (P.outputs == 0) P.outputs = TKZ_OUT_ALL;
    P.outputs |= TKZ_OUT_IDS;
    // overflowing windows: a chunk never splits a document, so it never splits a document's rows either; row offsets are shifted
    // by the chunk's slot base and document-row offsets by its row base, like doc_tok_off.  (Offsets come as 32-bit pairs.)
    const bool overflow = (P.hf_flags & TKZ_HF_OVERFLOW) != 0;
    if (overflow && (P.outputs & TKZ_OUT_OFFSETS_PACKED)) P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS;
    TRY(ensure_host(ctx, ctx->h_doc_tok_off, (n_docs + 1) * 8));
    uint64_t* h_dto = (uint64_t*)ctx->h_doc_tok_off.p;
    if (overflow) TRY(ensure_host(ctx, ctx->h_doc_row_off, (n_docs + 1) * 8));
    uint64_t* h_dro = (uint64_t*)ctx->h_doc_row_off.p;
    auto stage_in = [&](size_t i) -> int {
        const int b = (int)(i & 1);
        const uint64_t d0 = cb[i], d1 = cb[i + 1], base = doc_off[d0], nb = doc_off[d1] - base, nd = d1 - d0;
        TRY(ensure(ctx, ctx->in_text[b], nb));
        TRY(ensure(ctx, ctx->in_doc_off[b], (nd + 1) * 8));
        TRY(ensure_host(ctx, ctx->h_doc_stage[b], (nd + 1) * 8));
        uint64_t* st = (uint64_t*)ctx->h_doc_stage[b].p;
        for (uint64_t k = 0; k <= nd; k++) st[k] = doc_off[d0 + k] - base;
        if (nb) CK(cudaMemcpyAsync(ctx->in_text[b].p, text + base, nb, cudaMemcpyHostToDevice, ctx->s_h2d));
        CK(cudaMemcpyAsync(ctx->in_doc_off[b].p, st, (nd + 1) * 8, cudaMemcpyHostToDevice, ctx->s_h2d));
        CK(cudaEventRecord(ctx->ev_h2d[b], ctx->s_h2d));
        return TKZ_OK;
    };
    ResultArrays host{};
restart:
    cb.resize(2); chunk_target = ctx->chunk_bytes; ctx->kept_valid = false; ctx->call_uniq = 0;
    uint64_t W_total = 0; std::vector<std::array<uint64_t, 3>> wide_parts;
    TRY(stage_in(0));
    uint64_t T_total = 0, T_real = 0, R_total = 0;
    float ms_kernels = 0.f;
    for (size_t i = 0; cb[i] < n_docs; i++) {
        const int b = (int)(i & 1);
        const uint64_t d0 = cb[i], d1 = cb[i + 1], nd = d1 - d0, nb = doc_off[d1] - doc_off[d0];
        const auto tr0 = std::chrono::steady_clock::now();
        if (d1 < n_docs) {
            cb.push_back(next_boundary(d1, chunk_target));
            // buffer (i+1)&1 was read by the kernels of chunk i-1 and its staging area by the H2D of chunk i-1, which those kernels
            // waited for: both finished when the device path of chunk i-1 drained its stream.  No host wait for the copy of
            // chunk i: its kernels wait for it on the device (event below).
            TRY(stage_in(i + 1));
        }
        const auto tr1 = std::chrono::steady_clock::now();
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[b], 0));
        CK(cudaEventSynchronize(ctx->ev_d2h[b]));              // output set b is free once chunk i-2 has been copied out
        const auto tr2 = std::chrono::steady_clock::now();
        ctx->out_sel = b;
        tkz_batch_result dev{};
        int rc = encode_device_impl(ctx, (const uint8_t*)ctx->in_text[b].p, (const uint64_t*)ctx->in_doc_off[b].p, nd, nb, &P, &dev);
        const auto tr3 = std::chrono::steady_clock::now();
        if (getenv("TKZ_HOST_TRACE")) {
            auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            fprintf(stderr, "[trace] chunk %zu docs %llu bytes %llu stage %.3f wait_d2h %.3f device_call %.3f (kernels %.3f: split %.3f model %.3f scan %.3f emit %.3f)\n", i, (unsigned long long)nd, (unsigned long long)nb, ms(tr0, tr1), ms(tr1, tr2), ms(tr2, tr3), ctx->stats.ms_total, ctx->stats.ms_split, ctx->stats.ms_model, ctx->stats.ms_scan, ctx->stats.ms_emit);
        }
        if (rc != TKZ_OK) {
            cudaStreamSynchronize(ctx->s_h2d); cudaStreamSynchronize(ctx->s_d2h);
            out->err_doc = dev.err_doc >= 0 ? (int64_t)d0 + dev.err_doc : -1;
            ctx->out_sel = 0;
            return rc;
        }
        if ((P.outputs & TKZ_OUT_OFFSETS_PACKED) && !dev.offsets_packed) {
            // this chunk has too many tokens of 256-byte-or-longer pre-tokens for the side list: the whole call delivers 32-bit
            // offsets, start again
            CK(cudaStreamSynchronize(ctx->s_h2d)); CK(cudaStreamSynchronize(ctx->s_d2h));
            P.outputs = (P.outputs & ~TKZ_OUT_OFFSETS_PACKED) | TKZ_OUT_OFFSETS;
            goto restart;
        }
        ms_kernels += ctx->stats.ms_total;
        // kernel-bound chunk (its device time exceeds what ~45 GB/s of PCIe needs for its text): larger chunks from now on
        if ((double)ctx->stats.ms_total * 1e-3 > (double)nb / 45e9 && chunk_target < chunk_max) chunk_target *= 2;
        const uint64_t T = dev.n_tokens;
        // size the host arrays from the first chunk's density of slots (rows: of rows)
        uint64_t est = T_total + T;
        if (i == 0 && nb) est = (uint64_t)((double)T * ((double)N / (double)nb) * 1.03) + 4096;
        if (est < T_total + T) est = T_total + T;
        const uint64_t R = dev.n_rows;
        if (overflow) {
            uint64_t est_rows = R_total + R + 1;
            if (i == 0 && nb) est_rows = std::max<uint64_t>(est_rows, (uint64_t)((double)R * ((double)N / (double)nb) * 1.03) + 4096);
            TRY(ensure_host_keep(ctx, ctx->h_row_tok_off, est_rows * 8, R_total * 8));
        }
        // (every chunk delivers the same arrays: they depend on the model and the parameters)
        const auto cp = result_copies(ctx, dev);
        for (uint32_t k = 0; k < N_RESULT_ARRAYS; k++) {
            host[k] = nullptr;
            if (!cp[k].dev) continue;
            TRY(ensure_host_keep(ctx, *cp[k].host, est * cp[k].elem, T_total * cp[k].elem));
            if (T) CK(cudaMemcpyAsync((uint8_t*)cp[k].host->p + T_total * cp[k].elem, cp[k].dev, T * cp[k].elem, cudaMemcpyDeviceToHost, ctx->s_d2h));
            host[k] = cp[k].host->p;
        }
        if (dev.n_wide) {
            TRY(ensure_host_keep(ctx, ctx->h_wide, (W_total + dev.n_wide) * 16, W_total * 16));
            CK(cudaMemcpyAsync((uint8_t*)ctx->h_wide.p + W_total * 16, dev.wide_tokens, dev.n_wide * 16, cudaMemcpyDeviceToHost, ctx->s_d2h));
            wide_parts.push_back({W_total, dev.n_wide, T_total});
            W_total += dev.n_wide;
        }
        // chunk-relative CSR offsets -> call-relative on the device (same stream as the copy; the chunk's kernels have finished)
        if (T_total) add_base_u64_kernel<<<(unsigned)((nd + 1 + 255) / 256), 256, 0, ctx->s_d2h>>>((unsigned long long*)dev.doc_tok_off, nd + 1, T_total);
        CK(cudaMemcpyAsync(h_dto + d0, dev.doc_tok_off, (nd + 1) * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
        if (overflow) {
            if (T_total) add_base_u64_kernel<<<(unsigned)((R + 1 + 255) / 256), 256, 0, ctx->s_d2h>>>((unsigned long long*)dev.row_tok_off, R + 1, T_total);
            if (R_total) add_base_u64_kernel<<<(unsigned)((nd + 1 + 255) / 256), 256, 0, ctx->s_d2h>>>((unsigned long long*)dev.doc_row_off, nd + 1, R_total);
            CK(cudaMemcpyAsync((uint64_t*)ctx->h_row_tok_off.p + R_total, dev.row_tok_off, (R + 1) * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
            CK(cudaMemcpyAsync(h_dro + d0, dev.doc_row_off, (nd + 1) * 8, cudaMemcpyDeviceToHost, ctx->s_d2h));
        }
        CK(cudaEventRecord(ctx->ev_d2h[b], ctx->s_d2h));
        T_total += T; T_real += dev.n_real_tokens; R_total += R;
    }
    CK(cudaStreamSynchronize(ctx->s_d2h));
    CK(cudaStreamSynchronize(ctx->s_h2d));
    h_dto[n_docs] = T_total;
    if (W_total) wide_finish((WideRec*)ctx->h_wide.p, W_total, wide_parts);
    ctx->out_sel = 0;
    ctx->stats.ms_call_kernels = ms_kernels;
    set_result(out, n_docs, T_total, T_real, h_dto, host, W_total, ctx->h_wide.p);
    if (overflow) {
        ((uint64_t*)ctx->h_row_tok_off.p)[R_total] = T_total; h_dro[n_docs] = R_total;
        out->n_rows = R_total; out->row_tok_off = (const uint64_t*)ctx->h_row_tok_off.p; out->doc_row_off = h_dro;
    }
    return TKZ_OK;
}

}  // namespace

extern "C" int tkz_encode_batch(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                                const tkz_encode_params* params, tkz_batch_result* out) {
    if (!ctx || !out || !doc_off) return TKZ_ERR_INVALID_ARG;
    if (doc_off[0] != 0) { ctx->err = "doc_off[0] must be 0"; return TKZ_ERR_INVALID_ARG; }
    const uint64_t N = doc_off[n_docs];
    if (N && !text) return TKZ_ERR_INVALID_ARG;
    ON_DEVICE(ctx);
    if (n_docs >= 2 && N > ctx->chunk_bytes + ctx->chunk_bytes / 2) return encode_host_chunked(ctx, text, doc_off, n_docs, N, params, out);
    return encode_host_single(ctx, text, doc_off, n_docs, N, params, out);
}

// ------------------------------------------------------------------------------------------------ compact result
extern "C" int tkz_encode_batch_compact(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                                        const tkz_encode_params* params, int want_offsets, tkz_compact_result* out) {
    if (!ctx || !out) return TKZ_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    out->err_doc = -1;
    tkz_encode_params P{};
    if (params) P = *params;
    out->params = P;
    if (P.hf_flags) { ctx->err = "the compact result does not carry hf_compat (template / document offsets): use tkz_encode_batch"; return TKZ_ERR_INVALID_ARG; }
    if (P.outputs & TKZ_OUT_WORD_IDS) { ctx->err = "the compact result does not carry word ids: use tkz_encode_batch"; return TKZ_ERR_INVALID_ARG; }
    // on the device: truncation only; no padding slot and no constant array is materialised or copied
    tkz_encode_params Q = P;
    Q.has_padding = 0;
    Q.outputs = TKZ_OUT_IDS | TKZ_OUT_IDS_U16 | (want_offsets ? TKZ_OUT_OFFSETS_PACKED : 0u);
    tkz_batch_result r{};
    const int rc = tkz_encode_batch(ctx, text, doc_off, n_docs, &Q, &r);
    out->err_doc = r.err_doc;
    if (rc != TKZ_OK) return rc;
    out->n_docs = r.n_docs; out->n_kept = r.n_tokens; out->n_real_tokens = r.n_real_tokens;
    out->doc_kept_off = r.doc_tok_off; out->ids = r.ids; out->ids16 = r.ids16;
    out->offsets_packed = r.offsets_packed; out->offsets = r.offsets;
    out->n_wide = r.n_wide; out->wide_tokens = r.wide_tokens;
    return TKZ_OK;
}

extern "C" uint64_t tkz_compact_slots(const tkz_compact_result* r, uint64_t d0, uint64_t d1) {
    if (!r || d1 > r->n_docs || d0 > d1) return 0;
    const tkz_encode_params& P = r->params;
    if (!P.has_padding) return r->doc_kept_off[d1] - r->doc_kept_off[d0];
    uint64_t n = 0;
    for (uint64_t d = d0; d < d1; d++) { const uint64_t k = r->doc_kept_off[d + 1] - r->doc_kept_off[d]; n += k < P.pad_length ? P.pad_length : k; }
    return n;
}

// Encoding.fromTokens (ids, type_ids 0, offsets, special_tokens_mask 0, attention_mask 1: src/encoding.zig:246-294) followed by
// Encoding.pad (pad_id / pad_type_id / (0,0) / special 1 / attention 0, left or right: src/encoding.zig:385-463)
extern "C" int tkz_compact_expand(const tkz_compact_result* r, uint64_t d0, uint64_t d1, uint64_t* doc_tok_off, uint32_t* ids, uint32_t* offsets,
                                  uint32_t* attention_mask, uint32_t* type_ids, uint32_t* special_tokens_mask) {
    if (!r || d1 > r->n_docs || d0 > d1) return TKZ_ERR_INVALID_ARG;
    const tkz_encode_params& P = r->params;
    uint64_t o = 0;
    for (uint64_t d = d0; d < d1; d++) {
        const uint64_t k0 = r->doc_kept_off[d], k = r->doc_kept_off[d + 1] - k0;
        const uint64_t olen = (P.has_padding && k < P.pad_length) ? P.pad_length : k, npad = olen - k;
        const uint64_t real0 = o + ((P.has_padding && P.pad_left) ? npad : 0), pad0 = (P.has_padding && P.pad_left) ? o : o + k;
        if (doc_tok_off) doc_tok_off[d - d0] = o;
        if (ids) {
            if (r->ids16) for (uint64_t i = 0; i < k; i++) ids[real0 + i] = r->ids16[k0 + i];
            else memcpy(ids + real0, r->ids + k0, k * 4);
            for (uint64_t i = 0; i < npad; i++) ids[pad0 + i] = P.pad_id;
        }
        if (offsets) {
            if (r->offsets_packed) {
                // 0xFFFF: the token's offsets are in the side list (sorted by kept index); the first one of the document by binary
                // search, the following ones in order
                const WideRec* wt = (const WideRec*)r->wide_tokens; uint64_t wi = r->n_wide;
                for (uint64_t i = 0; i < k; i++) {
                    const uint32_t v = r->offsets_packed[k0 + i];
                    uint32_t s0 = v & 0xFFu, e0 = v >> 8;
                    if (v == 0xFFFFu) {
                        const uint64_t slot = k0 + i;
                        if (wi == r->n_wide) {
                            uint64_t lo = 0, hi = r->n_wide;
                            while (lo < hi) { const uint64_t mid = (lo + hi) / 2; const uint64_t sv = ((uint64_t)wt[mid].hi << 32) | wt[mid].lo; if (sv < slot) lo = mid + 1; else hi = mid; }
                            wi = lo;
                        }
                        while (wi < r->n_wide && ((((uint64_t)wt[wi].hi << 32) | wt[wi].lo) < slot)) wi++;
                        if (wi >= r->n_wide || ((((uint64_t)wt[wi].hi << 32) | wt[wi].lo) != slot)) return TKZ_ERR_INVALID_ARG;
                        s0 = wt[wi].s; e0 = wt[wi].e;
                    }
                    offsets[2 * (real0 + i)] = s0; offsets[2 * (real0 + i) + 1] = e0;
                }
            }
            else if (r->offsets) memcpy(offsets + 2 * real0, r->offsets + 2 * k0, k * 8);
            else return TKZ_ERR_INVALID_ARG;
            memset(offsets + 2 * pad0, 0, npad * 8);
        }
        if (attention_mask) { for (uint64_t i = 0; i < k; i++) attention_mask[real0 + i] = 1u; memset(attention_mask + pad0, 0, npad * 4); }
        if (type_ids) { memset(type_ids + real0, 0, k * 4); for (uint64_t i = 0; i < npad; i++) type_ids[pad0 + i] = P.pad_type_id; }
        if (special_tokens_mask) { memset(special_tokens_mask + real0, 0, k * 4); for (uint64_t i = 0; i < npad; i++) special_tokens_mask[pad0 + i] = 1u; }
        o += olen;
    }
    if (doc_tok_off) doc_tok_off[d1 - d0] = o;
    return TKZ_OK;
}

// ------------------------------------------------------------------------------------------------ decode
extern "C" int tkz_decode_upload(tkz_ctx* ctx, const tkz_decode_desc* d) {
    if (!ctx || !d || (d->n_ids && (!d->tok_off || (!d->tok_bytes && d->tok_off[d->n_ids])))) return TKZ_ERR_INVALID_ARG;
    if (d->decoder_kind < 0 || d->decoder_kind > 3) { ctx->err = "unknown decoder_kind"; return TKZ_ERR_INVALID_ARG; }
    ON_DEVICE(ctx);
    const uint64_t nb = d->n_ids ? d->tok_off[d->n_ids] : 0;
    TRY(upload(ctx, ctx->t_dec_bytes, d->tok_bytes, (size_t)nb));
    std::vector<unsigned long long> off(d->n_ids + 1, 0);
    for (uint32_t i = 0; i <= d->n_ids; i++) off[i] = d->n_ids ? d->tok_off[i] : 0;
    TRY(upload(ctx, ctx->t_dec_off, off.data(), off.size() * 8));
    uint32_t max_sp = 0;
    for (uint32_t i = 0; i < d->n_special; i++) max_sp = std::max(max_sp, d->special_ids[i]);
    std::vector<uint32_t> bits(d->n_special ? (size_t)(max_sp >> 5) + 1 : 1, 0);
    for (uint32_t i = 0; i < d->n_special; i++) bits[d->special_ids[i] >> 5] |= 1u << (d->special_ids[i] & 31u);
    TRY(upload(ctx, ctx->t_dec_special, bits.data(), bits.size() * 4));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->dt = DecodeTables{(const uint8_t*)ctx->t_dec_bytes.p, (const unsigned long long*)ctx->t_dec_off.p, d->n_ids,
                           (const uint32_t*)ctx->t_dec_special.p, d->n_special ? (uint32_t)bits.size() : 0u, d->decoder_kind};
    ctx->has_decode = true;
    return TKZ_OK;
}

extern "C" int tkz_decode_batch(tkz_ctx* ctx, const uint32_t* ids, const uint64_t* seq_off, uint64_t n_seqs, int skip_special_tokens,
                                tkz_decode_result* out) {
    if (!ctx || !out || !seq_off) return TKZ_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    if (!ctx->has_decode) { ctx->err = "no decode tables uploaded"; return TKZ_ERR_INVALID_ARG; }
    if (seq_off[0] != 0) { ctx->err = "seq_off[0] must be 0"; return TKZ_ERR_INVALID_ARG; }
    const uint64_t n_tok = seq_off[n_seqs];
    if (n_tok && !ids) return TKZ_ERR_INVALID_ARG;
    if (n_tok >= 0xFFFFFFF0ull || n_seqs >= 0xFFFFFFF0ull) { ctx->err = "too many ids in one decode batch"; return TKZ_ERR_INVALID_ARG; }
    ON_DEVICE(ctx);
    cudaStream_t st = ctx->stream;
    unsigned long long* hctrl = (unsigned long long*)ctx->h_ctrl.p;
    const DecodeTables& t = ctx->dt;
    TRY(ensure(ctx, ctx->a_dec_ids, n_tok * 4));
    TRY(ensure(ctx, ctx->a_dec_seq_off, (n_seqs + 1) * 8));
    TRY(ensure(ctx, ctx->a_dec_len, (n_tok + 2) * 4));
    TRY(ensure(ctx, ctx->a_dec_olen, (n_seqs + 2) * 4));
    TRY(ensure(ctx, ctx->a_dec_boff, (n_seqs + 2) * 8));
    TRY(ensure(ctx, ctx->a_scan_tmp, (scan_tmp_elems(n_tok) + scan_tmp_elems(n_seqs)) * 8));
    if (n_tok) CK(cudaMemcpyAsync(ctx->a_dec_ids.p, ids, n_tok * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->a_dec_seq_off.p, seq_off, (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
    uint32_t* tok_len = (uint32_t*)ctx->a_dec_len.p;
    const uint32_t* d_ids = (const uint32_t*)ctx->a_dec_ids.p;
    const unsigned long long* d_seq = (const unsigned long long*)ctx->a_dec_seq_off.p;
    unsigned long long* ctrl = (unsigned long long*)ctx->a_ctrl.p;
    ctrl_reset_kernel<<<1, 1, 0, st>>>(ctrl);
    if (n_tok) dec_len_kernel<<<(unsigned)((n_tok + 255) / 256), 256, 0, st>>>(t, d_ids, n_tok, skip_special_tokens, tok_len, ctrl + 1);
    TRY(readback(ctx, hctrl + 42, ctrl + 1, 8));
    CK(cudaStreamSynchronize(st));
    // token byte offsets are u32: a batch that decodes to 4 GiB or more (the round trip of a 4 GiB encode) must be split
    if (hctrl[42] >= 0xFFFFF000ull) { ctx->err = "decoded batch must be < 4 GiB (u32 byte offsets): split the batch"; return TKZ_ERR_INVALID_ARG; }
    exclusive_scan<uint32_t>(tok_len, n_tok, tok_len, (unsigned long long*)ctx->a_scan_tmp.p, st);      // tok_len[n_tok] = raw bytes
    TRY(readback(ctx, hctrl + 40, tok_len + n_tok, 4));
    CK(cudaStreamSynchronize(st));
    const uint64_t raw_bytes = (uint32_t)hctrl[40];
    TRY(ensure(ctx, ctx->a_dec_raw, raw_bytes));
    uint8_t* raw = (uint8_t*)ctx->a_dec_raw.p;
    if (n_tok) dec_gather_kernel<<<(unsigned)((n_tok + 255) / 256), 256, 0, st>>>(t, d_ids, n_tok, tok_len, raw);
    unsigned long long* byte_off = (unsigned long long*)ctx->a_dec_boff.p;
    const uint8_t* d_bytes = raw;
    uint64_t out_bytes = raw_bytes;
    const unsigned seq_blocks = (unsigned)((n_seqs + 1 + 255) / 256), warp_blocks = (unsigned)((n_seqs * 32 + 255) / 256);
    if (t.decoder_kind == 1 || t.decoder_kind == 3) {
        uint32_t* olen = (uint32_t*)ctx->a_dec_olen.p;
        if (n_seqs) {
            if (t.decoder_kind == 1) dec_filter_kernel<1, false><<<warp_blocks, 256, 0, st>>>(raw, d_seq, tok_len, n_seqs, olen, nullptr, nullptr);
            else dec_filter_kernel<3, false><<<warp_blocks, 256, 0, st>>>(raw, d_seq, tok_len, n_seqs, olen, nullptr, nullptr);
        }
        exclusive_scan<uint32_t>(olen, n_seqs, olen, (unsigned long long*)ctx->a_scan_tmp.p, st);
        TRY(readback(ctx, hctrl + 41, olen + n_seqs, 4));
        CK(cudaStreamSynchronize(st));
        out_bytes = (uint32_t)hctrl[41];
        TRY(ensure(ctx, ctx->a_dec_out, out_bytes));
        uint8_t* ob = (uint8_t*)ctx->a_dec_out.p;
        if (n_seqs) {
            if (t.decoder_kind == 1) dec_filter_kernel<1, true><<<warp_blocks, 256, 0, st>>>(raw, d_seq, tok_len, n_seqs, nullptr, olen, ob);
            else dec_filter_kernel<3, true><<<warp_blocks, 256, 0, st>>>(raw, d_seq, tok_len, n_seqs, nullptr, olen, ob);
        }
        dec_widen_kernel<<<seq_blocks, 256, 0, st>>>(olen, n_seqs + 1, byte_off);
        d_bytes = ob;
    } else {
        dec_seq_off_kernel<<<seq_blocks, 256, 0, st>>>(d_seq, n_seqs, tok_len, byte_off);
    }
    CK(cudaGetLastError());
    TRY(ensure_host(ctx, ctx->h_dec_bytes, out_bytes));
    TRY(ensure_host(ctx, ctx->h_dec_off, (n_seqs + 1) * 8));
    if (out_bytes) CK(cudaMemcpyAsync(ctx->h_dec_bytes.p, d_bytes, out_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ctx->h_dec_off.p, byte_off, (n_seqs + 1) * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    out->n_seqs = n_seqs; out->n_bytes = out_bytes;
    out->byte_off = (const uint64_t*)ctx->h_dec_off.p; out->bytes = (const uint8_t*)ctx->h_dec_bytes.p;
    return TKZ_OK;
}
