// tkz_overflow.cuh -- overflowing windows (TKZ_HF_OVERFLOW): Hugging Face Encoding::truncate(max_length, stride, Right) keeps every
// window of a long document as an encoding of its own, each with the template and its own padding.
//
// Runs after one of the two pipelines has encoded the batch untruncated, unpadded and without template tokens into a staging
// output set (CSR over documents, real tokens only).  With L = max_length - template tokens and step = L - stride, a document of
// n tokens has rows(n) = 1 for n <= L, else 1 + ceil((n - L) / step); row k covers tokens [k * step, min(k * step + L, n)).
//   ovf_doc_rows_kernel   rows per document                                  -> scan -> doc_row_off
//   ovf_row_len_kernel    each row's document, window length and slot count  -> scan -> row_tok_off
//   ovf_copy_kernel       one warp per row: the window from staging into its slots, with the constants of a real token (the
//                         template's sequence type id only in a document's first row, as tokenizers does)
//   ovf_doc_off_kernel    doc_tok_off[d] = row_tok_off[doc_row_off[d]]
// The template's special tokens and the padding are the shared epilogue's (pad_prologue / pad_epilogue), rows standing in for
// documents.
#pragma once
#include "tkz_emit.cuh"

namespace tkz {

__device__ __forceinline__ unsigned long long ovf_rows(unsigned long long n, unsigned long long L, unsigned long long step) {
    return n <= L ? 1ull : 1ull + (n - L + step - 1) / step;
}

// per document: its row count to doc_rows[d]; the real tokens of all rows (n + (rows - 1) * stride) summed into *rows_real
__global__ void __launch_bounds__(256) ovf_doc_rows_kernel(const unsigned long long* __restrict__ stage_off, uint32_t n_docs, unsigned long long L,
                                                           unsigned long long step, unsigned long long* __restrict__ doc_rows,
                                                           unsigned long long* rows_real) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long real = 0;
    if (d < n_docs) {
        const unsigned long long n = stage_off[d + 1] - stage_off[d], r = ovf_rows(n, L, step);
        doc_rows[d] = r;
        real = n + (r - 1) * (L - step);
    }
    for (int k = 16; k > 0; k >>= 1) real += __shfl_xor_sync(0xFFFFFFFFu, real, k);
    if (lane_id() == 0 && real) atomicAdd(rows_real, real);
}

// per row: its document (doc_row_off strictly increases: every document has a row), window length and slot count
__global__ void __launch_bounds__(256) ovf_row_len_kernel(EmitParams p, const unsigned long long* __restrict__ stage_off,
                                                          const unsigned long long* __restrict__ doc_row_off, uint32_t n_docs, uint32_t n_rows,
                                                          unsigned long long L, unsigned long long step, unsigned long long* __restrict__ row_len,
                                                          uint32_t* __restrict__ row_real, uint32_t* __restrict__ row_doc) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    uint32_t lo = 0, hi = n_docs - 1;                     // last d with doc_row_off[d] <= r
    while (lo < hi) { const uint32_t mid = lo + (hi - lo + 1) / 2; if (doc_row_off[mid] <= r) lo = mid; else hi = mid - 1; }
    const unsigned long long n = stage_off[lo + 1] - stage_off[lo], start = (r - doc_row_off[lo]) * step;
    const unsigned long long len = n - start < L ? n - start : L;
    row_real[r] = (uint32_t)len;
    row_doc[r] = lo;
    unsigned long long kept;
    row_len[r] = doc_out_len(p, len, &kept);              // (len <= L: nothing is cut)
}

// the staging arrays (real tokens of every document back to back; offsets / word ids only when the call delivers them)
struct OvfStage { const uint32_t* ids; const uint16_t* ids16; const uint2* offsets; const uint32_t* word_ids; };

// one warp per row: lane-strided, so loads from staging and stores to the row are coalesced.  WID: word ids
template <bool WID>
__global__ void __launch_bounds__(256) ovf_copy_kernel(EmitParams p, EmitOut o, OvfStage s, uint32_t n_rows, unsigned long long step,
                                                       const unsigned long long* __restrict__ stage_off,
                                                       const unsigned long long* __restrict__ doc_row_off,
                                                       const unsigned long long* __restrict__ row_tok_off,
                                                       const uint32_t* __restrict__ row_real, const uint32_t* __restrict__ row_doc) {
    const uint32_t r = (uint32_t)(((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (r >= n_rows) return;
    const uint32_t d = row_doc[r], len = row_real[r];
    const unsigned long long k = r - doc_row_off[d], src = stage_off[d] + k * step;
    // (tokenizers gives the template's sequence type id to the tokens of the first row only; overflowing rows keep type id 0)
    EmitParams q = p;
    if (k) q.seq_type = 0;
    const unsigned long long added = tpl_added(p);
    const unsigned long long dst = row_tok_off[r] + ((p.has_pad && p.pad_left) ? row_tok_off[r + 1] - row_tok_off[r] - len - added : 0) +
                                   ((p.hf_flags & 1u) ? p.n_pre : 0u);
    for (uint32_t i = lane_id(); i < len; i += 32) {
        const uint32_t id = (p.outputs & 64u) ? (uint32_t)s.ids16[src + i] : s.ids[src + i];
        const uint2 of = (p.outputs & 2u) ? s.offsets[src + i] : make_uint2(0u, 0u);
        emit_real<WID>(q, o, dst + i, id, of.x, of.y, WID ? s.word_ids[src + i] : 0u);
    }
}

// documents' slot offsets from their first rows (d = 0 .. n_docs: doc_row_off[n_docs] is the row count, row_tok_off of it the slots)
__global__ void ovf_doc_off_kernel(const unsigned long long* __restrict__ doc_row_off, const unsigned long long* __restrict__ row_tok_off, uint32_t n_docs,
                                   unsigned long long* __restrict__ doc_tok_off) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d <= n_docs) doc_tok_off[d] = row_tok_off[doc_row_off[d]];
}

}  // namespace tkz
