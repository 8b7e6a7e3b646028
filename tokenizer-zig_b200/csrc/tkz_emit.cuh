// tkz_emit.cuh -- K5: Encoding.fromTokens + truncate + pad fused into the output write.
//
// Replaces Encoding.fromTokens (src/encoding.zig:246-294: ids, type_ids = 0, offsets, special_token_mask = 0,
// attention_mask = 1), Encoding.truncate (src/encoding.zig:363-380: keep the first max_length, stride ignored) and
// Encoding.pad (src/encoding.zig:385-463: right / left fill with pad_id, pad_type_id, offset (0,0), special 1,
// attention 0; no-op when already long enough).  Post-processing inserts nothing (src/config.zig:551-555).
// Output is CSR over documents: slots of document d = [doc_tok_off[d], doc_tok_off[d+1]).
#pragma once
#include "tkz_common.cuh"

namespace tkz {

struct EmitParams {
    int has_trunc; unsigned long long max_length;
    int has_pad; unsigned long long pad_length;
    uint32_t pad_id, pad_type_id; int pad_left;
    uint32_t outputs;
    // hf_compat (tkz_encode_params.hf_flags; 0 = the reference): single-sequence template -- what processor.zig:41-152 declares
    // and leaves as TODO -- and offsets relative to the document.  Both device pipelines serve it.
    uint32_t hf_flags;
    uint32_t n_pre, n_suf, pre_id[4], pre_type[4], suf_id[4], suf_type[4], seq_type;
};
__device__ __forceinline__ uint32_t tpl_added(const EmitParams& p) { return (p.hf_flags & 1u) ? p.n_pre + p.n_suf : 0u; }

// slots a document occupies after truncate + pad
// (*kept = real tokens kept; with a template the added tokens count against max_length, as tokenizers' post_process does,
// and towards the padded length)
__device__ __forceinline__ unsigned long long doc_out_len(const EmitParams& p, unsigned long long t, unsigned long long* kept) {
    unsigned long long k = t;
    const unsigned long long add = tpl_added(p);
    if (p.has_trunc) { const unsigned long long budget = p.max_length > add ? p.max_length - add : 0; if (k > budget) k = budget; }
    *kept = k;
    return (p.has_pad && k + add < p.pad_length) ? p.pad_length : k + add;
}

// per document: real token count -> output slot count; the real count also to doc_real when the padding / template
// kernels need it (doc_real != nullptr)
__global__ void doc_len_kernel(EmitParams p, const uint32_t* __restrict__ word_tok_off, const uint32_t* __restrict__ doc_word_off, uint32_t n_docs,
                               unsigned long long* __restrict__ doc_len, uint32_t* __restrict__ doc_real) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_docs) return;
    const unsigned long long t = word_tok_off[doc_word_off[d + 1]] - word_tok_off[doc_word_off[d]];
    if (doc_real) doc_real[d] = (uint32_t)t;
    unsigned long long kept;
    doc_len[d] = doc_out_len(p, t, &kept);
}

struct EmitOut { uint32_t* ids; uint32_t* offsets; uint32_t* attention; uint32_t* type_ids; uint32_t* special;
                 uint16_t* offsets16;        // one u16 per token (start | end << 8), only when every pre-token is < 256 bytes
                 uint16_t* ids16;            // ids as u16 instead of `ids` (outputs & 64: every id of the vocabulary is < 65536)
                 uint4* spans;               // SpanToken records (token.zig:19-33): {id, start, end, type_id | flags << 8} (outputs & 128)
                 uint4* wide; unsigned int* wide_count; uint32_t wide_cap;   // offsets16: tokens that do not fit a byte pair {slot lo, hi, start, end}
                 uint32_t* word_ids; };      // outputs & 256: the token's pre-token index in its document, TKZ_NONE for specials / padding

// words with more than EMIT_BIG tokens (whole documents, MiB-long unbroken words) are not copied by one warp: they are
// queued here and copied by the whole grid (emit_big_kernel)
constexpr uint32_t EMIT_BIG = 2048;
// item = {src pool position, token count, dst lo, dst hi}; shift[] = offset base (hf_compat); wid[] = word id (WID forms)
struct BigList { uint4* items; unsigned int* count; uint32_t cap; uint32_t* shift; uint32_t* wid; };
template <bool WID = false>
__device__ __forceinline__ bool big_push(const BigList& b, uint32_t src, uint32_t cnt, unsigned long long dst, uint32_t shift = 0, uint32_t wid = 0) {
    const uint32_t i = atomicAdd(b.count, 1u);
    if (i >= b.cap) return false;
    b.items[i] = make_uint4(src, cnt, (uint32_t)dst, (uint32_t)(dst >> 32));
    if (b.shift) b.shift[i] = shift;
    if (WID) b.wid[i] = wid;
    return true;
}

__device__ __forceinline__ void emit_id(const EmitParams& p, const EmitOut& o, unsigned long long dst, uint32_t id) {
    if (p.outputs & 64u) o.ids16[dst] = (uint16_t)id; else o.ids[dst] = id;
}
// WID: the call asked for word ids (TKZ_OUT_WORD_IDS), wid = the token's; a compile-time switch, so that the kernels of the
// calls without them stay as they are
template <bool WID = false>
__device__ __forceinline__ void emit_real(const EmitParams& p, const EmitOut& o, unsigned long long dst, uint32_t id, uint32_t s, uint32_t e, uint32_t wid = 0) {
    emit_id(p, o, dst, id);
    if (WID) o.word_ids[dst] = wid;
    if (p.outputs & 2u) reinterpret_cast<uint2*>(o.offsets)[dst] = make_uint2(s, e);
    if (p.outputs & 32u) {
        // one u16 per token; a token of a long pre-token that does not fit goes to the side list (sized for all of them)
        if (e < 256u && (s | (e << 8)) != 0xFFFFu) o.offsets16[dst] = (uint16_t)(s | (e << 8));
        else {
            o.offsets16[dst] = 0xFFFFu;
            const uint32_t k = atomicAdd(o.wide_count, 1u);
            if (k < o.wide_cap) o.wide[k] = make_uint4((uint32_t)dst, (uint32_t)(dst >> 32), s, e);
        }
    }
    if (p.outputs & 4u) o.attention[dst] = 1u;
    const uint32_t ty = (p.hf_flags & 1u) ? p.seq_type : 0u;
    if (p.outputs & 8u) o.type_ids[dst] = ty;
    if (p.outputs & 16u) o.special[dst] = 0u;
    if (p.outputs & 128u) o.spans[dst] = make_uint4(id, s, e, ty & 0xFFu);
}
// a special token of the template: offsets (0, 0), special 1, attention 1 (SpanToken.initSpecial: flags.is_special, bit 0); no word
template <bool WID = false>
__device__ __forceinline__ void emit_special(const EmitParams& p, const EmitOut& o, unsigned long long dst, uint32_t id, uint32_t ty) {
    emit_id(p, o, dst, id);
    if (p.outputs & 2u) reinterpret_cast<uint2*>(o.offsets)[dst] = make_uint2(0u, 0u);
    if (p.outputs & 32u) o.offsets16[dst] = 0;
    if (p.outputs & 4u) o.attention[dst] = 1u;
    if (p.outputs & 8u) o.type_ids[dst] = ty;
    if (p.outputs & 16u) o.special[dst] = 1u;
    if (p.outputs & 128u) o.spans[dst] = make_uint4(id, 0u, 0u, (ty & 0xFFu) | 0x0100u);
    if (WID) o.word_ids[dst] = TKZ_NONE;
}

// one lane per word; words with many tokens are copied by the whole warp.  WID: word ids (word w is pre-token
// w - doc_word_off[d] of its document d)
template <bool WID>
__global__ void __launch_bounds__(256) emit_words_kernel(EmitParams p, EmitOut o, uint32_t n_words,
                                                         const uint32_t* __restrict__ word_start, const uint32_t* __restrict__ word_doc,
                                                         const uint32_t* __restrict__ word_tok_off, const uint32_t* __restrict__ doc_word_off,
                                                         const unsigned long long* __restrict__ doc_tok_off,
                                                         const uint32_t* __restrict__ pool_id, const uint32_t* __restrict__ pool_s,
                                                         const uint32_t* __restrict__ pool_e, BigList bl, const uint64_t* __restrict__ doc_off) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = lane_id();
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cnt = 0, src = 0, sh = 0, wid = 0; unsigned long long dst = 0; unsigned long long room = 0;
    if (w < n_words) {
        const uint32_t t0 = word_tok_off[w];
        cnt = word_tok_off[w + 1] - t0;
        if (cnt) {
            const uint32_t d = word_doc[w];
            const unsigned long long doc_t0 = word_tok_off[doc_word_off[d]];
            const unsigned long long doc_t = (unsigned long long)word_tok_off[doc_word_off[d + 1]] - doc_t0;
            unsigned long long kept;
            const unsigned long long olen = doc_out_len(p, doc_t, &kept);
            const unsigned long long j0 = (unsigned long long)t0 - doc_t0;          // index of the word's first token in its document
            room = j0 < kept ? kept - j0 : 0;                                       // truncation: tokens j >= kept are dropped
            const unsigned long long shift = ((p.has_pad && p.pad_left) ? olen - kept - tpl_added(p) : 0) + ((p.hf_flags & 1u) ? p.n_pre : 0u);
            dst = doc_tok_off[d] + shift + j0;
            src = word_start[w];
            if (p.hf_flags & 2u) sh = src - (uint32_t)doc_off[d];                   // pre-token start within its document
            if (WID) wid = w - doc_word_off[d];
            if ((unsigned long long)cnt > room) cnt = (uint32_t)room;
        }
    }
    // short words: each lane copies its own tokens
    if (cnt > 0 && cnt <= 4) {
        for (uint32_t k = 0; k < cnt; k++) emit_real<WID>(p, o, dst + k, pool_id[src + k], pool_s[src + k] + sh, pool_e[src + k] + sh, wid);
    }
    // very long words: queued for the grid-wide copy
    if (cnt > EMIT_BIG && big_push<WID>(bl, src, cnt, dst, sh, wid)) cnt = 0;
    // long words: warp-cooperative copy
    uint32_t big = __ballot_sync(FULL, cnt > 4);
    while (big) {
        const int l = __ffs(big) - 1; big &= big - 1;
        const uint32_t c = __shfl_sync(FULL, cnt, l), s = __shfl_sync(FULL, src, l), hs = __shfl_sync(FULL, sh, l);
        const uint32_t wi = WID ? __shfl_sync(FULL, wid, l) : 0u;
        const unsigned long long dd = __shfl_sync(FULL, dst, l);
        for (uint32_t k = lane; k < c; k += 32) emit_real<WID>(p, o, dd + k, pool_id[s + k], pool_s[s + k] + hs, pool_e[s + k] + hs, wi);
    }
}

// grid-wide copy of the queued big words: every block takes a strided share of every item
template <bool WID>
__global__ void __launch_bounds__(256) emit_big_kernel(EmitParams p, EmitOut o, BigList bl, const uint32_t* __restrict__ pool_id,
                                                       const uint32_t* __restrict__ pool_s, const uint32_t* __restrict__ pool_e) {
    uint32_t n = *bl.count; if (n > bl.cap) n = bl.cap;
    for (uint32_t k = 0; k < n; k++) {
        const uint4 it = bl.items[k];
        const uint32_t sh = bl.shift ? bl.shift[k] : 0u;
        const uint32_t wid = WID ? bl.wid[k] : 0u;
        const unsigned long long dst = (unsigned long long)it.z | ((unsigned long long)it.w << 32);
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < it.y; i += gridDim.x * blockDim.x)
            emit_real<WID>(p, o, dst + i, pool_id[it.x + i], pool_s[it.x + i] + sh, pool_e[it.x + i] + sh, wid);
    }
}

// whole-array fill with one 16-byte pattern (grid-stride 16-byte stores; the last partial 16 bytes in 2-byte steps by one
// thread).  When most slots of a batch are padding (BERT-style pad to 512 around ~30 tokens), filling the arrays with the
// padding values at streaming-store speed BEFORE the real tokens are written beats one warp per document writing the gaps.
__global__ void __launch_bounds__(256) fill16_kernel(uint4* __restrict__ p, unsigned long long nbytes, uint4 v) {
    const unsigned long long n16 = nbytes >> 4;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) __stcs(p + i, v);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const uint16_t h[8] = {(uint16_t)v.x, (uint16_t)(v.x >> 16), (uint16_t)v.y, (uint16_t)(v.y >> 16), (uint16_t)v.z, (uint16_t)(v.z >> 16), (uint16_t)v.w, (uint16_t)(v.w >> 16)};
        uint16_t* q = reinterpret_cast<uint16_t*>(p + n16);
        for (uint32_t k = 0; k < (uint32_t)((nbytes & 15ull) >> 1); k++) q[k] = h[k];
    }
}

}  // namespace tkz
