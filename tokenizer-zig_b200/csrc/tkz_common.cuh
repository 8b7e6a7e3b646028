// tkz_common.cuh -- shared definitions of the B200 batch encoder (host table builders + device lookups).
//
// Data layout in HBM (see DESIGN.md):
//   text            u8[N]          all documents back to back (caller's buffer, read-only)
//   doc_off         u64[n_docs+1]
//   word_start/end  u32[W]         pre-token spans (absolute byte positions), text order
//   word_doc        u32[W]         owning document
//   doc_word_off    u32[n_docs+1]  first word of each document
//   pool_*          u32[N]         per-word scratch AND token pool, indexed by the word's byte position: a pre-token of
//                                  L bytes yields at most L symbols/tokens, so word w owns pool[word_start[w] .. +L)
//                                  (the device-arena replacement of src/arena.zig's per-thread symbol/heap buffers)
//   word_ntok       u32[W]         tokens produced per word;  word_tok_off u32[W+1] its exclusive scan
//   out arrays                     CSR encoding (ids, offsets, masks), see include/tokzig_b200.h
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define TKZ_NONE 0xFFFFFFFFu        // "no rank" / "no id"
#define TKZ_DIRTY 0xFFFFFFFEu       // cached pair rank must be looked up again

namespace tkz {

// ------------------------------------------------------------------ merge table  (std.AutoHashMap(u64, PairVal), bpe.zig:40)
struct MergeEnt { uint32_t first, second, rank, new_id; };   // rank == TKZ_NONE: empty slot

__host__ __device__ __forceinline__ uint32_t pair_hash32(uint32_t a, uint32_t b) {
    uint32_t h = (a * 0x9E3779B1u) ^ ((b + 0x7F4A7C15u) * 0x85EBCA77u);
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12;
    return h;
}

// ------------------------------------------------------------------ single-codepoint table (BPE initial symbols, bpe.zig:185-211)
// key = the 2..4 bytes of the UTF-8 sequence packed little endian (never 0); ASCII goes through a direct 128-entry table
struct CharEnt { uint32_t key, id; };                         // key == 0: empty
__host__ __device__ __forceinline__ uint32_t char_hash32(uint32_t k) {
    k ^= k >> 16; k *= 0x7FEB352Du; k ^= k >> 15; k *= 0x846CA68Bu; k ^= k >> 16;
    return k;
}
// std.unicode.utf8ByteSequenceLength; 0 = invalid lead byte
__host__ __device__ __forceinline__ int utf8_seq_len(uint32_t b) {
    if (b < 0x80) return 1;
    if ((b & 0xE0) == 0xC0) return 2;
    if ((b & 0xF0) == 0xE0) return 3;
    if ((b & 0xF8) == 0xF0) return 4;
    return 0;
}

// ------------------------------------------------------------------ WordPiece vocabulary (StringHashMap(u32), wordpiece.zig:15)
// FNV-1a 64 over the candidate bytes (prefix bytes first for continuation pieces); exact match is verified on bytes.
struct WpEnt { uint64_t hash; uint32_t id, str_off, len, used; };   // 24 B
#define TKZ_FNV_OFFSET 0xCBF29CE484222325ULL
#define TKZ_FNV_PRIME 0x100000001B3ULL
__host__ __device__ __forceinline__ uint64_t fnv1a_step(uint64_t h, uint32_t byte) { return (h ^ (uint64_t)byte) * TKZ_FNV_PRIME; }
__host__ __device__ __forceinline__ uint32_t wp_slot(uint64_t h) { return (uint32_t)(h ^ (h >> 29) ^ (h >> 47)); }

#define TKZ_MAX_PREFIX 64           // continuing_subword_prefix longer than this is rejected at upload

// ------------------------------------------------------------------ device-side model (passed by value to kernels)
struct DevModel {
    int kind;
    int has_pretok;                  // class_lut given
    int norm_identity;               // no byte changes
    int norm_has_drop;               // the normalizer removes bytes -> compaction pass first
    const uint8_t* lut;              // device: [0..256) normalised byte, [256..512) class of the RAW byte (class_lut[norm[b]])
    // BPE
    const uint32_t* char_ascii;      // [128] id or TKZ_NONE
    const CharEnt* char_tab; uint32_t char_mask;
    const MergeEnt* merges; uint32_t merge_mask; uint32_t n_merges;
    // windowed schedule (tkz_bpe_block.cuh): per merge-table slot, how far a competing merge can reach: low byte = WL of the
    // pair's first symbol, high byte = WR of its second symbol; valid only when windowed_ok (table proven "proper" at upload)
    const uint16_t* merge_win; int windowed_ok;
    int has_unk; uint32_t unk_id;
    // WordPiece
    const WpEnt* wp_tab; uint32_t wp_mask;
    const uint8_t* wp_pool;
    uint32_t prefix_len; uint64_t prefix_state;      // FNV state after the prefix bytes
    uint8_t prefix[TKZ_MAX_PREFIX];
    uint32_t max_key_first;          // longest vocab key (bytes): longest candidate worth testing at start == 0
    uint32_t max_key_cont;           // longest (key minus prefix) among keys that begin with the prefix
    uint64_t max_chars;
};

// error word: (word index or byte position of the failing word) << 8 | code, so that atomicMin keeps the first failing word in
// text order; 0xFF.. = none
#define TKZ_ERRW_NONE 0xFFFFFFFFFFFFFFFFULL
#define TKZ_ECODE_UTF8 3
#define TKZ_ECODE_UNK 2

__device__ __forceinline__ void report_error(unsigned long long* errw, uint32_t word, uint32_t code) {
    atomicMin(errw, ((unsigned long long)word << 8) | code);
}

// ------------------------------------------------------------------ device lookups
__device__ __forceinline__ uint32_t merge_rank_lookup(const DevModel& m, uint32_t a, uint32_t b, uint32_t* new_id) {
    if (m.n_merges == 0) return TKZ_NONE;
    uint32_t slot = pair_hash32(a, b) & m.merge_mask;
    for (;;) {
        const uint4 e = __ldg(reinterpret_cast<const uint4*>(m.merges) + slot);
        if (e.z == TKZ_NONE) return TKZ_NONE;
        if (e.x == a && e.y == b) { if (new_id) *new_id = e.w; return e.z; }
        slot = (slot + 1) & m.merge_mask;
    }
}
// rank + new id + window of the pair (a, b); TKZ_NONE when the pair has no merge
__device__ __forceinline__ uint32_t merge_lookup_win(const DevModel& m, uint32_t a, uint32_t b, uint32_t* new_id, uint32_t* win) {
    if (m.n_merges == 0) return TKZ_NONE;
    uint32_t slot = pair_hash32(a, b) & m.merge_mask;
    for (;;) {
        const uint4 e = __ldg(reinterpret_cast<const uint4*>(m.merges) + slot);
        if (e.z == TKZ_NONE) return TKZ_NONE;
        if (e.x == a && e.y == b) { *new_id = e.w; *win = __ldg(m.merge_win + slot); return e.z; }
        slot = (slot + 1) & m.merge_mask;
    }
}
__device__ __forceinline__ uint32_t char_lookup(const DevModel& m, uint32_t key, int len) {
    if (len == 1) return __ldg(m.char_ascii + (key & 0x7F));
    uint32_t slot = char_hash32(key) & m.char_mask;
    for (;;) {
        const uint2 e = __ldg(reinterpret_cast<const uint2*>(m.char_tab) + slot);
        if (e.x == 0) return TKZ_NONE;
        if (e.x == key) return e.y;
        slot = (slot + 1) & m.char_mask;
    }
}

// ------------------------------------------------------------------ warp / block primitives
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
    const uint32_t lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= (uint32_t)d) v += t; }
    return v;
}
__device__ __forceinline__ unsigned long long warp_incl_scan64(unsigned long long v) {
    const uint32_t lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= (uint32_t)d) v += t; }
    return v;
}
__device__ __forceinline__ unsigned long long warp_min64(unsigned long long v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { unsigned long long t = __shfl_xor_sync(0xFFFFFFFFu, v, d); v = t < v ? t : v; }
    return v;
}
// exclusive scan over a block of `NW` warps; `sh` = NW+1 u64 slots; returns exclusive prefix, *total = block sum
template <int NW>
__device__ __forceinline__ unsigned long long block_excl_scan64(unsigned long long v, unsigned long long* sh, unsigned long long* total) {
    const uint32_t lane = lane_id(), wid = threadIdx.x >> 5;
    unsigned long long inc = warp_incl_scan64(v);
    if (lane == 31) sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned long long x = lane < NW ? sh[lane] : 0ULL;
        unsigned long long xi = warp_incl_scan64(x);
        if (lane < NW) sh[lane] = xi - x;
        if (lane == 31) sh[NW] = xi;
    }
    __syncthreads();
    unsigned long long r = sh[wid] + inc - v;
    *total = sh[NW];
    __syncthreads();
    return r;
}

// 32-bit block exclusive scan with ONE barrier per call: `sh` holds 2 * (NW + 1) u32 and is double-buffered on `phase`
// (callers alternate phase 0/1 between consecutive calls), every thread sums the warp totals below its own warp itself.
template <int NW>
__device__ __forceinline__ uint32_t block_excl_scan32(uint32_t v, uint32_t* sh, uint32_t phase, uint32_t* total) {
    const uint32_t lane = lane_id(), wid = threadIdx.x >> 5;
    uint32_t* s = sh + (phase & 1u) * (NW + 1);
    const uint32_t inc = warp_incl_scan(v);
    if (lane == 31) s[wid] = inc;
    __syncthreads();
    // every warp scans the NW warp totals with shuffles (one shared-memory read per lane)
    static_assert(NW <= 32, "one lane per warp total");
    const uint32_t x = lane < NW ? s[lane] : 0u;
    uint32_t xi = x;
#pragma unroll
    for (int d = 1; d < NW; d <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, xi, d); if (lane >= (uint32_t)d) xi += y; }
    *total = __shfl_sync(0xFFFFFFFFu, xi, NW - 1);
    const uint32_t base = __shfl_sync(0xFFFFFFFFu, xi - x, wid);
    return base + inc - v;
}

// the same for one-bit values: ballot + popc instead of five shuffle steps; a one-warp block needs neither shared memory
// nor the barrier
template <int NW>
__device__ __forceinline__ uint32_t block_excl_scan_bit(bool v, uint32_t* sh, uint32_t phase, uint32_t* total) {
    const uint32_t lane = lane_id(), wid = threadIdx.x >> 5;
    const uint32_t mk = __ballot_sync(0xFFFFFFFFu, v);
    const uint32_t ex = (uint32_t)__popc(mk & ((1u << lane) - 1u));
    if (NW == 1) { *total = (uint32_t)__popc(mk); __syncwarp(); return ex; }
    uint32_t* s = sh + (phase & 1u) * (NW + 1);
    if (lane == 0) s[wid] = (uint32_t)__popc(mk);
    __syncthreads();
    static_assert(NW <= 32, "one lane per warp total");
    const uint32_t x = lane < NW ? s[lane] : 0u;
    uint32_t xi = x;
#pragma unroll
    for (int d = 1; d < NW; d <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, xi, d); if (lane >= (uint32_t)d) xi += y; }
    *total = __shfl_sync(0xFFFFFFFFu, xi, NW - 1);
    const uint32_t base = __shfl_sync(0xFFFFFFFFu, xi - x, wid);
    return base + ex;
}

}  // namespace tkz
