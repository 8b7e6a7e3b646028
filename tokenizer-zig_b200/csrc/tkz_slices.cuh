// tkz_slices.cuh -- the slice pipeline: Tokenizer.encode (src/lib.zig:109-160) for a batch in TWO passes over 1 KiB text
// slices, one WARP per slice (no block-level barrier anywhere; a block only shares the byte LUT).
//
//   pass A  slice_words_kernel  normalise (config.zig:364-379) + pre-tokenize (config.zig:405-450, pretokenizer.zig:49-241)
//                               + model per pre-token (bpe.zig:173-263 / wordpiece.zig:141-222):
//           0  the slice (+ 16 bytes before, 48 behind) arrives in shared memory by ONE bulk copy (cp.async.bulk +
//              mbarrier, double-buffered per warp: slice i+1 is in flight while slice i is processed)
//           1  byte classes: 4 bytes per instruction (range compares on packed bytes, class sets given as byte ranges at
//              upload) or, for arbitrary tables, a per-byte look-up; the byte map is applied in place
//           2  word-start masks (neighbour bits by shuffle), prefix over lanes, list of the words that START in the slice
//           3  32 words per round, one per lane: 128-bit key from shared memory, ONE 32-byte probe of the per-batch word
//              table in L2 returns key + tokens (words of one or two tokens carry them in the slot).  First sight of a
//              word: atom.cas.b128 claims the slot, the claiming warp runs the model on it right there (warp-cooperative,
//              symbols in shared memory) and publishes the value; a word whose owner is still computing is polled after
//              the warp has published its own words (owners never wait, so polling cannot deadlock).  Words of 16..31
//              bytes go the same way through 64-byte slots.  Result: the TOKENS of the slice's words, in text order, in
//              a compact per-slice run of the token stream (one record per token, TW_REC_*: 4 bytes = id u16 + offsets
//              u8,u8 when every id of the model fits 16 bits, else id u32 + offsets; ids only: u16 or u32), the token
//              count of the slice and the token prefix at every document start.
//   [word-list kernels on the few pre-tokens longer than TW_MAX_INLINE bytes (tkz_bpe.cuh / tkz_bpe_block.cuh /
//    tkz_wordpiece.cuh), long_fix_kernel adds their token counts]
//   scan over slices
//   pass B  slice_emit_kernel   Encoding.fromTokens + truncate + pad (encoding.zig:246-294, 363-463): a streaming copy of
//                               the token stream to its final position, widened to the arrays the call asked for
//
// Exact because the model is a pure function of the normalised pre-token bytes and the reference's offsets are pre-token
// relative (lib.zig:133-137 never adds the pre-token start): every occurrence of a word gets identical records.  The table
// key is the word itself (<= 15 bytes + length compared as 128 bits, 16..31 bytes as 256 bits) or, for 32..64 bytes, a 64-bit
// tag verified byte by byte against a representative occurrence -- there is no hash-collision case.  The table lives for one batch.
//
// History (profiles/r01_*): a one-launch variant (pass A + decoupled look-back + emit) measured 2x slower -- slices that
// run the model take 5-10 us longer than their neighbours and every later tile waits for them; a block-per-4-KiB-tile
// variant ran at 31 % occupancy because a block keeps its registers and shared memory until its slowest warp is done.
// Hence warp-autonomous slices.  Round 1 handed 8-byte word entries from A to B and let B expand them (1.37 G warp
// instructions for 235 M tokens); now A writes tokens and B only moves them.
#pragma once
#include "tkz_bpe.cuh"
#include "tkz_common.cuh"
#include "tkz_emit.cuh"
#include "tkz_split.cuh"
#include "tkz_wordpiece.cuh"

namespace tkz {

constexpr int TW_THREADS = 256, TW_WARPS = 8, TW_SEG = 32, TW_SLICE = 32 * TW_SEG;      // slice = 1 KiB = one 32-byte segment per lane
constexpr int TW_PRE = 16, TW_POST = 48, TW_STAGE = TW_PRE + TW_SLICE + TW_POST;         // staged window: 16 B before, 48 B behind the slice
constexpr int TW_BLOCKS_PER_SM = 3;                // pass A: 3 blocks of 8 warps -> 80 registers per thread and ~150 KB of shared memory per SM, which leaves
                                                   // ~90 KB of L1 for the table probes; 4 blocks -> 64 registers: the round loop spills (B200, c2b 1 GiB: 4.93 ms
                                                   // against 4.25)
constexpr uint32_t TW_TOK_CHUNK = 16384;           // tokens a warp claims from the token stream with one atomic (then sub-allocates)
constexpr uint32_t TW_SLICE_TOK_MAX = TW_SLICE + 256;   // tokens the words that start in one slice can have (<= their bytes)
constexpr uint32_t TW_MAX_SHORT = 15;             // bytes next to the length byte in the 128-bit key
constexpr uint32_t TW_MAX_MED = 64;               // words of 32..64 bytes: 64-bit tag + byte verification; symbols fit shared memory
constexpr uint32_t TW_MAX_INLINE = 255;           // longest pre-token a warp tokenizes inside pass A (offsets fit a byte)
constexpr int TW_MAX_PROBE = 32;
constexpr uint32_t TW_POOLF = 0x80000000u;        // value flag: token records are in upool[a .. a + ntok)
constexpr uint32_t TW_ERRF = 0x40000000u;         // value flag: the model rejected the word
constexpr uint32_t TW_LONGF = 0x20000000u;        // in registers only: the word joins the long list (a = its length)
constexpr uint32_t TW_NONE = 0xFFFFFFFFu;
constexpr uint32_t TW_MAX_SLICE_LONG = 4;         // long words (> 255 bytes) that can START in one 1 KiB slice

// token stream records, chosen per call (encode_slices) and compiled into both passes.  Offsets fit a byte each (a word of
// pass A has <= 255 bytes); ids fit 16 bits when every id the model can emit is below 65536.
constexpr int TW_REC_ID32 = 0;                    // u32 id (ids only)
constexpr int TW_REC_WIDE = 1;                    // {u32 id, start | end << 8 | the word's position in the slice << 16}
constexpr int TW_REC_ID16 = 2;                    // u16 id (ids only, 16-bit vocabulary)
constexpr int TW_REC4 = 3;                        // u32: id | start << 16 | end << 24 (16-bit vocabulary, pre-token offsets)
constexpr int TW_REC_WORD = 4;                    // {u32 id | k << 22, as TW_REC_WIDE}: k = the word's index in the slice's word list
                                                  // (< 1024), for word ids (TKZ_OUT_WORD_IDS; ids below 2^22)

// 32-byte slot = one L2 sector.  Short words (<= 15 bytes): k0..k3 = the normalised bytes, length in the top byte of k3
// (so a used key is never all zero).  Medium words live in their own slot range: k0,k1 = 64-bit tag (top bit set),
// k2,k3 = representative occurrence (text position, length), published after the tag.
// Value: b = flags | (ntok + 1) << 16 | end0 << 8 | start0; b == 0: not computed yet (the owner stores (a, b) with one
// 8-byte store, after (c, d)).  Without TW_POOLF (0, 1 or 2 tokens): a = id of token 0, c = id of token 1,
// d = end1 << 8 | start1.  With TW_POOLF: a = first record in upool, ntok of them.
struct __align__(32) WordSlot { uint32_t k0, k1, k2, k3, a, b, c, d; };
static_assert(sizeof(WordSlot) == 32, "one sector");

// powers of the medium-word hash multiplier (host-initialised, see tkz_api.cu): PW[j] = MUL^j mod 2^64
__constant__ unsigned long long c_med_pw[TW_MAX_MED];
#define TKZ_MED_HASH_MUL 0x9E3779B97F4A7C15ULL

// 64-byte slot for words of 16..31 bytes (one per lane, like short words): k = [length, bytes 0..14], k2 = bytes 15..30.
// The first half is claimed with atom.cas.b128 (length >= 16 keeps it non-zero), the owner then stores k2 and sets c;
// a, b = the value as in WordSlot (two-token words go to the record pool here: c is taken).
struct __align__(64) WordSlot32 { uint32_t k[4]; uint32_t a, b, c, d; uint32_t k2[4]; uint32_t pad[4]; };
static_assert(sizeof(WordSlot32) == 64, "two sectors");

// byte classes as ranges (filled at upload when the class table allows it): non-WORD bytes are all < 0x80 and form at
// most TW_MAX_RANGES runs per class.  add_lo / add_hi are the packed-byte addends of the range test (see tw_classify4).
constexpr int TW_MAX_RANGES = 6;
struct ClassRanges {
    int usable;                                    // 0: the kernel must use the byte LUT
    int n_delim, n_iso;
    int norm_lower;                                // the byte map is exactly A-Z -> a-z (else identity when usable)
    uint32_t d_lo[TW_MAX_RANGES], d_hi[TW_MAX_RANGES], i_lo[TW_MAX_RANGES], i_hi[TW_MAX_RANGES];
};

struct SliceArgs {
    const uint8_t* text; uint64_t n;
    const uint64_t* doc_off; uint32_t n_docs;
    uint32_t n_slices;
    uint32_t n_bulk;                              // slices [0, n_bulk) have their whole staged window inside the text
    const uint32_t* slice_doc_lo;                 // first document with doc_off >= slice start (n_slices + 1 entries)
    WordSlot* table; uint32_t table_shift; uint32_t med_base, med_mask;          // slot = hash >> table_shift
    WordSlot32* table32; uint32_t table32_mask;
    unsigned long long* upool; uint32_t upool_cap; unsigned int* upool_count;     // token records: id | start << 32 | end << 48
    uint32_t* lscratch;                           // per warp of the grid: 4 * 256 u32, symbol arrays of words of 65..255 bytes
    void* tok; uint32_t tok_cap; unsigned int* tok_count;                         // token stream: tok_cap records of the kind TW_REC_*
    uint32_t* slice_tok_off; uint32_t* slice_ntok_inline; uint32_t* slice_ntok;   // slice_ntok (+ long words) is scanned -> token base
    uint32_t* slice_long;                         // first long-list index << 3 | count of the long words that start in the slice
    uint32_t* doc_tok_local;                      // per document: tokens of its slice before its first word
    uint32_t* long_start; uint32_t* long_end; uint32_t* long_slice; uint32_t* long_ins; unsigned int* n_long; uint32_t long_cap;
    unsigned int* abort_flag;
    unsigned long long* errw;                     // min over failing words of (byte position << 8 | code)
    unsigned long long* n_words; unsigned int* n_uniq; unsigned int* n_uncached;
    ClassRanges cr;
    int has_iso;                                  // some byte is its own pre-token (punctuation split)
    // TW_REC_WORD only: words that start in each slice, index of each document's first word in its slice's word list, the
    // long words' indices in their slice's word list
    uint32_t* slice_nword; uint32_t* doc_word_local; uint32_t* long_k;
};

// first document that starts at or after each tile (slice) start; entry n_tiles = n_docs + 1.  One thread per tile.
__global__ void tile_doc_index_kernel(const uint64_t* __restrict__ doc_off, uint32_t n_docs, uint32_t n_tiles, uint32_t tile_bytes,
                                      uint32_t* __restrict__ tile_doc_lo) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile < n_tiles) tile_doc_lo[tile] = lower_bound_u64(doc_off, 0, n_docs + 1, (uint64_t)tile * tile_bytes);
    else if (tile == n_tiles) tile_doc_lo[tile] = n_docs + 1;
}

struct __align__(16) SliceShared {                                      // per warp
    uint32_t raw[2][TW_STAGE / 4];                        // staged text windows (bulk copy destination), normalised in place
    unsigned long long bar[2];                            // mbarriers of the two windows
    uint32_t cont32[(TW_SLICE + 32) / 32 + 2];            // bit p: byte p continues the word that started before it
    uint32_t docbits[(TW_SLICE + 32) / 32 + 2];           // bit p: a document starts at slice_base + p
    uint16_t wlist[TW_SLICE];                             // start positions of the slice's words (bit 15: ISOLATE byte); a round
                                                          // replaces the entries it has read by the token prefix of its words
                                                          // (tokens of the slice's words before word k, read by the epilogue)
    uint32_t mscr[4][TW_MAX_MED];                         // model scratch: ids, starts, ends, pair ranks
    uint32_t wbytes[TW_MAX_MED / 4];                      // normalised bytes of the word the warp is tokenizing
    uint32_t seg_smask[32], seg_wex[32];                  // per 32-byte segment: word-start bits, words of the slice before it
    uint32_t doc_lo_hi[2];                                // documents that start inside the slice: [lo, hi)
    uint32_t lbuf[TW_MAX_SLICE_LONG][3];                  // long words of the slice: position, length, token index of insertion
    uint4 plist[32];                                      // words of 3+ tokens whose records wait to be copied from the pool: {first record, count, stream position}
};
struct BlockShared {
    uint32_t lut[256];                                    // [7:0] normalised byte, bit 8 WORD, bit 9 ISOLATE
    uint4 lenmask[16];                                    // key mask by length
    SliceShared w[TW_WARPS];
};

// ---------------------------------------------------------------- bulk copy + mbarrier (sm_90+: UBLKCP / SYNCS in SASS)
__device__ __forceinline__ uint32_t tw_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tw_mbar_init(unsigned long long* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(tw_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tw_bulk_load(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(tw_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(tw_smem_u32(dst)), "l"(src), "r"(bytes), "r"(tw_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tw_mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tTW_WAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra TW_DONE_%=;\n\tbra TW_WAIT_%=;\n\tTW_DONE_%=:\n\t}"
                 :: "r"(tw_smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void tw_ld256(const WordSlot* s, uint32_t (&r)[8]) {
    asm volatile("ld.global.ca.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(s) : "memory");
}
// same, straight from L2 (a slot that is looked at again must not be served from a stale L1 line)
__device__ __forceinline__ void tw_ld256_cg(const void* s, uint32_t (&r)[8]) {
    asm volatile("ld.global.cg.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(s) : "memory");
}
__device__ __forceinline__ uint4 tw_ld_value(const WordSlot* s) {
    uint4 v;
    asm volatile("ld.global.relaxed.gpu.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(&s->a) : "memory");
    return v;
}
// (c, d) first, then (a, b): a reader that sees b != 0 sees the second token too
__device__ __forceinline__ void tw_st_value(WordSlot* s, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    if (c | d) {
        asm volatile("st.global.relaxed.gpu.v2.u32 [%0], {%1,%2};" :: "l"(&s->c), "r"(c), "r"(d) : "memory");
        __threadfence();
    }
    asm volatile("st.global.relaxed.gpu.v2.u32 [%0], {%1,%2};" :: "l"(&s->a), "r"(a), "r"(b) : "memory");
}
// returns the previous 128-bit key
__device__ __forceinline__ void tw_cas128(WordSlot* s, const uint32_t (&key)[4], uint32_t (&old)[4]) {
    unsigned long long v0 = (unsigned long long)key[0] | ((unsigned long long)key[1] << 32), v1 = (unsigned long long)key[2] | ((unsigned long long)key[3] << 32);
    unsigned long long o0, o1;
    asm volatile("{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
                 "atom.global.relaxed.gpu.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(o0), "=l"(o1) : "l"(0ULL), "l"(0ULL), "l"(v0), "l"(v1), "l"(s) : "memory");
    old[0] = (uint32_t)o0; old[1] = (uint32_t)(o0 >> 32); old[2] = (uint32_t)o1; old[3] = (uint32_t)(o1 >> 32);
}
// multiply-add mix of the four key words, folded once; the slot is taken from the TOP bits of the last product
__device__ __forceinline__ uint32_t tw_key_hash(uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3) {
    uint32_t h = k0 * 0x9E3779B1u + k1 * 0x85EBCA77u;
    h += k2 * 0xC2B2AE3Du + k3 * 0x27D4EB2Fu;
    h ^= h >> 15;
    return h * 0x2C1B3C6Du;
}

// model on a word of <= TW_MAX_MED normalised bytes held in shared memory; tokens in scr[0] ids, scr[1] starts, scr[2] ends
template <int MODEL>
__device__ __noinline__ uint32_t tw_model_small(const DevModel& m, const uint8_t* bytes, uint32_t len, uint32_t (*scr)[TW_MAX_MED]) {
    uint32_t n;
    if (MODEL == TKZ_MODEL_BPE) n = bpe_encode_word_src(m, PlainSrc{bytes}, len, scr[0], scr[1], scr[2], scr[3]);
    else n = wp_encode_word_src(m, PlainSrc{bytes}, len, scr[0], scr[1], scr[2]);
    __syncwarp();
    return n;
}
// model on a word of 65..TW_MAX_INLINE bytes read from the text; symbol arrays in global scratch (4 * len u32)
template <int MODEL>
__device__ __noinline__ uint32_t tw_model_long(const DevModel& m, const uint8_t* lut_raw, const uint8_t* wt, uint32_t len, uint32_t* g) {
    uint32_t n;
    if (MODEL == TKZ_MODEL_BPE) n = bpe_encode_word_src(m, GlobalLutSrc{lut_raw, wt}, len, g, g + len, g + 2 * len, g + 3 * len);
    else n = wp_encode_word_src(m, GlobalLutSrc{lut_raw, wt}, len, g, g + len, g + 2 * len);
    __syncwarp();
    return n;
}

struct WordVal { uint32_t a, b, c, d; };                 // value of a word in slot encoding
struct WholeWarpOut { WordVal v; bool abort; };          // result of the out-of-line word handlers

// tokens (ids/ss/ee, n of them; n == TKZ_NONE: rejected) -> value; words of more than two tokens (more than one when
// !two_inline) go to the record pool.  Warp-collective; false = pool exhausted.
__device__ __forceinline__ bool tw_make_value(const SliceArgs& a, const uint32_t* ids, const uint32_t* ss, const uint32_t* ee, uint32_t n,
                                              bool two_inline, WordVal& v) {
    const uint32_t lane = lane_id();
    v.a = 0; v.c = 0; v.d = 0;
    if (n == TKZ_NONE) { v.b = TW_ERRF | (1u << 16); return true; }
    if (n == 0) { v.b = 1u << 16; return true; }
    if (n == 1) { v.a = ids[0]; v.b = (2u << 16) | (ee[0] << 8) | ss[0]; return true; }
    if (n == 2 && two_inline) { v.a = ids[0]; v.b = (3u << 16) | (ee[0] << 8) | ss[0]; v.c = ids[1]; v.d = (ee[1] << 8) | ss[1]; return true; }
    uint32_t off = 0;
    if (lane == 0) off = atomicAdd(a.upool_count, n);
    off = __shfl_sync(0xFFFFFFFFu, off, 0);
    if ((unsigned long long)off + n > a.upool_cap) { v.b = 1u << 16; return false; }
    for (uint32_t k = lane; k < n; k += 32)
        __stcg(a.upool + off + k, (unsigned long long)ids[k] | ((unsigned long long)ss[k] << 32) | ((unsigned long long)ee[k] << 48));
    __threadfence();
    __syncwarp();
    v.a = off; v.b = ((n + 1) << 16) | TW_POOLF;
    return true;
}

// ---------------------------------------------------------------- byte classes, four bytes per instruction
// x = 4 packed bytes.  A byte b < 0x80 lies in [lo, hi] iff bit 7 of (b + 0x80 - lo) is set and bit 7 of (b + 0x7F - hi) is
// not; with b taken as b & 0x7F no carry crosses a byte.  Returns the masks in bit 7 of each byte.  N is a compile-time
// count: the addends are then read straight from the kernel parameters as instruction operands.
template <int N>
__device__ __forceinline__ uint32_t tw_in_ranges4(uint32_t x7, const uint32_t* lo, const uint32_t* hi) {
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < N; k++) acc |= (x7 + lo[k]) & ~(x7 + hi[k]);
    return acc;
}
// bits 7, 15, 23, 31 -> a nibble in the TOP four bits (no two partial products share a bit)
__device__ __forceinline__ uint32_t tw_gather4(uint32_t hi_bits) { return hi_bits * 0x00204081u; }

// the class sets the range form is compiled for: ND runs of DELIM bytes (1..3), NI runs of ISOLATE bytes (0 or 4):
// whitespace splits (config.zig:440-450) and the BERT splits (config.zig:405-438, pretokenizer.zig:81-133); any other table
// takes the per-byte look-up
__host__ __device__ __forceinline__ bool tw_ranges_supported(int nd, int ni) { return nd >= 1 && nd <= 3 && (ni == 0 || ni == 4); }

// classify (+ normalise in place) the 8 words of a lane's 32-byte segment held in shared memory
template <int NORM, int ND, int NI>          // NORM: 0 identity, 1 A-Z -> a-z
__device__ __forceinline__ void tw_classify_segment_ranges(const ClassRanges& cr, uint32_t* seg, uint32_t& word_out, uint32_t& iso_out) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(seg), v1 = *reinterpret_cast<const uint4*>(seg + 4);
    uint32_t x[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    uint32_t word = 0, iso = 0;
#pragma unroll
    for (int q = 7; q >= 0; q--) {
        const uint32_t x7 = x[q] & 0x7F7F7F7Fu;
        const uint32_t nh = ~x[q] & 0x80808080u;                                  // bytes below 0x80
        const uint32_t dl = tw_in_ranges4<ND>(x7, cr.d_lo, cr.d_hi);
        uint32_t is = 0;
        if (NI) is = tw_in_ranges4<NI>(x7, cr.i_lo, cr.i_hi) & nh;
        const uint32_t wd = ~(dl & nh) & ~is & 0x80808080u;                       // WORD: neither (bytes >= 0x80 are WORD)
        word = __funnelshift_l(tw_gather4(wd), word, 4);
        if (NI) iso = __funnelshift_l(tw_gather4(is), iso, 4);
        if (NORM == 1) {
            const uint32_t up = (x7 + 0x3F3F3F3Fu) & ~(x7 + 0x25252525u) & nh;   // 'A' (0x41) .. 'Z' (0x5A)
            x[q] |= up >> 2;                                                      // + 0x20
        }
    }
    if (NORM == 1) {
        *reinterpret_cast<uint4*>(seg) = make_uint4(x[0], x[1], x[2], x[3]);
        *reinterpret_cast<uint4*>(seg + 4) = make_uint4(x[4], x[5], x[6], x[7]);
    }
    word_out = word; iso_out = iso;
}
// one word (4 bytes) the same way: returns nibbles in the low 4 bits
template <int NORM, int ND, int NI>
__device__ __forceinline__ void tw_classify_word_ranges(const ClassRanges& cr, uint32_t* wp, uint32_t& word_nib, uint32_t& iso_nib) {
    uint32_t x = *wp;
    const uint32_t x7 = x & 0x7F7F7F7Fu, nh = ~x & 0x80808080u;
    const uint32_t dl = tw_in_ranges4<ND>(x7, cr.d_lo, cr.d_hi);
    uint32_t is = 0;
    if (NI) is = tw_in_ranges4<NI>(x7, cr.i_lo, cr.i_hi) & nh;
    const uint32_t wd = ~(dl & nh) & ~is & 0x80808080u;
    word_nib = tw_gather4(wd) >> 28; iso_nib = tw_gather4(is) >> 28;
    if (NORM == 1) {
        const uint32_t up = (x7 + 0x3F3F3F3Fu) & ~(x7 + 0x25252525u) & nh;
        *wp = x | (up >> 2);
    }
}
// phase 1 in range form: the lane's segment, the 32 bytes behind the slice (lanes 0..7: class nibbles, lanes 8..11 only
// normalise), the byte before it (lane 12)
template <int NORM, int ND, int NI>
__device__ __forceinline__ void tw_phase1_ranges(const ClassRanges& cr, uint32_t* tw, uint32_t& word, uint32_t& iso, uint32_t& hw, uint32_t& hi, uint32_t& prev_byte_word) {
    const uint32_t FULL = 0xFFFFFFFFu, lane = lane_id();
    tw_classify_segment_ranges<NORM, ND, NI>(cr, tw + lane * 8, word, iso);
    uint32_t wn = 0, in_ = 0;
    if (lane < 12) tw_classify_word_ranges<NORM, ND, NI>(cr, tw + TW_SLICE / 4 + lane, wn, in_);
    else if (lane == 12) { uint32_t tmp = tw[-1]; tw_classify_word_ranges<0, ND, NI>(cr, &tmp, wn, in_); }
    prev_byte_word = __shfl_sync(FULL, wn, 12) >> 3;
    const uint32_t sh4 = (lane & 7u) * 4u;
    hw = __reduce_or_sync(FULL, lane < 8 ? wn << sh4 : 0u);
    hi = NI ? __reduce_or_sync(FULL, lane < 8 ? in_ << sh4 : 0u) : 0u;
}
// arbitrary tables: one look-up per byte (identity byte map: 256-bit class tables held by lanes 0..7 and read by shuffle,
// because 32 lanes x arbitrary bytes serialise on the banks of a shared-memory LUT)
template <bool NORM_ID, bool HAS_ISO>
__device__ __forceinline__ void tw_classify_segment_lut(const uint32_t* lut, uint32_t cw_word, uint32_t cw_iso, uint32_t* seg, uint32_t& word_out, uint32_t& iso_out) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(seg), v1 = *reinterpret_cast<const uint4*>(seg + 4);
    const uint32_t x[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    uint32_t word = 0, iso = 0, nrm[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        uint32_t o = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t b = (x[q] >> (8 * j)) & 0xFFu;
            if (NORM_ID) {
                word |= ((__shfl_sync(0xFFFFFFFFu, cw_word, b >> 5) >> (b & 31u)) & 1u) << (q * 4 + j);
                if (HAS_ISO) iso |= ((__shfl_sync(0xFFFFFFFFu, cw_iso, b >> 5) >> (b & 31u)) & 1u) << (q * 4 + j);
            } else {
                const uint32_t e = lut[b];
                word |= ((e >> 8) & 1u) << (q * 4 + j);
                if (HAS_ISO) iso |= ((e >> 9) & 1u) << (q * 4 + j);
                o |= (e & 0xFFu) << (8 * j);
            }
        }
        nrm[q] = o;
    }
    if (!NORM_ID) {
        *reinterpret_cast<uint4*>(seg) = make_uint4(nrm[0], nrm[1], nrm[2], nrm[3]);
        *reinterpret_cast<uint4*>(seg + 4) = make_uint4(nrm[4], nrm[5], nrm[6], nrm[7]);
    }
    word_out = word; iso_out = iso;
}

// exclusive prefix + total of per-lane values < 2^BITS with BITS ballots (no dependent shuffle chain)
template <int BITS>
__device__ __forceinline__ uint32_t tw_ballot_prefix(uint32_t v, uint32_t lt_mask, uint32_t& total) {
    uint32_t ex = 0, tot = 0;
#pragma unroll
    for (int b = 0; b < BITS; b++) {
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, (v >> b) & 1u);
        ex += __popc(m & lt_mask) << b; tot += __popc(m) << b;
    }
    total = tot;
    return ex;
}

// 128-bit key of the word of `len` (<= 15) bytes at slice position p: the normalised bytes, length in the top byte
__device__ __forceinline__ void tw_build_key(const uint32_t* tw, const uint4* lenmask, uint32_t p, uint32_t len, uint32_t (&key)[4]) {
    const uint32_t wi = p >> 2, shb = (p & 3u) * 8u;
    const uint32_t x0 = tw[wi], x1 = tw[wi + 1], x2 = tw[wi + 2], x3 = tw[wi + 3], x4 = tw[wi + 4];
    const uint4 mk = lenmask[len];
    key[0] = __funnelshift_r(x0, x1, shb) & mk.x;
    key[1] = __funnelshift_r(x1, x2, shb) & mk.y;
    key[2] = __funnelshift_r(x2, x3, shb) & mk.z;
    key[3] = (__funnelshift_r(x3, x4, shb) & mk.w) | (len << 24);
}

// 256-bit key of the word of `len` (16..31) bytes at slice position p: key[0..3] = [len, bytes 0..14], key[4..7] = bytes 15..30
__device__ __forceinline__ void tw_build_key32(const uint32_t* tw, const uint4* lenmask, uint32_t p, uint32_t len, uint32_t (&key)[8]) {
    const uint32_t wi = p >> 2, shb = (p & 3u) * 8u;
    uint32_t w[8];
    uint32_t x = tw[wi];
#pragma unroll
    for (int i = 0; i < 8; i++) { const uint32_t y = tw[wi + 1 + i]; w[i] = __funnelshift_r(x, y, shb); x = y; }
    const uint4 mk = lenmask[len - 16];                            // bytes 16.. of the word: keep len - 16 of them
    w[4] &= mk.x; w[5] &= mk.y; w[6] &= mk.z; w[7] &= mk.w;
    key[0] = len | (w[0] << 8);
#pragma unroll
    for (int i = 1; i < 8; i++) key[i] = (w[i - 1] >> 24) | (w[i] << 8);
}
__device__ __forceinline__ uint32_t tw_key_hash32(const uint32_t (&k)[8]) {
    uint32_t h = k[0] * 0x9E3779B1u;
#pragma unroll
    for (int i = 1; i < 8; i++) h = (h ^ k[i] ^ (h >> 15)) * (0x85EBCA77u + 2u * (uint32_t)i * 0x9E3779B1u);
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 13;
    return h;
}

// One word of 16..31 bytes this warp saw first: model + publish into its WordSlot32.  Out of line.
template <int MODEL>
__device__ __forceinline__ WholeWarpOut tw_own_word32(const DevModel& m, const SliceArgs& a, SliceShared& sh, const uint32_t* tw, uint32_t wp_, uint32_t wlen, uint32_t bslot) {
    const uint32_t lane = lane_id();
    WholeWarpOut out{{0u, 0u, 0u, 0u}, false};
    uint8_t* const wbytes = reinterpret_cast<uint8_t*>(sh.wbytes);
    wbytes[lane] = (reinterpret_cast<const uint8_t*>(tw) + wp_)[lane];     // the whole word is in the slice + halo
    __syncwarp();
    const uint32_t n = tw_model_small<MODEL>(m, wbytes, wlen, sh.mscr);
    if (!tw_make_value(a, sh.mscr[0], sh.mscr[1], sh.mscr[2], n, false, out.v)) out.abort = true;
    if (lane == 0) asm volatile("st.global.relaxed.gpu.v2.u32 [%0], {%1,%2};" :: "l"(&a.table32[bslot].a), "r"(out.v.a), "r"(out.v.b) : "memory");
    __syncwarp();
    return out;
}

// One word that needs the whole warp (longer than 31 bytes, or no table slot within the probe limit): finds its end, then
// medium words (<= 64 bytes) go through the tag table, 65..255 bytes are tokenized uncached, longer ones are returned with
// TW_LONGF (a = length) and join the long list.  Kept out of line so that its registers do not weigh on the round loop.
template <int MODEL>
__device__ __forceinline__ WholeWarpOut tw_whole_warp_word(const DevModel& m, const SliceArgs& a, const uint32_t* lut, SliceShared& sh, const uint32_t* tw,
                                                        uint32_t s, uint32_t wp_, uint32_t wl_, uint32_t* lscr) {
    const uint64_t slice_base = (uint64_t)s * TW_SLICE;
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = lane_id();
    uint8_t* const wbytes = reinterpret_cast<uint8_t*>(sh.wbytes);
    WholeWarpOut out{{0u, 1u << 16, 0u, 0u}, false};
    const uint64_t start = slice_base + wp_;
    uint32_t wlen = wl_;
    if (wl_ > 32) {
        // end of the word: first non-WORD byte or the next document start, 32 bytes per step
        // next document start behind the word's first byte: inside the slice from the document-start bits (one 32-bit
        // word per lane), else the first document of the following slices (no binary search)
        uint64_t limit;
        {
            uint32_t wd = sh.docbits[lane];
            const uint32_t q1 = wp_ + 1;                        // first candidate position
            if (lane < (q1 >> 5)) wd = 0;
            else if (lane == (q1 >> 5)) wd &= 0xFFFFFFFFu << (q1 & 31u);
            const uint32_t any = __ballot_sync(FULL, wd != 0);
            if (any) {
                const int l0 = __ffs(any) - 1;
                limit = slice_base + 32u * (uint32_t)l0 + (uint32_t)(__ffs(__shfl_sync(FULL, wd, l0)) - 1);
            } else {
                const uint32_t dn = sh.doc_lo_hi[1];             // first document that starts at or after the next slice
                limit = dn <= a.n_docs ? __ldg(a.doc_off + dn) : a.n;
            }
            if (limit > a.n) limit = a.n;
        }
        // WordPiece only needs the LENGTH of a word above max_input_chars_per_word (wordpiece.zig:149-158)
        uint64_t q = start + 32;
        bool found = false;
        for (int round = 0; round < 7 && !found; round++) {       // the next 224 bytes one per lane: every word that stays inline (<= 255 bytes) ends here
            const uint64_t qq = q + lane;
            const bool stop = qq >= limit || ((lut[__ldg(a.text + qq)] >> 8) & 1u) == 0;
            const uint32_t sm = __ballot_sync(FULL, stop);
            if (sm) { q += (uint32_t)__ffs(sm) - 1; found = true; } else q += 32;
        }
        if (!found) {
            // long unbroken run (up to MiBs): 512 bytes per step, one aligned 16-byte load per lane
            const uint32_t pre = (uint32_t)((16u - (uint32_t)(q & 15u)) & 15u);
            {
                const uint64_t qq = q + lane;
                const bool stop = lane < pre && (qq >= limit || ((lut[__ldg(a.text + qq)] >> 8) & 1u) == 0);
                const uint32_t sm = __ballot_sync(FULL, stop);
                if (sm) { q += (uint32_t)__ffs(sm) - 1; found = true; } else q += pre;
            }
            while (!found) {
                const uint64_t qq = q + 16u * lane;
                uint32_t mask = 0;                                  // bit j: the word stops at byte qq + j
                if (qq + 16 <= limit) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4*>(a.text + qq));
                    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int j = 0; j < 16; j++) mask |= ((((lut[(w4[j >> 2] >> (8 * (j & 3))) & 0xFFu] >> 8) & 1u) ^ 1u) << j);
                } else {
                    for (int j = 0; j < 16; j++) if (qq + j >= limit || ((lut[__ldg(a.text + qq + j)] >> 8) & 1u) == 0) { mask |= 1u << j; break; }
                }
                const uint32_t sm = __ballot_sync(FULL, mask != 0);
                if (sm) {
                    const int l0 = __ffs(sm) - 1;
                    q += 16u * (uint32_t)l0 + (uint32_t)(__ffs(__shfl_sync(FULL, mask, l0)) - 1);
                    found = true;
                } else q += 512;
            }
        }
        wlen = (uint32_t)(q - start);
    }
    WordVal xv{0u, 1u << 16, 0u, 0u};                    // default: no tokens
    if (MODEL == TKZ_MODEL_WORDPIECE && (uint64_t)wlen > m.max_chars && wlen <= TW_MAX_INLINE) {
        // one [UNK] spanning the word (wordpiece.zig:149-158); MissingUnkToken when the vocabulary has none.  (Longer words
        // take the long list: wordpiece_warp_kernel applies the same rule with 32-bit offsets.)
        uint32_t* scr = sh.mscr[0];
        if (lane == 0) { scr[0] = m.unk_id; scr[1] = 0; scr[2] = wlen; }
        __syncwarp();
        if (!tw_make_value(a, scr, scr + 1, scr + 2, m.has_unk ? 1u : TKZ_NONE, false, xv)) out.abort = true;
    } else if (wlen > TW_MAX_INLINE) {
        // long list: tokenized per occurrence by the word-list kernels between the two passes (block-level BPE)
        xv.a = wlen; xv.b = TW_LONGF | (1u << 16);
    } else if (wlen > TW_MAX_MED) {
        // 65..255 bytes: not deduplicated, symbols in the warp's global scratch
        if (lane == 0) atomicAdd(a.n_uncached, 1u);
        const uint32_t n = tw_model_long<MODEL>(m, m.lut, a.text + start, wlen, lscr);
        __threadfence_block();
        if (!tw_make_value(a, lscr, lscr + wlen, lscr + 2 * wlen, n, false, xv)) out.abort = true;
        __syncwarp();
    } else {
        // <= 64 bytes: normalised bytes into shared memory
        if (wlen <= 32) {                                // the whole word is in the slice + halo
            const uint8_t* tb = reinterpret_cast<const uint8_t*>(tw) + wp_;
            wbytes[lane] = tb[lane];
        } else {
            uint32_t bb = 0;
            if (2 * lane < wlen) bb = lut[__ldg(a.text + start + 2 * lane)] & 0xFFu;
            if (2 * lane + 1 < wlen) bb |= (lut[__ldg(a.text + start + 2 * lane + 1)] & 0xFFu) << 8;
            reinterpret_cast<uint16_t*>(wbytes)[lane] = (uint16_t)bb;
        }
        __syncwarp();
        int mode = 0;                                   // 0 compute, do not publish | 1 owner | 2 value found
        WordSlot* ms = nullptr;
        if (wlen > TW_MAX_SHORT) {
            // medium word: 64-bit tag = mixed polynomial hash of the normalised bytes, exactness by comparing with
            // the representative occurrence
            unsigned long long h = 0;
            if (2 * lane < wlen) h += (unsigned long long)(wbytes[2 * lane] + 1u) * c_med_pw[2 * lane];
            if (2 * lane + 1 < wlen) h += (unsigned long long)(wbytes[2 * lane + 1] + 1u) * c_med_pw[2 * lane + 1];
            for (int d = 16; d > 0; d >>= 1) h += __shfl_xor_sync(FULL, h, d);
            h ^= wlen; h ^= h >> 29; h *= 0xD6E8FEB86659FD93ULL; h ^= h >> 32;
            const unsigned long long tag = h | 0x8000000000000000ULL;
            unsigned long long* const tab64 = reinterpret_cast<unsigned long long*>(a.table + a.med_base);
            uint32_t slot = (uint32_t)h & a.med_mask;
            for (int probe = 0; probe < TW_MAX_PROBE && mode == 0; probe++) {
                unsigned long long* kp = tab64 + (size_t)slot * 4;       // [0] tag, [1] representative, [2] value
                unsigned long long cur = 0;
                if (lane == 0) {
                    cur = __ldcg(kp);
                    if (cur == 0) {
                        cur = atomicCAS(kp, 0ULL, tag);
                        if (cur == 0) {
                            __stcg(kp + 1, (unsigned long long)(uint32_t)start | ((unsigned long long)wlen << 32));
                            __threadfence();
                            atomicAdd(a.n_uniq, 1u);
                            cur = 1;                               // marker: owned
                        }
                    }
                }
                cur = __shfl_sync(FULL, cur, 0);
                if (cur == 1) { mode = 1; ms = a.table + a.med_base + slot; break; }
                if (cur == tag) {
                    unsigned long long rm = 0;
                    if (lane == 0) rm = __ldcg(kp + 1);
                    rm = __shfl_sync(FULL, rm, 0);
                    if (rm == 0) break;                            // representative not published yet: compute privately
                    bool eq = (uint32_t)(rm >> 32) == wlen;
                    if (eq) {
                        const uint8_t* __restrict__ rp = a.text + (uint32_t)rm;
                        if (2 * lane < wlen) eq = eq && (lut[__ldg(rp + 2 * lane)] & 0xFFu) == wbytes[2 * lane];
                        if (2 * lane + 1 < wlen) eq = eq && (lut[__ldg(rp + 2 * lane + 1)] & 0xFFu) == wbytes[2 * lane + 1];
                    }
                    if (__all_sync(FULL, eq)) { mode = 2; ms = a.table + a.med_base + slot; break; }
                }
                slot = (slot + 1) & a.med_mask;
            }
        }
        if (mode == 2) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (lane == 0) { do { v = tw_ld_value(ms); } while (v.y == 0); }
            xv.a = __shfl_sync(FULL, v.x, 0); xv.b = __shfl_sync(FULL, v.y, 0);
        } else {
            if (mode == 0 && lane == 0) atomicAdd(a.n_uncached, 1u);
            const uint32_t n = tw_model_small<MODEL>(m, wbytes, wlen, sh.mscr);
            if (!tw_make_value(a, sh.mscr[0], sh.mscr[1], sh.mscr[2], n, false, xv)) out.abort = true;
            if (mode == 1 && lane == 0) tw_st_value(ms, xv.a, xv.b, 0u, 0u);
        }
    }
    out.v = xv;
    return out;
}

// One word this warp saw first (short key): model + publish.  Out of line for the same reason.
template <int MODEL>
__device__ __forceinline__ WholeWarpOut tw_own_word(const DevModel& m, const SliceArgs& a, SliceShared& sh, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3,
                                                 uint32_t bslot) {
    const uint32_t lane = lane_id();
    WholeWarpOut out{{0u, 0u, 0u, 0u}, false};
    if (lane < 4) sh.wbytes[lane] = lane == 0 ? b0 : (lane == 1 ? b1 : (lane == 2 ? b2 : (b3 & 0x00FFFFFFu)));
    __syncwarp();
    const uint32_t n = tw_model_small<MODEL>(m, reinterpret_cast<const uint8_t*>(sh.wbytes), b3 >> 24, sh.mscr);
    if (!tw_make_value(a, sh.mscr[0], sh.mscr[1], sh.mscr[2], n, true, out.v)) out.abort = true;
    if (lane == 0) tw_st_value(a.table + bslot, out.v.a, out.v.b, out.v.c, out.v.d);
    __syncwarp();
    return out;
}

// one token into the stream at index i: of = start | end << 8, ph = the word's position in the slice << 16, k = the word's
// index in the slice's word list (TW_REC_WORD)
template <int REC>
__device__ __forceinline__ void tw_put_token(void* tok, uint32_t i, uint32_t id, uint32_t of, uint32_t ph, uint32_t k = 0) {
    if (REC == TW_REC_WIDE) static_cast<uint2*>(tok)[i] = make_uint2(id, of | ph);
    else if (REC == TW_REC_WORD) static_cast<uint2*>(tok)[i] = make_uint2(id | (k << 22), of | ph);
    else if (REC == TW_REC4) static_cast<uint32_t*>(tok)[i] = id | (of << 16);
    else if (REC == TW_REC_ID16) static_cast<uint16_t*>(tok)[i] = (uint16_t)id;
    else static_cast<uint32_t*>(tok)[i] = id;
}

// copies the token records of the listed words (three or more tokens each) from the pool into the token stream: four lanes
// per word, eight words per step, so that the L2 round trips of a whole slice overlap (one at a time they were 17 % of the
// kernel's stall samples)
template <int REC>
__device__ __forceinline__ void tw_flush_pooled(const SliceArgs& a, const uint4* plist, uint32_t n) {
    const uint32_t lane = lane_id();
    __syncwarp();
    for (uint32_t e = lane >> 2; e < n; e += 8) {
        const uint4 q = plist[e];
        for (uint32_t i = lane & 3u; i < q.y; i += 4) {
            const unsigned long long r = __ldcg(a.upool + q.x + i);       // written in THIS launch by the word's owner: L2, not the read-only path
            const uint32_t of = ((uint32_t)(r >> 32) & 0xFFu) | (((uint32_t)(r >> 48) & 0xFFu) << 8);
            if (REC == TW_REC_WORD) tw_put_token<REC>(a.tok, q.z + i, (uint32_t)r, of, q.w & 0xFFFF0000u, q.w & 0xFFFFu);   // (q.w = p << 16 | k)
            else tw_put_token<REC>(a.tok, q.z + i, (uint32_t)r, of, q.w);
        }
    }
    __syncwarp();
}

// CLS: 0 byte ranges + identity byte map, 1 byte ranges + ASCII lower-case, 2 LUT + identity, 3 LUT + arbitrary byte map
// REC: the token stream's record kind (TW_REC_*)
// pass A: one warp per 1 KiB slice, slices strided over all warps of the grid (3 blocks of 8 warps per SM)
template <int MODEL, int CLS, int REC>
__global__ void __launch_bounds__(TW_THREADS, TW_BLOCKS_PER_SM) slice_words_kernel(const __grid_constant__ DevModel m, const __grid_constant__ SliceArgs a) {
    extern __shared__ __align__(128) unsigned char tw_smem_raw[];
    BlockShared& bs = *reinterpret_cast<BlockShared*>(tw_smem_raw);
    constexpr bool RANGES = CLS < 2;
    constexpr bool NORM_ID = CLS == 0 || CLS == 2;
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    {
        const uint32_t c = m.lut[256 + t];
        bs.lut[t] = (uint32_t)m.lut[t] | ((c == 0) ? 0x100u : 0u) | ((c == 2) ? 0x200u : 0u);
    }
    if (t < 16) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; q++) { const int nb = (int)t - 4 * q; w[q] = nb >= 4 ? 0xFFFFFFFFu : (nb <= 0 ? 0u : ((1u << (8 * nb)) - 1u)); }
        bs.lenmask[t] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    SliceShared& sh = bs.w[wid];
    if (lane == 0) { tw_mbar_init(&sh.bar[0]); tw_mbar_init(&sh.bar[1]); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();                                            // the only block-level barrier
    // class bits of byte values 32 * lane .. 32 * lane + 31 (lanes 0..7), for the shuffle look-up of the LUT + identity mode
    uint32_t cw_word = 0, cw_iso = 0;
    if (CLS == 2 && lane < 8) for (int j = 0; j < 32; j++) { const uint32_t e = bs.lut[32 * lane + j]; cw_word |= ((e >> 8) & 1u) << j; cw_iso |= ((e >> 9) & 1u) << j; }
    const uint32_t stride = gridDim.x * TW_WARPS;
    const uint32_t gwarp = blockIdx.x * TW_WARPS + wid;
    bool warp_abort = false;

    // a slice whose whole staged window lies inside the text is fetched by a bulk copy; the last one or two slices of the
    // batch are loaded byte by byte with bounds checks
    auto bulk_ok = [&](uint32_t sl) -> bool { return sl < a.n_bulk; };
    auto issue = [&](uint32_t sl, uint32_t buf) {
        const uint64_t base = (uint64_t)sl * TW_SLICE;
        if (sl == 0) tw_bulk_load(reinterpret_cast<uint8_t*>(sh.raw[buf]) + TW_PRE, a.text, TW_SLICE + TW_POST, &sh.bar[buf]);
        else tw_bulk_load(sh.raw[buf], a.text + base - TW_PRE, TW_STAGE, &sh.bar[buf]);
    };

    uint32_t s = gwarp;
    uint32_t meta = (lane < 2 && s < a.n_slices) ? __ldg(a.slice_doc_lo + s + lane) : 0u;
    uint32_t tcur = 0, tend = 0;                                // the warp's current chunk of the token stream
    uint32_t buf = 0, phase = 0;                                // staging window in use, parity bits of the two mbarriers
    uint32_t words_total = 0;
    if (lane == 0 && bulk_ok(s)) issue(s, 0);
    for (; s < a.n_slices; s += stride, buf ^= 1u) {
        const uint64_t slice_base = (uint64_t)s * TW_SLICE;
        const uint32_t d_lo = __shfl_sync(FULL, meta, 0);
        if (lane < 2) sh.doc_lo_hi[lane] = meta;                   // the epilogue reads them back (not kept in registers)
        meta = (lane < 2 && s + stride < a.n_slices) ? __ldg(a.slice_doc_lo + s + stride + lane) : 0u;
        uint32_t* const rawb = sh.raw[buf];
        uint32_t* const tw = rawb + TW_PRE / 4;                    // word 0 = bytes 0..3 of the slice
        uint8_t* const tb = reinterpret_cast<uint8_t*>(tw);
        // the warp's next slice goes into the other window now (its readers finished at the end of the previous iteration)
        if (lane == 0 && bulk_ok(s + stride)) {
            if (!NORM_ID) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the window was normalised in place
            issue(s + stride, buf ^ 1u);
        }
        // ---- phase 1: document-start bits; classify + normalise one 32-byte segment per lane
        for (uint32_t i = lane; i < (TW_SLICE + 32) / 32 + 2; i += 32) { sh.docbits[i] = 0; sh.cont32[i] = 0; }
        __syncwarp();
        for (uint32_t d = d_lo + lane; d <= a.n_docs; d += 32) {
            const uint64_t off = __ldg(a.doc_off + d);
            if (off > slice_base + TW_SLICE + 32) break;
            const uint32_t p = (uint32_t)(off - slice_base);
            atomicOr(&sh.docbits[p >> 5], 1u << (p & 31));
        }
        const bool tail = !bulk_ok(s);
        if (!tail) { tw_mbar_wait(&sh.bar[buf], (phase >> buf) & 1u); phase ^= 1u << buf; }
        else {
            // bytes at or beyond n read as 0 and are masked out of the class bits below
            for (uint32_t i = lane; i < TW_STAGE / 4; i += 32) {
                uint32_t v = 0;
                for (int j = 0; j < 4; j++) {
                    const long long q = (long long)slice_base - TW_PRE + 4 * i + j;
                    if (q >= 0 && (uint64_t)q < a.n) v |= (uint32_t)__ldg(a.text + q) << (8 * j);
                }
                rawb[i] = v;
            }
            __syncwarp();
        }
        uint32_t word, iso, hw, hi, prev_byte_word;
        if (RANGES) {
            constexpr int NRM = CLS == 1 ? 1 : 0;
            switch (a.cr.n_delim * 2 + (a.cr.n_iso ? 1 : 0)) {
                case 2: tw_phase1_ranges<NRM, 1, 0>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
                case 3: tw_phase1_ranges<NRM, 1, 4>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
                case 4: tw_phase1_ranges<NRM, 2, 0>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
                case 5: tw_phase1_ranges<NRM, 2, 4>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
                case 6: tw_phase1_ranges<NRM, 3, 0>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
                default: tw_phase1_ranges<NRM, 3, 4>(a.cr, tw, word, iso, hw, hi, prev_byte_word); break;
            }
        } else {
            if (a.has_iso) tw_classify_segment_lut<NORM_ID, true>(bs.lut, cw_word, cw_iso, tw + lane * 8, word, iso);
            else tw_classify_segment_lut<NORM_ID, false>(bs.lut, cw_word, cw_iso, tw + lane * 8, word, iso);
            const uint32_t he = bs.lut[tb[TW_SLICE + lane]];
            if (!NORM_ID) { tb[TW_SLICE + lane] = (uint8_t)he; if (lane < 16) tb[TW_SLICE + 32 + lane] = (uint8_t)bs.lut[tb[TW_SLICE + 32 + lane]]; }
            hw = __ballot_sync(FULL, (he >> 8) & 1u); hi = __ballot_sync(FULL, (he >> 9) & 1u);
            prev_byte_word = (bs.lut[tb[-1]] >> 8) & 1u;
        }
        if (slice_base == 0) prev_byte_word = 0;
        if (tail) {
            // validity: bytes of the lane's segment / of the halo that lie inside the text
            const long long rem = (long long)a.n - (long long)(slice_base + (uint64_t)lane * TW_SEG);
            const uint32_t valid = rem >= 32 ? FULL : (rem <= 0 ? 0u : ((1u << rem) - 1u));
            word &= valid; iso &= valid;
            const long long hrem = (long long)a.n - (long long)(slice_base + TW_SLICE);
            const uint32_t hvalid = hrem >= 32 ? FULL : (hrem <= 0 ? 0u : ((1u << hrem) - 1u));
            hw &= hvalid; hi &= hvalid;
        }
        __syncwarp();

        // ---- phase 2: word starts, continuation bits, word list
        uint32_t nW;
        {
            uint32_t smask, wex;
            uint32_t prev_word = __shfl_up_sync(FULL, word >> 31, 1);
            if (lane == 0) prev_word = prev_byte_word;
            const uint32_t ds = sh.docbits[lane];
            smask = iso | (word & (~((word << 1) | prev_word) | ds));
            sh.cont32[lane] = word & ~smask;
            // halo bytes: continuation bits (same formula)
            const uint32_t w31 = __shfl_sync(FULL, word >> 31, 31);
            const uint32_t hs = hi | (hw & (~((hw << 1) | w31) | sh.docbits[32]));
            if (lane == 0) sh.cont32[32] = hw & ~hs;
            const uint32_t cnt = __popc(smask);
            const uint32_t inc = warp_incl_scan(cnt);
            wex = inc - cnt; nW = __shfl_sync(FULL, inc, 31);
            sh.seg_smask[lane] = smask; sh.seg_wex[lane] = wex;
            uint32_t sm = smask, k = wex;
            while (sm) {
                const int b = __ffs(sm) - 1; sm &= sm - 1;
                sh.wlist[k++] = (uint16_t)((lane * TW_SEG + b) | (((iso >> b) & 1u) << 15));
            }
        }
        words_total += nW;
        // reserve the slice's run of the token stream: the warp sub-allocates from a chunk it claimed with one atomic
        if (tcur + TW_SLICE_TOK_MAX > tend) {
            uint32_t c = 0;
            if (lane == 0) c = atomicAdd(a.tok_count, TW_TOK_CHUNK);
            tcur = __shfl_sync(FULL, c, 0); tend = tcur + TW_TOK_CHUNK;
            if ((unsigned long long)tend > a.tok_cap) { warp_abort = true; tend = tcur; }
        }
        const bool can_store = tcur + TW_SLICE_TOK_MAX <= tend;
        const uint32_t tbase = tcur;
        __syncwarp();

        // ---- phase 3: one word per lane
        uint32_t run = 0;                                           // tokens of the slice's words so far
        uint32_t n_long_here = 0, n_pl = 0;
        for (uint32_t k0 = 0; k0 < nW; k0 += 32) {
            const uint32_t k = k0 + lane;
            const bool have = k < nW;
            // straight-line first probe for every lane (lanes past the end repeat the slice's last word, result ignored)
            const uint32_t pw = sh.wlist[have ? k : nW - 1];
            const uint32_t p = pw & 0x0FFFu;
            uint32_t len;
            {
                const uint32_t q = p + 1, w = q >> 5;
                const uint32_t x = __funnelshift_r(sh.cont32[w], sh.cont32[w + 1], q & 31u);
                len = (uint32_t)__ffs((int)~x);                     // 1 + continuing bytes; 0 when 32 or more continue
                if (len == 0) len = 33;
                if (pw & 0x8000u) len = 1;
            }
            const bool is_short = len <= TW_MAX_SHORT;
            uint32_t key[4];
            tw_build_key(tw, bs.lenmask, p, is_short ? len : TW_MAX_SHORT, key);
            uint32_t myslot = tw_key_hash(key[0], key[1], key[2], key[3]) >> a.table_shift;
            WordVal v;
            int state;                                              // 0 done, 1 owner, 2 pending, 3 whole warp needed, 4 keep probing
            {
                uint32_t r[8];
                tw_ld256(a.table + myslot, r);
                v.a = r[4]; v.b = r[5]; v.c = r[6]; v.d = r[7];
                const bool hit = is_short && r[0] == key[0] && r[1] == key[1] && r[2] == key[2] && r[3] == key[3] && r[5] != 0;
                state = (!have || hit) ? 0 : (is_short ? 4 : 3);
            }
            if (__any_sync(FULL, state != 0)) {
                // ---- rare: first sight of a word, a collision, a word whose owner is still computing, a long word
                const uint32_t tmask = (0xFFFFFFFFu >> a.table_shift);
                if (state == 4) {
                    uint32_t slot = myslot;
                    state = 3;
#pragma unroll 1
                    for (int probe = 0; probe < TW_MAX_PROBE; probe++) {
                        WordSlot* sl = a.table + slot;
                        uint32_t r[8];
                        tw_ld256(sl, r);
                        if (r[0] == key[0] && r[1] == key[1] && r[2] == key[2] && r[3] == key[3]) {
                            if (r[5] != 0) { v.a = r[4]; v.b = r[5]; v.c = r[6]; v.d = r[7]; state = 0; } else { state = 2; myslot = slot; }
                            break;
                        }
                        if ((r[0] | r[1] | r[2] | r[3]) == 0) {
                            uint32_t old[4];
                            tw_cas128(sl, key, old);
                            if ((old[0] | old[1] | old[2] | old[3]) == 0) { state = 1; myslot = slot; break; }
                            if (old[0] == key[0] && old[1] == key[1] && old[2] == key[2] && old[3] == key[3]) { state = 2; myslot = slot; break; }
                        }
                        slot = (slot + 1) & tmask;
                    }
                }
                // words this warp saw first: run the model now and publish the value
                uint32_t owners = __ballot_sync(FULL, state == 1);
                if (owners && lane == 0) atomicAdd(a.n_uniq, (unsigned int)__popc(owners));
                while (owners) {
                    const int l = __ffs(owners) - 1; owners &= owners - 1;
                    const WholeWarpOut r = tw_own_word<MODEL>(m, a, sh, __shfl_sync(FULL, key[0], l), __shfl_sync(FULL, key[1], l),
                                                              __shfl_sync(FULL, key[2], l), __shfl_sync(FULL, key[3], l), __shfl_sync(FULL, myslot, l));
                    if (r.abort) warp_abort = true;
                    if ((int)lane == l) { v = r.v; state = 0; }
                }
                // words of 16..31 bytes: one per lane through the 64-byte slots (state 5 probing, 6 pending, 7 owner)
                if (state == 3 && len >= 16 && len <= 31) state = 5;
                if (__any_sync(FULL, state == 5)) {
                    uint32_t k32[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    uint32_t slot = 0;
                    if (state == 5) { tw_build_key32(tw, bs.lenmask, p, len, k32); slot = tw_key_hash32(k32) & a.table32_mask; }
                    // warp-uniform probe rounds: a lane that meets a half-published key simply looks again next round
#pragma unroll 1
                    for (int it = 0; it < 4 * TW_MAX_PROBE && __any_sync(FULL, state == 5); it++) {
                        if (state == 5) {
                            WordSlot32* sl = a.table32 + slot;
                            uint32_t r[8];
                            tw_ld256_cg(sl, r);
                            bool same1 = r[0] == k32[0] && r[1] == k32[1] && r[2] == k32[2] && r[3] == k32[3];
                            if (!same1 && (r[0] | r[1] | r[2] | r[3]) == 0) {
                                const uint32_t k1[4] = {k32[0], k32[1], k32[2], k32[3]};
                                uint32_t old[4];
                                tw_cas128(reinterpret_cast<WordSlot*>(sl), k1, old);
                                if ((old[0] | old[1] | old[2] | old[3]) == 0) {
                                    // owner: second half, then the flag
                                    asm volatile("st.global.relaxed.gpu.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(sl->k2), "r"(k32[4]), "r"(k32[5]), "r"(k32[6]), "r"(k32[7]) : "memory");
                                    __threadfence();
                                    asm volatile("st.global.relaxed.gpu.u32 [%0], %1;" :: "l"(&sl->c), "r"(1u) : "memory");
                                    state = 7; myslot = slot;
                                } else if (old[0] != k1[0] || old[1] != k1[1] || old[2] != k1[2] || old[3] != k1[3]) slot = (slot + 1) & a.table32_mask;
                                // (same first half inserted by somebody else meanwhile: look at this slot again next round)
                            } else if (same1) {
                                if (r[6] != 0) {                       // second half is there: compare it
                                    uint32_t q0, q1, q2, q3;
                                    asm volatile("ld.global.relaxed.gpu.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(q0), "=r"(q1), "=r"(q2), "=r"(q3) : "l"(sl->k2) : "memory");
                                    if (q0 == k32[4] && q1 == k32[5] && q2 == k32[6] && q3 == k32[7]) {
                                        myslot = slot;
                                        if (r[5] != 0) { v.a = r[4]; v.b = r[5]; v.c = 0; v.d = 0; state = 0; } else state = 6;
                                    } else slot = (slot + 1) & a.table32_mask;
                                }
                            } else slot = (slot + 1) & a.table32_mask;
                        }
                    }
                    if (state == 5) state = 3;                      // no slot within the limit: whole-warp path, uncached
                    uint32_t own32 = __ballot_sync(FULL, state == 7);
                    if (own32 && lane == 0) atomicAdd(a.n_uniq, (unsigned int)__popc(own32));
                    while (own32) {
                        const int l = __ffs(own32) - 1; own32 &= own32 - 1;
                        const WholeWarpOut r = tw_own_word32<MODEL>(m, a, sh, tw, __shfl_sync(FULL, p, l), __shfl_sync(FULL, len, l), __shfl_sync(FULL, myslot, l));
                        if (r.abort) warp_abort = true;
                        if ((int)lane == l) { v = r.v; state = 0; }
                    }
                    uint32_t pend32 = __ballot_sync(FULL, state == 6);
                    while (pend32) {
                        if (state == 6) {
                            uint32_t x, y;
                            asm volatile("ld.global.relaxed.gpu.v2.u32 {%0,%1}, [%2];" : "=r"(x), "=r"(y) : "l"(&a.table32[myslot].a) : "memory");
                            if (y != 0) { v.a = x; v.b = y; v.c = 0; v.d = 0; state = 0; }
                        }
                        pend32 = __ballot_sync(FULL, state == 6);
                        if (pend32) __nanosleep(64);              // the owner is running the model: leave it the issue slots
                    }
                }
                // words that need the whole warp: longer than 31 bytes, or no slot within the probe limit
                uint32_t todo = __ballot_sync(FULL, state == 3);
                while (todo) {
                    const int l = __ffs(todo) - 1; todo &= todo - 1;
                    const WholeWarpOut r = tw_whole_warp_word<MODEL>(m, a, bs.lut, sh, tw, s, __shfl_sync(FULL, p, l), __shfl_sync(FULL, len, l), a.lscratch + (size_t)(blockIdx.x * TW_WARPS + wid) * (4 * 256));
                    if (r.abort) warp_abort = true;
                    if ((int)lane == l) { v = r.v; state = 0; }
                }
                // words whose owner (another warp) was still computing
                uint32_t pend = __ballot_sync(FULL, state == 2);
                while (pend) {
                    if (state == 2) {
                        const uint4 q = tw_ld_value(a.table + myslot);
                        if (q.y != 0) { v.a = q.x; v.b = q.y; v.c = q.z; v.d = q.w; state = 0; }
                    }
                    pend = __ballot_sync(FULL, state == 2);
                    if (pend) __nanosleep(64);
                }
            }
            // ---- tokens + token prefix
            uint32_t nt = 0;
            const uint32_t flags = have ? (v.b & 0xE0000000u) : 0u;
            if (have) nt = ((v.b >> 16) & 0x1FFFu) - 1u;
            if (flags & (TW_ERRF | TW_LONGF)) nt = 0;
            uint32_t ex, tot;
            if (!__any_sync(FULL, nt > 3)) ex = tw_ballot_prefix<2>(nt, lt_mask, tot);
            else { const uint32_t inc = warp_incl_scan(nt); ex = inc - nt; tot = __shfl_sync(FULL, inc, 31); }
            const uint32_t dst = tbase + run + ex;                  // stream position of the word's first token
            if (can_store && nt && !(flags & TW_POOLF)) {
                // (the word's position in the slice goes into TW_REC_WIDE / TW_REC_WORD records only: it is read by the hf_compat
                // mode of pass B that reports offsets relative to the document; k, the word's index, into TW_REC_WORD records)
                tw_put_token<REC>(a.tok, dst, v.a, v.b & 0xFFFFu, p << 16, k);
                if (nt == 2) tw_put_token<REC>(a.tok, dst + 1, v.c, v.d & 0xFFFFu, p << 16, k);
            }
            // words with three or more tokens: listed now, copied from the pool at the end of the slice
            const uint32_t pooled = __ballot_sync(FULL, can_store && nt && (flags & TW_POOLF));
            if (pooled) {
                const uint32_t np = __popc(pooled);
                if (n_pl + np > 32) { tw_flush_pooled<REC>(a, sh.plist, n_pl); n_pl = 0; }
                if ((pooled >> lane) & 1u) sh.plist[n_pl + __popc(pooled & lt_mask)] = make_uint4(v.a, nt, dst, (p << 16) | (REC == TW_REC_WORD ? k : 0u));
                n_pl += np;
            }
            if (__any_sync(FULL, flags & (TW_ERRF | TW_LONGF))) {
                if (flags & TW_ERRF) atomicMin(a.errw, ((unsigned long long)(slice_base + p) << 8) | (MODEL == TKZ_MODEL_BPE ? TKZ_ECODE_UTF8 : TKZ_ECODE_UNK));
                // long words of the slice, in text order: position, length, index of insertion in the slice's token run
                const uint32_t lm = __ballot_sync(FULL, (flags & TW_LONGF) != 0);
                if (flags & TW_LONGF) {
                    const uint32_t j = n_long_here + __popc(lm & lt_mask);
                    if (j < TW_MAX_SLICE_LONG) { sh.lbuf[j][0] = p | (REC == TW_REC_WORD ? k << 16 : 0u); sh.lbuf[j][1] = v.a; sh.lbuf[j][2] = run + ex; }
                }
                n_long_here += __popc(lm);
            }
            if (have) sh.wlist[k] = (uint16_t)(run + ex);      // (the round's wlist entries were read at its top, before the votes)
            run += tot;
        }
        if (n_pl) tw_flush_pooled<REC>(a, sh.plist, n_pl);
        if (can_store) tcur += run;
        // long words -> one contiguous run of the long list
        uint32_t lfirst = 0;
        if (n_long_here) {
            if (n_long_here > TW_MAX_SLICE_LONG) { n_long_here = TW_MAX_SLICE_LONG; warp_abort = true; }   // cannot happen (each is > 255 bytes)
            if (lane == 0) lfirst = atomicAdd(a.n_long, n_long_here);
            lfirst = __shfl_sync(FULL, lfirst, 0);
            __syncwarp();
            if (lfirst + n_long_here > a.long_cap) { warp_abort = true; n_long_here = 0; }
            else if (lane < n_long_here) {
                const uint32_t st = (uint32_t)(slice_base + (REC == TW_REC_WORD ? sh.lbuf[lane][0] & 0xFFFFu : sh.lbuf[lane][0]));
                a.long_start[lfirst + lane] = st; a.long_end[lfirst + lane] = st + sh.lbuf[lane][1];
                a.long_slice[lfirst + lane] = s; a.long_ins[lfirst + lane] = sh.lbuf[lane][2];
                if (REC == TW_REC_WORD) a.long_k[lfirst + lane] = sh.lbuf[lane][0] >> 16;
            }
        }
        if (lane == 0) {
            a.slice_tok_off[s] = tbase;
            a.slice_ntok_inline[s] = can_store ? run : 0u;
            a.slice_ntok[s] = run;
            a.slice_long[s] = (lfirst << 3) | n_long_here;
            if (REC == TW_REC_WORD) a.slice_nword[s] = nW;
        }
        __syncwarp();
        // ---- token prefix at every document start inside the slice
        {
            const uint32_t dlo = sh.doc_lo_hi[0], dhi = sh.doc_lo_hi[1];
            for (uint32_t d = dlo + lane; d < dhi; d += 32) {
                const uint32_t q = (uint32_t)(__ldg(a.doc_off + d) - (uint64_t)s * TW_SLICE);
                const uint32_t sg = q >> 5;
                const uint32_t idx = sh.seg_wex[sg] + __popc(sh.seg_smask[sg] & ((1u << (q & 31u)) - 1u));
                a.doc_tok_local[d] = idx < nW ? (uint32_t)sh.wlist[idx] : run;
                if (REC == TW_REC_WORD) a.doc_word_local[d] = idx;
            }
        }
        __syncwarp();
    }
    if (lane == 0 && words_total) atomicAdd(a.n_words, (unsigned long long)words_total);
    if (__any_sync(FULL, warp_abort) && lane == 0) atomicExch(a.abort_flag, 1u);
}

// after the word-list kernels: the tokens of every long word join its tile's count and the token prefix of the documents
// that start behind it in the same tile
__global__ void long_fix_kernel(const uint32_t* __restrict__ long_start, const uint32_t* __restrict__ long_slice, const uint32_t* __restrict__ long_ntok,
                                uint32_t n_long, const uint32_t* __restrict__ tile_doc_lo, const uint64_t* __restrict__ doc_off,
                                uint32_t* tile_ntok, uint32_t* doc_tok_local, unsigned long long* long_tok_total) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_long) return;
    const uint32_t n = long_ntok[i];
    if (n == TKZ_NONE || n == 0) return;
    const uint32_t tile = long_slice[i];
    atomicAdd(tile_ntok + tile, n);
    atomicAdd(long_tok_total, (unsigned long long)n);
    const uint64_t pos = long_start[i];
    for (uint32_t d = tile_doc_lo[tile]; d < tile_doc_lo[tile + 1]; d++) if (doc_off[d] > pos) atomicAdd(doc_tok_local + d, n);
}

// ------------------------------------------------------------------ pass B
struct SliceEmitArgs {
    const uint64_t* doc_off; uint32_t n_docs; uint32_t n_slices; const uint32_t* slice_doc_lo;
    const void* tok;                              // the token stream (records of the kind TW_REC_*)
    const uint32_t* slice_tok_off; const uint32_t* slice_ntok_inline; const uint32_t* slice_long;
    const uint32_t* slice_tokbase;                // exclusive scan of the slice token counts (n_slices + 1)
    const uint32_t* long_start; const uint32_t* long_ins; const uint32_t* long_ntok;
    const uint32_t* pool_id; const uint32_t* pool_s; const uint32_t* pool_e;
    const uint32_t* doc_tok_local;
    const uint32_t* doc_tok_start;                // !PLAIN: global real-token index at each document start (n_docs + 1)
    unsigned long long* doc_tok_off;              // PLAIN: written here; !PLAIN: read (CSR after truncate / pad)
    unsigned long long* errw; uint32_t err_code;
    BigList big;
    // TW_REC_WORD: exclusive scan of the words that start in each slice, global index of each document's first word, the long
    // words' indices in their slice's word list
    const uint32_t* slice_wordbase; const uint32_t* doc_word_base; const uint32_t* long_k;
};

// one token of the stream -> the arrays the call asked for.  OUTS = the TKZ_OUT_* mask when known at compile time
// (ids only / ids + offsets + attention), 0 = read it from the parameters.  WID (TW_REC_WORD records): id carries the word's
// index in its slice's word list in bits 22.., wb = the slice's first word relative to the document's
template <uint32_t OUTS, bool WID = false>
__device__ __forceinline__ void te_put(const EmitParams& p, const EmitOut& o, unsigned long long dst, uint32_t id, uint32_t of, uint32_t hs, uint32_t wb = 0) {
    const uint32_t outputs = OUTS ? OUTS : p.outputs;
    if (WID) { o.word_ids[dst] = wb + (id >> 22); id &= 0x3FFFFFu; }
    uint32_t s = of & 0xFFu, e = (of >> 8) & 0xFFu, ty = 0u;
    if (p.hf_flags) {                                            // hf_compat (tkz_emit.cuh): document-relative offsets, the sequence's type id
        if (p.hf_flags & 2u) { const uint32_t b = hs + (of >> 16); s += b; e += b; }
        if (p.hf_flags & 1u) ty = p.seq_type;
    }
    if (outputs & 64u) o.ids16[dst] = (uint16_t)id; else o.ids[dst] = id;
    if (outputs & 2u) reinterpret_cast<uint2*>(o.offsets)[dst] = make_uint2(s, e);
    if (outputs & 4u) o.attention[dst] = 1u;
    if (outputs & 8u) o.type_ids[dst] = ty;
    if (outputs & 16u) o.special[dst] = 0u;
    if (outputs & 32u) o.offsets16[dst] = (uint16_t)of;
    if (outputs & 128u) o.spans[dst] = make_uint4(id, s, e, ty & 0xFFu);
}

// Pass B reads the token stream through two windows of TE_WIN bytes per warp in shared memory, filled by bulk copies
// (cp.async.bulk + mbarrier, as pass A stages its text).  While the warp writes the tokens of one window the next one is
// in flight: the rest of the slice's run, else the first window of the warp's next slice.  A window starts at the 16-byte
// boundary at or below the first record asked for, so a run needs no alignment in the stream; the neighbouring records a
// window holds as well are never written out.  (B200, c2b 1 GiB: per-lane loads of 4 records, 4 in flight, issued only
// after the previous slice was written, took 1.20 ms of pass B; see DESIGN 4.1 for this version.)
constexpr uint32_t TE_WIN = 1024;

__shared__ __align__(128) unsigned char te_smem[TW_WARPS][2 * TE_WIN + 16];   // per warp: two windows, their mbarriers

template <int REC>
struct TeWindows {
    static constexpr uint32_t RB = (REC == TW_REC_WIDE || REC == TW_REC_WORD) ? 8 : (REC == TW_REC_ID16 ? 2 : 4);   // bytes per record
    static constexpr uint32_t RPG = 16 / RB, RPW = TE_WIN / RB;                             // records per 16 bytes, per window
    uint32_t cur, clo, chi;              // the window being read and the records [clo, chi) it holds
    uint32_t nlo, nhi, npend;            // the other window: its records, whether its copy is in flight
    uint32_t phase;                      // parity bits of the two mbarriers
    uint32_t run_end, next_lo, next_hi;  // end of the current slice's run; the run of the warp's next slice

    __device__ __forceinline__ unsigned char* win() const { return te_smem[threadIdx.x >> 5]; }
    __device__ __forceinline__ unsigned long long* bar() const { return reinterpret_cast<unsigned long long*>(win() + 2 * TE_WIN); }
    // records [lo, hi) of the stream tok (as many as fit) into the other window; warp-uniform, that window is idle
    __device__ __forceinline__ void issue(const void* tok, uint32_t lo, uint32_t hi) {
        const uint32_t b = cur ^ 1u, a0 = lo & ~(RPG - 1u), a1 = min(a0 + RPW, (hi + RPG - 1u) & ~(RPG - 1u));
        nlo = a0; nhi = a1; npend = 1;
        __syncwarp();                    // every lane is done reading the window
        if (lane_id() == 0) tw_bulk_load(win() + b * TE_WIN, static_cast<const unsigned char*>(tok) + (size_t)a0 * RB, (a1 - a0) * RB, bar() + b);
    }
    // the copy in flight becomes the window being read; then the next window this warp will need goes in flight
    __device__ __forceinline__ void advance(const void* tok) {
        const uint32_t b = cur ^ 1u;
        tw_mbar_wait(bar() + b, (phase >> b) & 1u);
        phase ^= 1u << b;
        cur = b; clo = nlo; chi = nhi; npend = 0;
        if (chi < run_end) issue(tok, chi, run_end);
        else if (next_lo < next_hi) issue(tok, next_lo, next_hi);
    }
    // make the window being read hold record r of the current slice's run (warp-uniform)
    __device__ __forceinline__ void ensure(const void* tok, uint32_t r) {
        if (r - clo < chi - clo) return;
        if (npend && r - nlo < nhi - nlo) { advance(tok); return; }
        if (npend) {                     // a window that is not needed: drained.  (The plain kernel asks for a slice's records
                                         // in increasing order, starting at its run, so it never gets here; kept so that any
                                         // order of requests stays correct.)
            const uint32_t b = cur ^ 1u;
            tw_mbar_wait(bar() + b, (phase >> b) & 1u);
            phase ^= 1u << b; npend = 0;
        }
        issue(tok, r, run_end);
        advance(tok);
    }
    __device__ __forceinline__ void drain() {
        if (npend) { const uint32_t b = cur ^ 1u; tw_mbar_wait(bar() + b, (phase >> b) & 1u); npend = 0; }
        __syncwarp();
    }
};

// record q of a window -> (id, start | end << 8 [| position << 16]), the form te_put takes
template <int REC>
__device__ __forceinline__ void te_rec(const unsigned char* w, uint32_t q, uint32_t& id, uint32_t& of) {
    if (REC == TW_REC_WIDE || REC == TW_REC_WORD) { const uint2 r = reinterpret_cast<const uint2*>(w)[q]; id = r.x; of = r.y; }
    else if (REC == TW_REC4) { const uint32_t r = reinterpret_cast<const uint32_t*>(w)[q]; id = r & 0xFFFFu; of = r >> 16; }
    else if (REC == TW_REC_ID16) { id = reinterpret_cast<const uint16_t*>(w)[q]; of = 0; }
    else { id = reinterpret_cast<const uint32_t*>(w)[q]; of = 0; }
}

// ids + offsets + attention of 4 tokens at a 4-aligned destination slot: 16-byte stores (offsets: two of them)
__device__ __forceinline__ void te_put4(const EmitParams& p, const EmitOut& o, unsigned long long dst, const uint32_t (&id)[4], const uint32_t (&of)[4],
                                        uint32_t hs) {
    uint32_t s[4], e[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
        s[u] = of[u] & 0xFFu; e[u] = (of[u] >> 8) & 0xFFu;
        if (p.hf_flags & 2u) { const uint32_t b = hs + (of[u] >> 16); s[u] += b; e[u] += b; }
    }
    *reinterpret_cast<uint4*>(o.ids + dst) = make_uint4(id[0], id[1], id[2], id[3]);
    reinterpret_cast<uint4*>(o.offsets + 2 * dst)[0] = make_uint4(s[0], e[0], s[1], e[1]);
    reinterpret_cast<uint4*>(o.offsets + 2 * dst)[1] = make_uint4(s[2], e[2], s[3], e[3]);
    *reinterpret_cast<uint4*>(o.attention + dst) = make_uint4(1u, 1u, 1u, 1u);
}

// n tokens whose records start at index q0 of window w -> destination slots d0 .. d0 + n - 1.  Ids + offsets + attention:
// 4 tokens per lane at 4-aligned slots, the head and tail groups that the range only partly covers token by token (source
// and destination alignment differ freely: the records are read from shared memory at any index).  The generic form:
// te_put per token.
template <uint32_t OUTS, int REC>
__device__ __forceinline__ void te_store(const EmitParams& p, const EmitOut& o, const unsigned char* w, uint32_t q0, uint32_t n, unsigned long long d0,
                                         uint32_t hs) {
    constexpr bool VEC = OUTS == 7u;
    constexpr uint32_t U = 4;
    const uint32_t lane = lane_id();
    if (!VEC) {
        for (uint32_t k = lane; k < n; k += 32) { uint32_t id, of; te_rec<REC>(w, q0 + k, id, of); te_put<OUTS, REC == TW_REC_WORD>(p, o, d0 + k, id, of, hs); }
        return;
    }
    const uint32_t head = (uint32_t)d0 & (U - 1u);          // slots of the first group before d0
    const uint32_t ng = (head + n + U - 1u) / U;
    for (uint32_t g = lane; g < ng; g += 32) {
        const uint32_t k0 = g * U - head;                   // (mod 2^32) token of the group's first slot
        if ((g > 0 || head == 0) && k0 + U <= n) {
            uint32_t id[U], of[U];
#pragma unroll
            for (uint32_t u = 0; u < U; u++) te_rec<REC>(w, q0 + k0 + u, id[u], of[u]);
            te_put4(p, o, d0 + k0, id, of, hs);
        } else {
#pragma unroll
            for (uint32_t u = 0; u < U; u++) {
                const uint32_t k = k0 + u;
                if (k < n) { uint32_t id, of; te_rec<REC>(w, q0 + k, id, of); te_put<OUTS>(p, o, d0 + k, id, of, hs); }
            }
        }
    }
}

// which kernels take the staged copy: without truncation / padding, ids + offsets + attention (16 B per token) and the
// generic form.  The rest keep per-lane loads at 8 (5) blocks per SM, which measured faster for them (B200, 1000 W):
// c2b 1 GiB pass B ids only 0.345 ms against 0.384 staged, ids16 + packed offsets 0.466 against 0.526; the c3 hf_compat
// step 32.6 ms against 33.4 with the staged truncation / padding form (4 blocks per SM, 8-byte records spill there)
template <bool PLAIN, uint32_t OUTS>
__host__ __device__ constexpr bool te_staged() { return PLAIN && (OUTS == 7u || OUTS == 0u); }

// copies the stream tokens [j0, j1) of a slice whose run starts at stream position src to dst0 + (j - j0): window by
// window, or with TE_U loads in flight per lane for the forms that are not staged
// (wb: see te_put; TW_REC_WORD records are never staged)
template <bool STAGED, uint32_t OUTS, int REC>
__device__ __forceinline__ void te_copy(TeWindows<REC>& w, const void* tok, const EmitParams& p, const EmitOut& o, uint32_t src, uint32_t j0, uint32_t j1,
                                        unsigned long long dst0, uint32_t hs = 0, uint32_t wb = 0) {
    if (!STAGED) {
        const uint32_t lane = lane_id();
        constexpr int TE_U = 4;                     // B200, c2b 1 GiB: pass B 1.42 ms with 2, 1.25 ms with 4 or 8 (8-byte records)
        for (uint32_t j = j0 + lane; j < j1; j += 32 * TE_U) {
            uint32_t id[TE_U], of[TE_U];
#pragma unroll
            for (int u = 0; u < TE_U; u++) { id[u] = 0; of[u] = 0; }
#pragma unroll
            for (int u = 0; u < TE_U; u++) if (j + 32 * u < j1) {
                const size_t i = (size_t)src + j + 32 * u;
                if (REC == TW_REC_WIDE || REC == TW_REC_WORD) { const uint2 r = __ldg(static_cast<const uint2*>(tok) + i); id[u] = r.x; of[u] = r.y; }
                else if (REC == TW_REC4) { const uint32_t r = __ldg(static_cast<const uint32_t*>(tok) + i); id[u] = r & 0xFFFFu; of[u] = r >> 16; }
                else if (REC == TW_REC_ID16) id[u] = __ldg(static_cast<const uint16_t*>(tok) + i);
                else id[u] = __ldg(static_cast<const uint32_t*>(tok) + i);
            }
#pragma unroll
            for (int u = 0; u < TE_U; u++) if (j + 32 * u < j1) te_put<OUTS, REC == TW_REC_WORD>(p, o, dst0 + (j + 32 * u - j0), id[u], of[u], hs, wb);
        }
        return;
    }
    uint32_t r = src + j0;
    const uint32_t r1 = src + j1;
    while (r < r1) {
        w.ensure(tok, r);
        const uint32_t re = min(r1, w.chi);
        te_store<OUTS, REC>(p, o, w.win() + w.cur * TE_WIN, r - w.clo, re - r, dst0 + (r - (src + j0)), hs);
        r = re;
    }
}

// PLAIN = no truncation and no padding: the output is the plain concatenation of all tokens in text order, so a token's
// destination is its global index.  Otherwise the tokens of the slice are cut by the documents that meet the slice.
// REC: the token stream's record kind, as pass A wrote it (TW_REC_WORD: !PLAIN, OUTS = 0 only).
// Staged forms: 4 blocks of 8 warps per SM (64 registers, no spill).  At 5 blocks (48 registers) and 6 (40) they spill, and
// pass B measured 1.11 and 1.17 ms against 0.99 (B200, c2b 1 GiB): the windows in flight hide the loads without more warps.
template <bool PLAIN, uint32_t OUTS, int REC>
__global__ void __launch_bounds__(TW_THREADS, te_staged<PLAIN, OUTS>() ? 4 : (PLAIN ? 8 : 5)) slice_emit_kernel(const __grid_constant__ SliceEmitArgs a, const __grid_constant__ EmitParams p,
                                                                const __grid_constant__ EmitOut o) {
    constexpr bool STAGED = te_staged<PLAIN, OUTS>();
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = lane_id(), wid = threadIdx.x >> 5;
    const uint32_t stride = gridDim.x * TW_WARPS;
    TeWindows<REC> w;
    if (STAGED && lane == 0) { tw_mbar_init(w.bar()); tw_mbar_init(w.bar() + 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncwarp();
    w.cur = 0; w.clo = w.chi = 0; w.nlo = w.nhi = 0; w.npend = 0; w.phase = 0;
    // slice metadata is fetched one slice ahead, two for the staged forms (the token window of the next slice is issued while
    // this one is written):
    // lanes 0..6 hold ntok_inline, tok_off, tokbase, tokbase[+1], long, doc_lo, doc_lo[+1]
    auto load_meta = [&](uint32_t s) -> uint32_t {
        if (s >= a.n_slices || lane >= 7) return 0u;
        const uint32_t* src = lane == 0 ? a.slice_ntok_inline + s : (lane == 1 ? a.slice_tok_off + s : (lane < 4 ? a.slice_tokbase + s + (lane - 2)
                              : (lane == 4 ? a.slice_long + s : a.slice_doc_lo + s + (lane - 5))));
        return __ldg(src);
    };
    uint32_t s = blockIdx.x * TW_WARPS + wid;
    uint32_t meta = load_meta(s), meta_next = STAGED ? load_meta(s + stride) : 0u;
    for (; s < a.n_slices; s += stride) {
        const uint32_t ntok = __shfl_sync(FULL, meta, 0);
        const uint32_t src = __shfl_sync(FULL, meta, 1);
        const uint32_t base = __shfl_sync(FULL, meta, 2), base_next = __shfl_sync(FULL, meta, 3);
        const uint32_t lg = __shfl_sync(FULL, meta, 4);
        const uint32_t d_lo = __shfl_sync(FULL, meta, 5), d_hi = __shfl_sync(FULL, meta, 6);
        if (STAGED) { meta = meta_next; meta_next = load_meta(s + 2 * stride); }
        else meta = load_meta(s + stride);
        if (STAGED) { w.run_end = src + ntok; w.next_lo = __shfl_sync(FULL, meta, 1); w.next_hi = w.next_lo + __shfl_sync(FULL, meta, 0); }
        if (PLAIN) {
            if (lg == 0) te_copy<STAGED, OUTS, REC>(w, a.tok, p, o, src, 0, ntok, base);
            else {
                // pieces: inline tokens up to the next long word's insertion index, then the long word (from the pool)
                uint32_t j = 0; unsigned long long g = base;
                const uint32_t lf = lg >> 3, ln = lg & 7u;
                for (uint32_t i = 0; i <= ln; i++) {
                    const uint32_t jn = i < ln ? __ldg(a.long_ins + lf + i) : ntok;
                    te_copy<STAGED, OUTS, REC>(w, a.tok, p, o, src, j, jn, g);
                    g += jn - j; j = jn;
                    if (i < ln) {
                        uint32_t cnt = __ldg(a.long_ntok + lf + i);
                        const uint32_t sp = __ldg(a.long_start + lf + i);
                        if (cnt == TKZ_NONE) { if (lane == 0) atomicMin(a.errw, ((unsigned long long)sp << 8) | a.err_code); cnt = 0; }
                        bool queued = false;
                        if (cnt > EMIT_BIG) { if (lane == 0) queued = big_push(a.big, sp, cnt, g); queued = __shfl_sync(FULL, queued, 0); }
                        if (!queued) for (uint32_t q = lane; q < cnt; q += 32) emit_real(p, o, g + q, a.pool_id[sp + q], a.pool_s[sp + q], a.pool_e[sp + q]);
                        g += cnt;
                    }
                }
            }
            for (uint32_t d = d_lo + lane; d < d_hi; d += 32) a.doc_tok_off[d] = (unsigned long long)base + __ldg(a.doc_tok_local + d);
        } else {
            // documents that own tokens of this slice: d_lo - 1 (continuing from an earlier slice) and those starting here
            if (base_next == base) continue;
            const uint32_t lf = lg >> 3, ln = lg & 7u;
            const uint32_t d_first = d_lo ? d_lo - 1 : 0;
            constexpr bool WID = REC == TW_REC_WORD;
            const uint32_t swb = WID ? __ldg(a.slice_wordbase + s) : 0u;                    // global index of the slice's first word
            for (uint32_t dc = d_first; dc < d_hi && dc < a.n_docs; dc += 31) {
                // lane l holds the token start of document dc + l (32 values: 31 documents and the end of the last one)
                const uint32_t dl = dc + lane;
                const uint32_t my_ds = dl <= a.n_docs ? __ldg(a.doc_tok_start + dl) : 0xFFFFFFFFu;
                const unsigned long long my_dto = dl < a.n_docs ? a.doc_tok_off[dl] : 0ull;
                const uint32_t my_dbyte = (p.hf_flags & 2u) && dl < a.n_docs ? (uint32_t)a.doc_off[dl] : 0u;     // hf_compat: byte position of the document
                const uint32_t my_wb = WID && dl < a.n_docs ? swb - __ldg(a.doc_word_base + dl) : 0u;           // (mod 2^32) the slice's first word in the document
                const uint32_t nd_here = min(31u, min(d_hi, a.n_docs) - dc);
                for (uint32_t e = 0; e < nd_here; e++) {
                    const uint32_t ds = __shfl_sync(FULL, my_ds, e), dn = __shfl_sync(FULL, my_ds, e + 1);
                    const unsigned long long dto = __shfl_sync(FULL, my_dto, e);
                    uint32_t g0 = max(ds, base), g1 = min(dn, base_next);      // real-token range of the document inside this slice
                    if (g0 >= g1) continue;
                    unsigned long long kept;
                    const unsigned long long olen = doc_out_len(p, (unsigned long long)(dn - ds), &kept);
                    const unsigned long long shift = ((p.has_pad && p.pad_left) ? olen - kept - tpl_added(p) : 0) + ((p.hf_flags & 1u) ? p.n_pre : 0u);
                    if ((unsigned long long)(g1 - ds) > kept) g1 = ds + (uint32_t)kept;             // truncation
                    if (g0 >= g1) continue;
                    const unsigned long long dbase = dto + shift;                                    // destination of the document's token 0
                    const uint32_t dbyte = __shfl_sync(FULL, my_dbyte, e);
                    const uint32_t hs = s * TW_SLICE - dbyte;                                        // (mod 2^32) slice start relative to the document
                    const uint32_t wb = WID ? __shfl_sync(FULL, my_wb, e) : 0u;
                    if (ln == 0) te_copy<STAGED, OUTS, REC>(w, a.tok, p, o, src, g0 - base, g1 - base, dbase + (g0 - ds), hs, wb);
                    else {
                        // slice-local real index r = g - base; pieces as in the PLAIN case, cut to [g0, g1)
                        uint32_t j = 0, r = 0;
                        for (uint32_t i = 0; i <= ln; i++) {
                            const uint32_t jn = i < ln ? __ldg(a.long_ins + lf + i) : ntok;
                            {   // inline piece: stream tokens [j, jn) = real indices [r, r + jn - j)
                                const uint32_t lo = max(g0 - base, r), hi2 = min(g1 - base, r + (jn - j));
                                if (lo < hi2) te_copy<STAGED, OUTS, REC>(w, a.tok, p, o, src, j + (lo - r), j + (hi2 - r), dbase + (base + lo - ds), hs, wb);
                            }
                            r += jn - j; j = jn;
                            if (i < ln) {
                                uint32_t cnt = __ldg(a.long_ntok + lf + i);
                                const uint32_t sp = __ldg(a.long_start + lf + i);
                                if (cnt == TKZ_NONE) { if (lane == 0) atomicMin(a.errw, ((unsigned long long)sp << 8) | a.err_code); cnt = 0; }
                                const uint32_t lo = max(g0 - base, r), hi2 = min(g1 - base, r + cnt);
                                if (lo < hi2) {
                                    const uint32_t c2 = hi2 - lo, sp2 = sp + (lo - r);
                                    const unsigned long long dd = dbase + (base + lo - ds);
                                    bool queued = false;
                                    const uint32_t ls = (p.hf_flags & 2u) ? sp - dbyte : 0u;         // the long word's start within its document
                                    const uint32_t wid = WID ? wb + __ldg(a.long_k + lf + i) : 0u;
                                    if (c2 > EMIT_BIG) { if (lane == 0) queued = big_push<WID>(a.big, sp2, c2, dd, ls, wid); queued = __shfl_sync(FULL, queued, 0); }
                                    if (!queued) for (uint32_t q = lane; q < c2; q += 32) emit_real<WID>(p, o, dd + q, a.pool_id[sp2 + q], a.pool_s[sp2 + q] + ls, a.pool_e[sp2 + q] + ls, wid);
                                }
                                r += cnt;
                            }
                        }
                    }
                }
            }
        }
    }
    if (STAGED) w.drain();        // no bulk copy may still write into the block's shared memory when it exits
}

// per document: global token index of its start, real token count, output slot count (feeds the scan -> CSR offsets)
// (word ids: global index of its first word, from the word base of its slice; doc_word_base == nullptr: not asked for)
__global__ void doc_finish2_kernel(const uint64_t* __restrict__ doc_off, uint32_t n_docs, const uint32_t* __restrict__ tile_tokbase,
                                   const uint32_t* __restrict__ doc_tok_local, EmitParams p, uint32_t* __restrict__ doc_tok_start,
                                   uint32_t* __restrict__ doc_real, unsigned long long* __restrict__ doc_tok_off,
                                   const uint32_t* __restrict__ slice_wordbase, const uint32_t* __restrict__ doc_word_local, uint32_t* __restrict__ doc_word_base) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d > n_docs) return;
    const uint32_t s0 = tile_tokbase[(uint32_t)(doc_off[d] / TW_SLICE)] + doc_tok_local[d];
    doc_tok_start[d] = s0;
    if (doc_word_base) doc_word_base[d] = slice_wordbase[(uint32_t)(doc_off[d] / TW_SLICE)] + doc_word_local[d];
    if (d < n_docs) {
        const uint32_t s1 = tile_tokbase[(uint32_t)(doc_off[d + 1] / TW_SLICE)] + doc_tok_local[d + 1];
        const unsigned long long tr = s1 - s0;
        doc_real[d] = (uint32_t)tr;
        unsigned long long kept;
        doc_tok_off[d] = doc_out_len(p, tr, &kept);
    }
}

// warp-wide fill of n u32 slots at p with v: scalar head up to 16-byte alignment, 16-byte stores, scalar tail
__device__ __forceinline__ void warp_fill_u32(uint32_t* p, unsigned long long n, uint32_t v) {
    const uint32_t lane = lane_id();
    const uint32_t head = (uint32_t)((4u - (uint32_t)(((uintptr_t)p >> 2) & 3u)) & 3u);
    const unsigned long long h = head < n ? head : n;
    if (lane < h) p[lane] = v;
    const unsigned long long n4 = (n - h) >> 2;
    uint4* p4 = reinterpret_cast<uint4*>(p + h);
    for (unsigned long long i = lane; i < n4; i += 32) p4[i] = make_uint4(v, v, v, v);
    const unsigned long long done = h + (n4 << 2);
    if (done + lane < n) p[done + lane] = v;
}

// padding slots from per-document real counts (src/encoding.zig:407-414, 418-425), one warp per document.  WID: word ids
template <bool WID>
__global__ void __launch_bounds__(256) emit_pad_real_kernel(EmitParams p, EmitOut o, uint32_t n_docs, const uint32_t* __restrict__ doc_real,
                                                            const unsigned long long* __restrict__ doc_tok_off) {
    const uint32_t d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (d >= n_docs) return;
    unsigned long long kept;
    const unsigned long long olen = doc_out_len(p, doc_real[d], &kept);
    const unsigned long long full = kept + tpl_added(p);
    if (p.hf_flags & 1u) {
        // hf_compat: the template's special tokens around the kept tokens (lanes 0-3 prefix, 8-11 suffix)
        const uint32_t lane = lane_id();
        const unsigned long long b0 = doc_tok_off[d] + ((p.has_pad && p.pad_left) ? olen - full : 0);
        if (lane < p.n_pre) emit_special<WID>(p, o, b0 + lane, p.pre_id[lane], p.pre_type[lane]);
        if (lane >= 8 && lane - 8 < p.n_suf) emit_special<WID>(p, o, b0 + p.n_pre + kept + (lane - 8), p.suf_id[lane - 8], p.suf_type[lane - 8]);
    }
    if (olen == full) return;
    const unsigned long long base = doc_tok_off[d] + (p.pad_left ? 0 : full);
    const unsigned long long npad = olen - full;
    if (p.outputs & 64u) { uint16_t* q = o.ids16 + base; for (unsigned long long i = lane_id(); i < npad; i += 32) q[i] = (uint16_t)p.pad_id; }
    else warp_fill_u32(o.ids + base, npad, p.pad_id);
    if (p.outputs & 2u) warp_fill_u32(o.offsets + 2 * base, 2 * npad, 0u);
    if (p.outputs & 4u) warp_fill_u32(o.attention + base, npad, 0u);
    if (p.outputs & 8u) warp_fill_u32(o.type_ids + base, npad, p.pad_type_id);
    if (p.outputs & 16u) warp_fill_u32(o.special + base, npad, 1u);
    if (p.outputs & 32u) { uint16_t* q = o.offsets16 + base; for (unsigned long long i = lane_id(); i < npad; i += 32) q[i] = 0; }
    if (p.outputs & 128u) { uint4* q = o.spans + base; for (unsigned long long i = lane_id(); i < npad; i += 32) q[i] = make_uint4(p.pad_id, 0u, 0u, 0x0400u); }
    if (WID) warp_fill_u32(o.word_ids + base, npad, TKZ_NONE);
}

// hf_compat: only the template's special tokens (the padding slots were filled array-wide), one thread per document
template <bool WID>
__global__ void __launch_bounds__(256) emit_frame_kernel(EmitParams p, EmitOut o, uint32_t n_docs, const uint32_t* __restrict__ doc_real,
                                                         const unsigned long long* __restrict__ doc_tok_off) {
    const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_docs) return;
    unsigned long long kept;
    const unsigned long long olen = doc_out_len(p, doc_real[d], &kept);
    const unsigned long long b0 = doc_tok_off[d] + ((p.has_pad && p.pad_left) ? olen - kept - tpl_added(p) : 0);
    for (uint32_t i = 0; i < p.n_pre; i++) emit_special<WID>(p, o, b0 + i, p.pre_id[i], p.pre_type[i]);
    for (uint32_t i = 0; i < p.n_suf; i++) emit_special<WID>(p, o, b0 + p.n_pre + kept + i, p.suf_id[i], p.suf_type[i]);
}

// document of the first failing word (byte position in the error word) -> ctrl[4]
__global__ void err_doc_kernel(unsigned long long* ctrl, const uint64_t* doc_off, uint32_t n_docs) {
    const unsigned long long ew = ctrl[0];
    unsigned long long d = 0;
    if (ew != TKZ_ERRW_NONE && n_docs) {
        const uint64_t pos = ew >> 8;
        const uint32_t ub = upper_bound_u64(doc_off, 0, n_docs, pos);      // first document starting after pos
        d = ub ? ub - 1 : 0;
    }
    ctrl[4] = d;
}

}  // namespace tkz
