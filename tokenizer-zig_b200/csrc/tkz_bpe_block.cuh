// tkz_bpe_block.cuh -- K3 for long pre-tokens (whole documents, unbroken words): one thread block per word, merges
// scheduled by WINDOWED LOCAL MINIMA instead of one global-minimum pair type per round.
//
// Reference semantics (src/model/bpe.zig:214-253): repeat { pair type with the strictly smallest rank; merge all its
// occurrences left to right }.  The number of rounds grows with the word (one per distinct pair type merged), each round
// touching the whole word: O(rounds x length), hopeless for a 1 KiB..4 MiB "word".
//
// For a PROPER merge table (checked once at upload, tkz_api.cu): ranks unique, and every merge that PRODUCES a symbol has a
// lower rank than every merge that CONSUMES it.  Then
//   (1) a pair created by the merge of rank r has a rank > r, so the round order equals strict rank order: an occurrence
//       (a,b) of rank r gets merged unless a or b is consumed earlier by a merge of rank < r;
//   (2) a can only be consumed from the left, BEFORE round r, by a merge (X,a) of rank < r whose X is built, by merges of
//       even lower rank, from the symbols directly left of a; X spans at most wl = max nsym(X) over the table entries (X,a)
//       of rank < r current symbols, and the FIRST merge of that chain is a pair that is present NOW, inside that span, with
//       rank < r.  Symmetrically for b (wr over the entries (b,Z) of rank < r).  The windows are stored per table entry
//       (merge_win, built in tkz_api.cu); early merges join short symbols, so low ranks have windows of 1-3 symbols.
// So an occurrence at position i with rank r may merge immediately when no present pair in [i-wl, i+wr] has a smaller
// rank ("windowed local minimum") -- every such occurrence of the whole word merges in the same step.  The global minimum
// always qualifies, so every step makes progress; typical text needs one or two dozen steps independent of the word length.
// Pairs of two equal symbols (A,A) are decided per RUN of A, because a run pairs up from its start (aaaaa -> aa aa a):
//   * run-window rule (runs up to BB_RUN_WALK symbols): nothing of lower rank within wl pairs left of the run's first A, nor
//     within wr pairs from the pair of its last A on, where the entry's wl / wr also cover nsym(A) -- the span from which an A
//     that would join the run and shift the pairing could still be built.  Then the run is the same run in round r and is
//     paired up now, every second pair from its start;
//   * longer runs wait for a step in which nothing else can merge; (A,A) is then the minimum rank of the whole word and its runs
//     are paired up by the reference round (run starts by a block-wide max-scan).  The word's minimum is only computed then.
// Tables that are not proper (or have windows > 250) never reach this kernel: bpe_warp_kernel keeps the literal rounds.
//
// State per current symbol: id, index of its first initial symbol, cached rank + window of the pair with its right
// neighbour, head flag; in shared memory up to `CAP` symbols, else in the word's slices of global scratch arrays.
// The initial symbols' byte offsets stay in the pool (pool_s / pool_e) and give the final (start, end) of every token.
#pragma once
#include "tkz_bpe.cuh"
#include "tkz_common.cuh"

namespace tkz {

constexpr uint32_t BB_RUN_WALK = 32;        // equal-symbol runs up to this length are handled by the run-window rule

struct BlockBpeArgs {
    const uint8_t* text;
    const uint32_t* word_start;
    const uint32_t* word_end;
    uint32_t n_words;
    uint32_t min_len, max_len;            // this launch takes words with min_len <= byte length <= max_len
    uint32_t* pool_id; uint32_t* pool_s; uint32_t* pool_e; uint32_t* pool_rk;
    uint32_t* g_first; uint16_t* g_win; uint8_t* g_flag;     // global state for words above the shared-memory capacity
    uint32_t* word_ntok;
    unsigned int* work_counter;
    unsigned long long* errw;
    int sentinel_errors;
    const uint8_t* skip;                  // optional, per word: already tokenized by bpe_grid_kernel (tkz_bpe_grid.cuh)
};

template <int NT>
__device__ __forceinline__ uint32_t block_min_u32(uint32_t v, uint32_t* sh /* NT/32 */) {
    for (int d = 16; d > 0; d >>= 1) { const uint32_t t = __shfl_xor_sync(0xFFFFFFFFu, v, d); v = t < v ? t : v; }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    uint32_t r = 0xFFFFFFFFu;
#pragma unroll
    for (int w = 0; w < NT / 32; w++) { const uint32_t x = sh[w]; r = x < r ? x : r; }
    return r;
}
// inclusive max-scan over the block (values in thread order), one element per thread; `carry` = running max from before
template <int NT>
__device__ __forceinline__ uint32_t block_incl_maxscan(uint32_t v, uint32_t* sh /* NT/32 */, uint32_t carry) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= (uint32_t)d) v = t > v ? t : v; }
    __syncthreads();
    if (lane == 31) sh[wid] = v;
    __syncthreads();
    uint32_t base = carry;
    for (uint32_t w = 0; w < wid; w++) { const uint32_t x = sh[w]; base = x > base ? x : base; }
    return v > base ? v : base;
}

// NT threads, CAP symbols of shared-memory state (15 bytes each)
template <int NT, int CAP, int MINB = 1>
__global__ void __launch_bounds__(NT, MINB) bpe_block_kernel(DevModel m, BlockBpeArgs a) {
    extern __shared__ __align__(16) uint8_t bb_smem[];
    uint32_t* const s_id = reinterpret_cast<uint32_t*>(bb_smem);
    uint32_t* const s_first = s_id + CAP;
    uint32_t* const s_rk = s_first + CAP;
    uint16_t* const s_win = reinterpret_cast<uint16_t*>(s_rk + CAP);
    uint8_t* const s_flag = reinterpret_cast<uint8_t*>(s_win + CAP);
    __shared__ uint32_t sc[2 * (NT / 32 + 1)];
    __shared__ uint32_t red[NT / 32];
    __shared__ uint32_t s_w, s_cnt[4];
    const uint32_t t = threadIdx.x;

    for (;;) {
        __syncthreads();
        if (t == 0) s_w = atomicAdd(a.work_counter, 1u);
        __syncthreads();
        const uint32_t w = s_w;
        if (w >= a.n_words) break;
        const uint32_t ws = a.word_start[w], len = a.word_end[w] - ws;
        if (len < a.min_len || len > a.max_len) continue;
        if (a.skip && a.skip[w]) continue;
        const uint8_t* __restrict__ wt = a.text + ws;
        const bool in_smem = len <= (uint32_t)CAP;
        uint32_t* ids = in_smem ? s_id : a.pool_id + ws;
        uint32_t* first = in_smem ? s_first : a.g_first + ws;
        uint32_t* rk = in_smem ? s_rk : a.pool_rk + ws;
        uint16_t* win = in_smem ? s_win : a.g_win + ws;
        uint8_t* flag = in_smem ? s_flag : a.g_flag + ws;
        uint32_t* const ps = a.pool_s + ws;      // byte offsets of the INITIAL symbols (kept until the end)
        uint32_t* const pe = a.pool_e + ws;

        // ---------------- initial symbols (bpe.zig:185-211), NT bytes per step
        uint32_t n = 0, phase = 0;
        if (t == 0) s_cnt[0] = 0;                 // malformed flag
        __syncthreads();
        for (uint32_t c0 = 0; c0 < len; c0 += NT, phase ^= 1u) {
            const uint32_t p = c0 + t;
            uint32_t id = TKZ_NONE; int L = 0;
            if (p < len) {
                const uint32_t b0 = m.lut[__ldg(wt + p)];
                bool bad = false;
                if ((b0 & 0xC0) == 0x80) {
                    bool covered = false;
                    for (uint32_t back = 1; back <= 3 && back <= p; back++) {
                        const uint32_t q = m.lut[__ldg(wt + p - back)];
                        if ((q & 0xC0) != 0x80) { covered = (uint32_t)utf8_seq_len(q) > back; break; }
                    }
                    bad = !covered;
                } else {
                    L = utf8_seq_len(b0);
                    if (L == 0 || p + (uint32_t)L > len) bad = true;
                    uint32_t key = b0;
                    for (int j = 1; j < L && !bad; j++) {
                        const uint32_t bj = m.lut[__ldg(wt + p + j)];
                        if ((bj & 0xC0) != 0x80) bad = true;
                        key |= bj << (8 * j);
                    }
                    if (!bad) { id = char_lookup(m, key, L); if (id == TKZ_NONE && m.has_unk) id = m.unk_id; }
                }
                if (bad) s_cnt[0] = 1;
            }
            uint32_t tot;
            const uint32_t ex = block_excl_scan_bit<NT / 32>(id != TKZ_NONE, sc, phase, &tot);
            if (id != TKZ_NONE) { const uint32_t k = n + ex; ids[k] = id; first[k] = k; ps[k] = p; pe[k] = p + (uint32_t)L; }
            n += tot;
        }
        __syncthreads();
        if (s_cnt[0]) {
            // malformed UTF-8: exact sequential iterator by one thread (rare); invalid lead / truncated tail is an error
            if (t == 0) {
                const uint32_t k = bpe_init_sequential(m, GlobalLutSrc{m.lut, wt}, len, ids, ps, pe);
                s_cnt[1] = k;
                if (k != TKZ_NONE) for (uint32_t i = 0; i < k; i++) first[i] = i;
            }
            __syncthreads();
            n = s_cnt[1];
            if (n == TKZ_NONE) {
                if (t == 0) { if (a.sentinel_errors) a.word_ntok[w] = TKZ_NONE; else { report_error(a.errw, w, TKZ_ECODE_UTF8); a.word_ntok[w] = 0; } }
                continue;
            }
        }
        const uint32_t n0 = n;                    // number of initial symbols
        // ---------------- pair ranks + windows
        for (uint32_t i = t; i + 1 < n; i += NT) {
            uint32_t nid, wv = 0;
            const uint32_t r = merge_lookup_win(m, ids[i], ids[i + 1], &nid, &wv);
            rk[i] = r; win[i] = (uint16_t)wv;
        }
        __syncthreads();

        // ---------------- merge steps
        while (n > 1) {
            // A. heads by the window rules.  The word's minimum rank is NOT needed for them; it is only computed when no pair
            // qualifies, which means the minimum is an equal-symbol pair in a run beyond the walk limit (the global minimum of any
            // other kind always qualifies).  The runs of that pair are then paired up in a step of their own -- exactly the
            // reference round for them; everything near them has been waiting (their rank is inside its window), everything else
            // was free to go first (tests/test_windowed_schedule_model.py: lazy_long_runs).
            bool any_ranked = false, any_head = false;
            for (uint32_t i = t; i < n; i += NT) {
                bool head = false;
                if (i + 1 < n) {
                    const uint32_t r = rk[i];
                    any_ranked |= r != TKZ_NONE;
                    if (r != TKZ_NONE && ids[i] != ids[i + 1]) {
                        const uint32_t wv = win[i], wl = wv & 0xFFu, wr = wv >> 8;
                        const uint32_t lo = i > wl ? i - wl : 0;
                        uint32_t hi = i + wr; if (hi > n - 2) hi = n - 2;
                        head = true;
                        for (uint32_t j = lo; j < i && head; j++) head = rk[j] >= r;
                        for (uint32_t j = i + 1; j <= hi && head; j++) head = rk[j] >= r;
                        // an equal rank inside the window is another occurrence of the same pair: it cannot overlap (a != b)
                    } else if (r != TKZ_NONE) {
                        // (A, A): the window goes around the whole run of A (its extent is part of the decision: the run
                        // pairs up from its start).  Nothing of lower rank left of the run within wl pairs, nor from the pair
                        // of its last A on within wr pairs => no A of the run is consumed and no A joins it before round r
                        // (the entry's window also covers nsym(A), see tkz_api.cu), so the run pairs up NOW as it will then.
                        const uint32_t x = ids[i];
                        uint32_t s0 = i, e0 = i + 2, c = 0;
                        while (c < BB_RUN_WALK && s0 > 0 && ids[s0 - 1] == x) { s0--; c++; }
                        c = 0;
                        while (c < BB_RUN_WALK && e0 < n && ids[e0] == x) { e0++; c++; }
                        if (!(s0 > 0 && ids[s0 - 1] == x) && !(e0 < n && ids[e0] == x) && ((i - s0) & 1u) == 0) {
                            const uint32_t wv = win[i], wl = wv & 0xFFu, wr = wv >> 8;
                            const uint32_t lo = s0 > wl ? s0 - wl : 0;
                            uint32_t hi = e0 - 2 + wr; if (hi > n - 2) hi = n - 2;
                            head = true;
                            for (uint32_t j = s0; j > lo && head;) { --j; head = rk[j] >= r; }
                            for (uint32_t j = e0 - 1; j <= hi && head; j++) head = rk[j] >= r;
                        }
                    }
                }
                flag[i] = head ? 1 : 0;
                any_head |= head;
            }
            if (!__syncthreads_or(any_ranked)) break;                      // bpe.zig:232-234: no pair has a rank
            if (!__syncthreads_or(any_head)) {
                // the reference round for the word's minimum-rank pair (A, A): every run of A pairs up from its start
                uint32_t lmin = TKZ_NONE;
                for (uint32_t i = t; i + 1 < n; i += NT) { const uint32_t r = rk[i]; lmin = r < lmin ? r : lmin; }
                const uint32_t gmin = block_min_u32<NT>(lmin, red);
                uint32_t A = 0;
                if (t == 0) s_cnt[3] = TKZ_NONE;
                __syncthreads();
                for (uint32_t i = t; i + 1 < n; i += NT) if (rk[i] == gmin) atomicMin(&s_cnt[3], i);
                __syncthreads();
                A = ids[s_cnt[3]];
                uint32_t carry = 0;                                        // run start (index + 1 of the last non-A), running max
                for (uint32_t c0 = 0; c0 < n; c0 += NT) {
                    const uint32_t i = c0 + t;
                    const bool isA = i < n && ids[i] == A;
                    const uint32_t brk = (i < n && !isA) ? i + 1 : 0;       // position after a non-A symbol
                    const uint32_t rs = block_incl_maxscan<NT>(brk, red, carry);   // for an A at i: start of its run
                    if (i < n) flag[i] = (isA && ((i - rs) & 1u) == 0 && i + 1 < n && ids[i + 1] == A) ? 1 : 0;
                    __syncthreads();
                    if (t == NT - 1) s_cnt[1] = rs;
                    __syncthreads();
                    carry = s_cnt[1];
                }
            }
            __syncthreads();
            // A2. heads fetch their new id (stashed in rk: a head's cached rank is dead)
            for (uint32_t i = t; i + 1 < n; i += NT) if (flag[i]) { uint32_t nid = 0; merge_rank_lookup(m, ids[i], ids[i + 1], &nid); rk[i] = nid; }
            __syncthreads();
            // B. in-place compaction, NT symbols per step (writes never pass the reads of later chunks)
            uint32_t wpos = 0; phase = 0;
            for (uint32_t c0 = 0; c0 < n; c0 += NT, phase ^= 1u) {
                const uint32_t i = c0 + t;
                bool keep = false, head = false, next_head = false;
                uint32_t x = 0, f = 0, r = TKZ_NONE; uint16_t wv = 0;
                if (i < n) {
                    head = flag[i] != 0;
                    keep = !(i > 0 && flag[i - 1]);
                    next_head = (i + 1 < n) && flag[i + 1];
                    x = ids[i]; f = first[i]; r = rk[i]; wv = win[i];
                }
                uint32_t tot;
                const uint32_t ex = block_excl_scan_bit<NT / 32>(keep, sc, phase, &tot);          // barrier: all reads done
                if (keep) {
                    const uint32_t q = wpos + ex;
                    ids[q] = head ? r : x;                                  // r holds the new id for heads
                    first[q] = f;
                    rk[q] = (head || next_head) ? TKZ_DIRTY : r;
                    win[q] = wv;
                }
                wpos += tot;
            }
            n = wpos;
            __syncthreads();
            // C. ranks of the pairs a merge touched
            for (uint32_t i = t; i < n; i += NT) {
                if (i + 1 < n) {
                    if (rk[i] == TKZ_DIRTY) { uint32_t nid, wv = 0; const uint32_t r = merge_lookup_win(m, ids[i], ids[i + 1], &nid, &wv); rk[i] = r; win[i] = (uint16_t)wv; }
                } else rk[i] = TKZ_NONE;
            }
            __syncthreads();
        }

        // ---------------- result (bpe.zig:256-260): token i = initial symbols first[i] .. first[i+1]-1
        __syncthreads();
        for (uint32_t c0 = 0; c0 < n; c0 += NT) {
            const uint32_t i = c0 + t;
            uint32_t id = 0, s = 0, e = 0;
            if (i < n) {
                id = ids[i];
                const uint32_t f0 = first[i], f1 = (i + 1 < n) ? first[i + 1] : n0;
                s = ps[f0]; e = pe[f1 - 1];
            }
            __syncthreads();                                                // reads of this chunk before its writes
            if (i < n) { a.pool_id[ws + i] = id; ps[i] = s; pe[i] = e; }
        }
        if (t == 0) a.word_ntok[w] = n;
    }
}

}  // namespace tkz
