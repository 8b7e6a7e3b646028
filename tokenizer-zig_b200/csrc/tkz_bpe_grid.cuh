// tkz_bpe_grid.cuh -- K3 for HUGE pre-tokens (unbroken words / whole documents above the shared-memory capacity of
// bpe_block_kernel, up to MiBs): ALL such words of a batch are merged together by ONE cooperative grid, the windowed
// local-minimum schedule of tkz_bpe_block.cuh applied to their concatenated symbol array.
//
// Why: one thread block per huge word (global-memory state, ~1 us of latency per dependent pass) left a 4 MiB word alone
// on one SM for half a second while the other 147 SMs idled.  Here every step is a handful of streaming passes over the
// symbols of all huge words, spread over the whole grid, separated by grid-wide barriers: the cost is HBM traffic
// (~70 B per live symbol per step), independent of how the bytes are distributed over words.
//
// Reference semantics: src/model/bpe.zig:185-211 (initial symbols), :214-253 (merge rounds), :256-260 (tokens).  The
// schedule is exact for PROPER merge tables (see tkz_bpe_block.cuh for the argument; improper tables never get here):
//   * a pair (a, b), a != b, of rank r merges as soon as no present pair inside its (rank-aware) window [i - wl, i + wr]
//     has a smaller rank; windows never reach into a neighbouring word (the pair behind a word's last symbol carries the
//     reserved rank TKZ_BOUNDARY and stops the scan);
//   * a pair of two equal symbols (A, A) in a run of up to BG_WALK symbols follows the run-window rule of
//     tkz_bpe_block.cuh; in a longer run it merges only when its rank is the minimum over its whole word -- exactly the
//     reference's current round for that word -- and then the run pairs up from its start (bpe.zig:236-251: "do not
//     advance i after a merge" never re-matches because new_id != A in a proper table); starts of long runs come from a
//     grid-wide max-scan of run boundaries.  Other heads of the same word merge in the same step: none of them has the
//     (A, A) pair in its window.
// Steps: DENSE (two streaming passes H / K over the whole array, K compacts into the other buffer and re-ranks the pairs
// a merge touched) while many pairs still have a rank, then SPARSE (pair list, merges in place, dead marks) -- see the
// comments at the two loops.  Flags that steer all blocks are double-buffered by step parity and reset only a full grid
// barrier after their last reader.
//
// State per live symbol, ping-ponged between two buffers by the compaction of every step: id, byte offsets (start, end)
// inside the word, cached rank + window of the pair with the right neighbour, index of the word.  Words with malformed
// UTF-8 (sequential re-decode needed, bpe_init_sequential) are left to bpe_block_kernel: `done[w]` stays 0.
#pragma once
#include <cooperative_groups.h>

#include "tkz_bpe_block.cuh"

namespace tkz {
namespace cg = cooperative_groups;

#define TKZ_BOUNDARY 0xFFFFFFFDu          // cached "rank" of the position behind a word's last symbol
constexpr int BG_NT = 1024;
constexpr uint32_t BG_WALK = 32;          // equal-symbol runs up to this length find their start by walking left
constexpr uint32_t BG_SPARSE_DIV = 16;     // the sparse phase starts when fewer than n / 16 pairs still have a rank (a listed pair costs ~10x a streamed symbol)
constexpr uint32_t BG_SPARSE_WALK = 1024;  // same in the sparse phase (walks skip dead symbols); longer runs go back to the dense steps
constexpr uint32_t BG_PENDING = 0xFFFFFFFEu;   // head mark of an (A, A) pair that waits for the run scan

struct GridBpeArgs {
    const uint8_t* text;
    const uint32_t* word_start; const uint32_t* word_end;       // the launch's word list
    const uint32_t* hw;                   // huge word h -> index in the word list            (n_huge)
    const uint32_t* hbase;                // huge word h -> first byte in the concatenation   (n_huge + 1, last = M)
    uint32_t n_huge, M;
    uint32_t sparse_walk;                 // longest run walk of the sparse phase (TKZ_GRID_SPARSE_WALK)
    uint32_t* id[2]; uint32_t* s[2]; uint32_t* e[2]; uint32_t* rk[2]; uint32_t* wid[2]; uint16_t* win[2];
    uint32_t* hn;                         // per symbol: TKZ_NONE, BG_PENDING, or the new id of the pair it heads
    uint32_t* wmin[2];                    // per huge word: smallest pair rank (double-buffered by step parity)
    uint32_t* wstart;                     // per huge word: first symbol in the final array (n_huge + 1)
    uint8_t* wbad;                        // per huge word: malformed UTF-8 seen
    uint32_t* blk;                        // [0, 32 G) heads per warp part (init: [0, G) symbols per block), [32 G, 33 G) last run boundary per block
    uint32_t* dbg;                        // TKZ_GRID_DEBUG: per step (first 256) n, heads, ns in H, ns in K
    uint32_t* gs;                         // scalars: [1 + parity] a mergeable pair exists, [3 + parity] run scan needed
    uint32_t* pool_id; uint32_t* pool_s; uint32_t* pool_e;      // results, indexed by the word's byte position
    uint32_t* word_ntok; uint8_t* done;   // per word of the list
};

// sum of arr[0 .. b) and of arr[0 .. G), to every thread of the block; red = 64 u32 of shared memory
__device__ __forceinline__ void bg_prefix_total(const uint32_t* arr, uint32_t G, uint32_t b, uint32_t* red, uint32_t& before, uint32_t& total) {
    const uint32_t t = threadIdx.x, lane = t & 31, wid = t >> 5;
    uint32_t v = 0, vb = 0;
    for (uint32_t k = t; k < G; k += BG_NT) { const uint32_t x = __ldcg(arr + k); v += x; if (k < b) vb += x; }
    for (int d = 16; d > 0; d >>= 1) { v += __shfl_xor_sync(0xFFFFFFFFu, v, d); vb += __shfl_xor_sync(0xFFFFFFFFu, vb, d); }
    __syncthreads();
    if (lane == 0) { red[wid] = v; red[32 + wid] = vb; }
    __syncthreads();
    uint32_t tv = 0, tb = 0;
#pragma unroll
    for (int w = 0; w < BG_NT / 32; w++) { tv += red[w]; tb += red[32 + w]; }
    total = tv; before = tb;
}
__device__ __forceinline__ uint32_t bg_block_sum(uint32_t v, uint32_t* red) {
    const uint32_t t = threadIdx.x, lane = t & 31, wid = t >> 5;
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    uint32_t tv = 0;
#pragma unroll
    for (int w = 0; w < BG_NT / 32; w++) tv += red[w];
    return tv;
}
// max of arr[0 .. b)
__device__ __forceinline__ uint32_t bg_prefix_max(const uint32_t* arr, uint32_t b, uint32_t* red) {
    const uint32_t t = threadIdx.x, lane = t & 31, wid = t >> 5;
    uint32_t v = 0;
    for (uint32_t k = t; k < b; k += BG_NT) { const uint32_t x = __ldcg(arr + k); v = x > v ? x : v; }
    for (int d = 16; d > 0; d >>= 1) { const uint32_t y = __shfl_xor_sync(0xFFFFFFFFu, v, d); v = y > v ? y : v; }
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    uint32_t tv = 0;
#pragma unroll
    for (int w = 0; w < BG_NT / 32; w++) { const uint32_t x = red[w]; tv = x > tv ? x : tv; }
    return tv;
}

__global__ void __launch_bounds__(BG_NT, 1) bpe_grid_kernel(const __grid_constant__ DevModel m, const __grid_constant__ GridBpeArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ uint32_t sc[2 * (BG_NT / 32 + 1)];
    __shared__ uint32_t red[64];
    __shared__ uint32_t s_x;
    const uint32_t t = threadIdx.x, b = blockIdx.x, G = gridDim.x;
    const uint32_t gt = b * BG_NT + t, gstride = G * BG_NT;
    const uint32_t FULL = 0xFFFFFFFFu;
    uint32_t phase = 0;
    // contiguous range of block b over n elements, a multiple of 4 * BG_NT long (so that a warp's 1/32 of it is a multiple of 128)
    auto range = [&](uint32_t n, uint32_t& lo, uint32_t& hi) {
        const unsigned long long per = ((((unsigned long long)n + G - 1) / G + 4 * BG_NT - 1) / (4 * BG_NT)) * (4 * BG_NT);
        const unsigned long long l = per * b, h = l + per;
        lo = (uint32_t)(l < n ? l : n); hi = (uint32_t)(h < n ? h : n);
        return per;
    };

    // ---------------- per-word state; initial symbols at their byte positions in buffer 0 (bpe.zig:185-211)
    for (uint32_t w = gt; w < a.n_huge; w += gstride) { a.wmin[0][w] = TKZ_NONE; a.wmin[1][w] = TKZ_NONE; a.wbad[w] = 0; }
    if (gt < 32) a.gs[gt] = 0;
    uint32_t lo, hi;
    range(a.M, lo, hi);
    {
        uint32_t cnt = 0;
        for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT) {
            const uint32_t g = c0 + t;
            if (t == 0) {                                                // last huge word that starts at or before c0
                uint32_t l = 0, h = a.n_huge;
                while (l < h) { const uint32_t mid = l + ((h - l) >> 1); if (__ldg(a.hbase + mid) <= c0) l = mid + 1; else h = mid; }
                s_x = l - 1;
            }
            __syncthreads();
            uint32_t w = s_x;
            if (g < hi) {
                while (g >= __ldg(a.hbase + w + 1)) w++;
                const uint32_t wi = __ldg(a.hw + w);
                const uint32_t ws = __ldg(a.word_start + wi), len = __ldg(a.word_end + wi) - ws, p = g - __ldg(a.hbase + w);
                const uint8_t* __restrict__ wt = a.text + ws;
                uint32_t id = TKZ_NONE; int L = 0;
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
                if (bad) { a.wbad[w] = 1; id = TKZ_NONE; }
                a.id[0][g] = id; a.s[0][g] = p; a.e[0][g] = p + (uint32_t)L; a.wid[0][g] = w;
                cnt += id != TKZ_NONE;
            }
            __syncthreads();
        }
        const uint32_t tot = bg_block_sum(cnt, red);
        if (t == 0) a.blk[b] = tot;
    }
    grid.sync();
    // ---------------- compaction of the symbols into buffer 1 (every pair rank still to be looked up)
    uint32_t n;
    {
        uint32_t before, total;
        bg_prefix_total(a.blk, G, b, red, before, total);
        uint32_t run = before;
        for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT, phase ^= 1u) {
            const uint32_t g = c0 + t;
            uint32_t id = TKZ_NONE;
            if (g < hi) id = a.id[0][g];
            uint32_t tot;
            const uint32_t ex = block_excl_scan32<BG_NT / 32>(id != TKZ_NONE ? 1u : 0u, sc, phase, &tot);
            if (id != TKZ_NONE) {
                const uint32_t q = run + ex;
                a.id[1][q] = id; a.s[1][q] = a.s[0][g]; a.e[1][q] = a.e[0][g]; a.wid[1][q] = a.wid[0][g]; a.rk[1][q] = TKZ_DIRTY; a.win[1][q] = 0;
            }
            run += tot;
        }
        n = total;
    }
    uint32_t cur = 1;
    grid.sync();

    // ---------------- ranks + windows of all pairs, smallest rank per word (once; afterwards pass K keeps them current)
    range(n, lo, hi);
    {
        uint32_t* const ids = a.id[1]; uint32_t* const rk = a.rk[1]; uint32_t* const wd = a.wid[1]; uint16_t* const win = a.win[1];
        bool any = false;
        for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT) {
            const uint32_t i = c0 + t;
            uint32_t r = TKZ_NONE, w = TKZ_NONE;
            if (i < hi) {
                w = wd[i];
                if (i + 1 < n && wd[i + 1] == w) {
                    if (!a.wbad[w]) { uint32_t nid, wv = 0; r = merge_lookup_win(m, ids[i], ids[i + 1], &nid, &wv); win[i] = (uint16_t)wv; }
                } else r = TKZ_BOUNDARY;
                rk[i] = r;
            }
            const bool finite = r < TKZ_BOUNDARY;
            const uint32_t fm = __ballot_sync(FULL, finite);
            if (fm) {
                // one atomic per warp when all its mergeable pairs belong to the same word (the usual case)
                const uint32_t w0 = __shfl_sync(FULL, w, __ffs(fm) - 1);
                if (__all_sync(FULL, !finite || w == w0)) {
                    uint32_t mn = finite ? r : TKZ_NONE;
                    for (int d = 16; d > 0; d >>= 1) { const uint32_t y = __shfl_xor_sync(FULL, mn, d); mn = y < mn ? y : mn; }
                    if ((t & 31) == 0) atomicMin(&a.wmin[0][w0], mn);
                } else if (finite) atomicMin(&a.wmin[0][w], r);
                any = true;
            }
        }
        if (__syncthreads_or(any ? 1 : 0) && t == 0) *(volatile uint32_t*)(a.gs + 1) = 1u;
    }
    grid.sync();

    // ---------------- merge steps: two passes (H heads, K compaction + new ranks), each warp streaming its own contiguous
    // part of the array, four consecutive symbols per lane (16-byte loads), no block barrier inside a pass.
    // (block 0 keeps counters for TKZ_GRID_DEBUG: gs[5] steps, gs[6] run scans, gs[7] initial symbols, gs[8..] ns in H / K)
    unsigned long long th = 0, tk = 0, ts = 0, t0 = 0;
    uint32_t n_scans = 0, n_sparse = 0, n_phases = 0;
    auto now = [] { unsigned long long x; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(x)); return x; };
    if (gt == 0) a.gs[7] = n;
    const uint32_t lane = t & 31, wq = t >> 5;
    uint32_t* const cnt = a.blk;                                 // heads per warp part: G * 32 entries; then G run boundaries
    uint32_t step = 0;
    for (;; step++) {
        const uint32_t par = step & 1u;
        if (*(volatile uint32_t*)(a.gs + 1 + par) == 0u) break;                   // bpe.zig:232-234 for every word
        if (gt == 0) t0 = now();
        uint32_t* const ids = a.id[cur]; uint32_t* const rk = a.rk[cur]; uint32_t* const wd = a.wid[cur]; uint16_t* const win = a.win[cur];
        const unsigned long long per = range(n, lo, hi);
        const uint32_t per_w = (uint32_t)(per / 32);                              // a multiple of 128
        const unsigned long long wl64 = per * b + (unsigned long long)per_w * wq;
        const uint32_t wlo = (uint32_t)(wl64 < n ? wl64 : n), whi = (uint32_t)(wl64 + per_w < n ? wl64 + per_w : n);

        // H. heads of this step and their new ids
        {
            for (uint32_t w = gt; w < a.n_huge; w += gstride) a.wmin[par ^ 1u][w] = TKZ_NONE;
            if (gt == 0) { a.gs[1 + (par ^ 1u)] = 0; a.gs[3 + (par ^ 1u)] = 0; a.gs[22 + (par ^ 1u)] = 0; }
            uint32_t heads = 0; bool pend = false;
            for (uint32_t c0 = wlo; c0 < whi; c0 += 128) {
                const uint32_t i0 = c0 + 4 * lane;
                uint32_t rr[4] = {TKZ_NONE, TKZ_NONE, TKZ_NONE, TKZ_NONE};
                if (i0 < whi) { const uint4 v = *reinterpret_cast<const uint4*>(rk + i0); rr[0] = v.x; rr[1] = v.y; rr[2] = v.z; rr[3] = v.w; }
                bool fin = false;
#pragma unroll
                for (int k = 0; k < 4; k++) { if (i0 + k >= n) rr[k] = TKZ_NONE; fin |= rr[k] < TKZ_BOUNDARY; }
                uint32_t hv[4] = {TKZ_NONE, TKZ_NONE, TKZ_NONE, TKZ_NONE};
                if (fin) {
                    uint32_t idv[5];
                    { const uint4 v = *reinterpret_cast<const uint4*>(ids + i0); idv[0] = v.x; idv[1] = v.y; idv[2] = v.z; idv[3] = v.w; }
                    idv[4] = i0 + 4 < n ? ids[i0 + 4] : TKZ_NONE;
                    const uint2 w2 = *reinterpret_cast<const uint2*>(win + i0);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t r = rr[k];
                        if (r >= TKZ_BOUNDARY) continue;
                        const uint32_t i = i0 + k, x = idv[k], y = idv[k + 1];
                        bool head = false;
                        if (x != y) {
                            const uint32_t wv = ((k < 2 ? w2.x : w2.y) >> ((k & 1) * 16)) & 0xFFFFu, wl = wv & 0xFFu, wr = wv >> 8;
                            const uint32_t jlo = i > wl ? i - wl : 0;
                            uint32_t jhi = i + wr; if (jhi > n - 2) jhi = n - 2;
                            head = true;
                            for (uint32_t j = i; j > jlo && head;) { --j; const uint32_t rj = rk[j]; if (rj == TKZ_BOUNDARY) break; head = rj >= r; }
                            for (uint32_t j = i + 1; j <= jhi && head; j++) { const uint32_t rj = rk[j]; if (rj == TKZ_BOUNDARY) break; head = rj >= r; }
                        } else {
                            // (A, A).  A run that ends within BG_WALK symbols on both sides: the run-window rule of
                            // tkz_bpe_block.cuh decides.  Longer runs wait for the reference round of their word.
                            uint32_t s0 = i, e0 = i + 2, c = 0;
                            while (c < BG_WALK && s0 > 0 && rk[s0 - 1] != TKZ_BOUNDARY && ids[s0 - 1] == x) { s0--; c++; }
                            const bool lopen = s0 > 0 && rk[s0 - 1] != TKZ_BOUNDARY && ids[s0 - 1] == x;
                            c = 0;
                            while (c < BG_WALK && e0 < n && rk[e0 - 1] != TKZ_BOUNDARY && ids[e0] == x) { e0++; c++; }
                            const bool ropen = e0 < n && rk[e0 - 1] != TKZ_BOUNDARY && ids[e0] == x;
                            if (!lopen && !ropen) {
                                if (((i - s0) & 1u) == 0) {
                                    const uint32_t wv = ((k < 2 ? w2.x : w2.y) >> ((k & 1) * 16)) & 0xFFFFu, wl = wv & 0xFFu, wr = wv >> 8;
                                    const uint32_t jlo = s0 > wl ? s0 - wl : 0;
                                    uint32_t jhi = e0 - 2 + wr; if (jhi > n - 2) jhi = n - 2;
                                    head = true;
                                    for (uint32_t j = s0; j > jlo && head;) { --j; const uint32_t rj = rk[j]; if (rj == TKZ_BOUNDARY) break; head = rj >= r; }
                                    for (uint32_t j = e0 - 1; j <= jhi && head; j++) { const uint32_t rj = rk[j]; if (rj == TKZ_BOUNDARY) break; head = rj >= r; }
                                }
                            } else if (r == a.wmin[par][wd[i]]) {
                                // the reference round of this word: runs of x pair up from their start
                                if (lopen) { hv[k] = BG_PENDING; pend = true; }
                                else head = ((i - s0) & 1u) == 0;
                            }
                        }
                        if (head) { uint32_t nid = 0; merge_rank_lookup(m, x, y, &nid); hv[k] = nid; heads++; }
                    }
                }
                if (i0 < whi) *reinterpret_cast<uint4*>(a.hn + i0) = make_uint4(hv[0], hv[1], hv[2], hv[3]);
            }
            for (int d = 16; d > 0; d >>= 1) heads += __shfl_xor_sync(FULL, heads, d);
            if (lane == 0) cnt[b * 32 + wq] = heads;
            if (__syncthreads_or(pend ? 1 : 0) && t == 0) *(volatile uint32_t*)(a.gs + 3 + par) = 1u;
        }
        grid.sync();
        if (*(volatile uint32_t*)(a.gs + 3 + par) != 0u) {
            n_scans++;
            // long equal-symbol runs: start of the run of every symbol = max-scan over the run boundaries before it
            {
                uint32_t last = 0;
                for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT) {
                    const uint32_t i = c0 + t;
                    if (i < hi && i > 0 && (rk[i - 1] == TKZ_BOUNDARY || ids[i - 1] != ids[i])) last = i;      // increasing in i
                }
                for (int d = 16; d > 0; d >>= 1) { const uint32_t y = __shfl_xor_sync(FULL, last, d); last = y > last ? y : last; }
                __syncthreads();
                if ((t & 31) == 0) red[t >> 5] = last;
                __syncthreads();
                if (t == 0) { uint32_t mx = 0; for (int w = 0; w < BG_NT / 32; w++) mx = red[w] > mx ? red[w] : mx; cnt[G * 32 + b] = mx; }
            }
            grid.sync();
            {
                uint32_t carry = bg_prefix_max(cnt + G * 32, b, red);
                for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT) {
                    const uint32_t i = c0 + t;
                    uint32_t v = 0;
                    if (i < hi && i > 0 && (rk[i - 1] == TKZ_BOUNDARY || ids[i - 1] != ids[i])) v = i;
                    const uint32_t rs = block_incl_maxscan<BG_NT>(v, red, carry);
                    if (i < hi && a.hn[i] == BG_PENDING) {
                        uint32_t hv = TKZ_NONE;
                        if (((i - rs) & 1u) == 0) {
                            uint32_t nid = 0; merge_rank_lookup(m, ids[i], ids[i + 1], &nid); hv = nid;
                            atomicAdd(&cnt[b * 32 + (uint32_t)((i - per * b) / per_w)], 1u);
                        }
                        a.hn[i] = hv;
                    }
                    __syncthreads();
                    if (t == BG_NT - 1) s_x = rs;
                    __syncthreads();
                    carry = s_x;
                }
            }
            grid.sync();
        }
        unsigned long long dth = 0;
        if (gt == 0) { const unsigned long long x = now(); dth = x - t0; th += dth; t0 = x; }

        // K. compaction into the other buffer (symbol i moves to i - #heads before i - 1) + ranks of the pairs a merge touched
        {
            const uint32_t nxt = cur ^ 1u;
            uint32_t before, total;
            bg_prefix_total(cnt, G * 32, b * 32, red, before, total);
            {
                const uint32_t own = __ldcg(cnt + b * 32 + lane);
                uint32_t inc = own;
                for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(FULL, inc, d); if (lane >= (uint32_t)d) inc += y; }
                before += __shfl_sync(FULL, inc - own, wq);
            }
            uint32_t run = before;
            uint32_t lmin = TKZ_NONE, lw = TKZ_NONE;                 // smallest new rank seen by this lane, and its word
            uint32_t nfin = 0;                                       // pairs with a rank among the symbols this lane wrote
            for (uint32_t c0 = wlo; c0 < whi; c0 += 128) {
                const uint32_t i0 = c0 + 4 * lane;
                const bool in = i0 < whi;
                uint32_t hh[6], idv[6], wv[6], sv[4], ev[5], rr[4], wn[4];
                {
                    uint4 v = make_uint4(TKZ_NONE, TKZ_NONE, TKZ_NONE, TKZ_NONE);
                    if (in) v = *reinterpret_cast<const uint4*>(a.hn + i0);
                    hh[0] = v.x; hh[1] = v.y; hh[2] = v.z; hh[3] = v.w;
#pragma unroll
                    for (int k = 0; k < 4; k++) if (i0 + k >= n) hh[k] = TKZ_NONE;
                }
                uint32_t hprev = __shfl_up_sync(FULL, hh[3], 1);
                hh[4] = __shfl_down_sync(FULL, hh[0], 1); hh[5] = __shfl_down_sync(FULL, hh[1], 1);
                if (lane == 0) hprev = (in && i0 > 0) ? a.hn[i0 - 1] : TKZ_NONE;
                if (lane == 31) { hh[4] = i0 + 4 < n ? a.hn[i0 + 4] : TKZ_NONE; hh[5] = i0 + 5 < n ? a.hn[i0 + 5] : TKZ_NONE; }
                uint32_t c = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) c += hh[k] != TKZ_NONE;
                uint32_t inc = c;
                for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(FULL, inc, d); if (lane >= (uint32_t)d) inc += y; }
                const uint32_t tot = __shfl_sync(FULL, inc, 31);
                uint32_t E = run + inc - c;                          // heads at positions < i0
                run += tot;
                {
                    uint4 v = make_uint4(0, 0, 0, 0), u = v, x = v, y = v, z = v; uint2 w2 = make_uint2(0, 0);
                    if (in) {
                        v = *reinterpret_cast<const uint4*>(ids + i0); u = *reinterpret_cast<const uint4*>(wd + i0);
                        x = *reinterpret_cast<const uint4*>(a.s[cur] + i0); y = *reinterpret_cast<const uint4*>(a.e[cur] + i0);
                        z = *reinterpret_cast<const uint4*>(rk + i0); w2 = *reinterpret_cast<const uint2*>(win + i0);
                    }
                    idv[0] = v.x; idv[1] = v.y; idv[2] = v.z; idv[3] = v.w; wv[0] = u.x; wv[1] = u.y; wv[2] = u.z; wv[3] = u.w;
                    sv[0] = x.x; sv[1] = x.y; sv[2] = x.z; sv[3] = x.w; ev[0] = y.x; ev[1] = y.y; ev[2] = y.z; ev[3] = y.w;
                    rr[0] = z.x; rr[1] = z.y; rr[2] = z.z; rr[3] = z.w;
                    wn[0] = w2.x & 0xFFFFu; wn[1] = w2.x >> 16; wn[2] = w2.y & 0xFFFFu; wn[3] = w2.y >> 16;
                }
                idv[4] = __shfl_down_sync(FULL, idv[0], 1); idv[5] = __shfl_down_sync(FULL, idv[1], 1);
                wv[4] = __shfl_down_sync(FULL, wv[0], 1); wv[5] = __shfl_down_sync(FULL, wv[1], 1);
                ev[4] = __shfl_down_sync(FULL, ev[0], 1);
                if (lane == 31) {
                    idv[4] = i0 + 4 < n ? ids[i0 + 4] : TKZ_NONE; idv[5] = i0 + 5 < n ? ids[i0 + 5] : TKZ_NONE;
                    wv[4] = i0 + 4 < n ? wd[i0 + 4] : TKZ_NONE; wv[5] = i0 + 5 < n ? wd[i0 + 5] : TKZ_NONE;
                    ev[4] = i0 + 4 < n ? a.e[cur][i0 + 4] : 0u;
                }
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t i = i0 + k;
                    const bool hd = hh[k] != TKZ_NONE;
                    const bool pv = (k ? hh[k - 1] : hprev) != TKZ_NONE;
                    if (i < n && in && !pv) {
                        const uint32_t q = i - E;
                        const uint32_t nid = hd ? hh[k] : idv[k];
                        uint32_t r = rr[k], wnew = wn[k];
                        if (hd || hh[k + 1] != TKZ_NONE) {
                            // the pair with the next surviving symbol changed: it is i + 2 behind a head, else i + 1 (itself a head?)
                            const uint32_t nbh = hd ? hh[k + 2] : hh[k + 1], nbid = hd ? idv[k + 2] : idv[k + 1], nbw = hd ? wv[k + 2] : wv[k + 1];
                            if (i + (hd ? 2u : 1u) >= n || nbw != wv[k]) r = TKZ_BOUNDARY;
                            else if (a.wbad[wv[k]]) r = TKZ_NONE;
                            else { uint32_t tmp, w_ = 0; r = merge_lookup_win(m, nid, nbh != TKZ_NONE ? nbh : nbid, &tmp, &w_); wnew = w_; }
                        }
                        a.id[nxt][q] = nid; a.s[nxt][q] = sv[k]; a.e[nxt][q] = hd ? ev[k + 1] : ev[k];
                        a.wid[nxt][q] = wv[k]; a.rk[nxt][q] = r; a.win[nxt][q] = (uint16_t)wnew;
                        if (r < TKZ_BOUNDARY) {
                            nfin++;
                            if (lw == TKZ_NONE) lw = wv[k];
                            if (wv[k] == lw) lmin = r < lmin ? r : lmin; else atomicMin(&a.wmin[par ^ 1u][wv[k]], r);
                        }
                    }
                    E += hd ? 1u : 0u;
                }
            }
            // smallest rank per word: one atomic per warp when all its lanes met the same word (the usual case)
            const uint32_t fm = __ballot_sync(FULL, lw != TKZ_NONE);
            if (fm) {
                const uint32_t w0 = __shfl_sync(FULL, lw, __ffs(fm) - 1);
                if (__all_sync(FULL, lw == TKZ_NONE || lw == w0)) {
                    for (int d = 16; d > 0; d >>= 1) { const uint32_t y = __shfl_xor_sync(FULL, lmin, d); lmin = y < lmin ? y : lmin; }
                    if (lane == 0) atomicMin(&a.wmin[par ^ 1u][w0], lmin);
                } else if (lw != TKZ_NONE) atomicMin(&a.wmin[par ^ 1u][lw], lmin);
            }
            if (__syncthreads_or(fm ? 1 : 0) && t == 0) *(volatile uint32_t*)(a.gs + 1 + (par ^ 1u)) = 1u;
            for (int d = 16; d > 0; d >>= 1) nfin += __shfl_xor_sync(FULL, nfin, d);
            if (lane == 0 && nfin) atomicAdd(a.gs + 22 + (par ^ 1u), nfin);
            if (gt == 0 && step < 256) { a.dbg[4 * step] = n; a.dbg[4 * step + 1] = total; a.dbg[4 * step + 2] = (uint32_t)dth; }
            n -= total;
            cur = nxt;
        }
        grid.sync();
        if (gt == 0) { const unsigned long long d = now() - t0; tk += d; if (step < 256) a.dbg[4 * step + 3] = (uint32_t)d; t0 = now(); }

        // ---------------- sparse phase.  Once less than 1/BG_SPARSE_DIV of the pairs still have a rank, copying the whole array
        // per step is the cost (long dependency chains resolve one link per step: dozens of steps with a handful of merges each).
        // The few pairs that still have a rank are kept in a list; merges are applied IN PLACE: the right symbol of a merged
        // pair is marked dead (dstep = the step it died in; a step sees the deaths of earlier steps only) and skipped when
        // neighbours / windows are walked.  Same head rule as pass H; two passes and two grid barriers per step.  One compaction
        // at the end.  An (A, A) run longer than
        // BG_SPARSE_WALK returns to the dense steps (run scan) after that compaction.
        // Scratch = the arrays of the other buffer: pair lists, dstep, hstep (step in which hn[i] was written).
        const uint32_t n_live = *(volatile uint32_t*)(a.gs + 22 + (par ^ 1u));
        if (gt == 0 && step < 256) a.dbg[1024 + step] = n_live;
        if ((unsigned long long)n_live * BG_SPARSE_DIV < n && n_live != 0u) {
            const uint32_t nxt = cur ^ 1u;
            uint32_t* const ids2 = a.id[cur]; uint32_t* const rk2 = a.rk[cur]; uint32_t* const wd2 = a.wid[cur]; uint16_t* const win2 = a.win[cur];
            uint32_t* const ev2 = a.e[cur];
            uint32_t* lst[2] = {a.id[nxt], a.s[nxt]};
            uint32_t* const dstep = a.rk[nxt]; uint32_t* const hstep = a.wid[nxt];
            range(n, lo, hi);
            for (uint32_t c0 = lo; c0 < hi; c0 += BG_NT) {
                const uint32_t i = c0 + t;
                bool fin = false;
                if (i < hi) { dstep[i] = 0; hstep[i] = 0; fin = rk2[i] < TKZ_BOUNDARY; }
                const uint32_t fm = __ballot_sync(FULL, fin);
                if (fm) {
                    uint32_t base = 0;
                    if (lane == 0) base = atomicAdd(a.gs + 18, (uint32_t)__popc(fm));
                    base = __shfl_sync(FULL, base, 0);
                    if (fin) lst[0][base + __popc(fm & ((1u << lane) - 1u))] = i;
                }
            }
            grid.sync();
            uint32_t gstep = 0, li = 0, sp = par ^ 1u;
            auto dead = [&](uint32_t i) { const uint32_t d = dstep[i]; return d != 0u && d < gstep; };
            auto next_live = [&](uint32_t i) { do { i++; } while (i < n && dead(i)); return i; };                // n: none
            auto prev_live = [&](uint32_t i) { while (i > 0) { i--; if (!dead(i)) return i; } return (uint32_t)TKZ_NONE; };
            auto head_id = [&](uint32_t i) { return hstep[i] == gstep ? a.hn[i] : (uint32_t)TKZ_NONE; };       // TKZ_NONE: not a head this step
            for (;;) {
                const uint32_t len = *(volatile uint32_t*)(a.gs + 18 + li);
                if (len == 0) break;
                gstep++;
                const uint32_t* const L = lst[li]; uint32_t* const Ln = lst[li ^ 1u];
                // H. heads (wmin[sp] = smallest rank per word: from pass K at the start, then from pass A of the step before)
                for (uint32_t w = gt; w < a.n_huge; w += gstride) a.wmin[sp ^ 1u][w] = TKZ_NONE;
                if (gt == 0) { a.gs[18 + (li ^ 1u)] = 0; a.gs[16 + ((gstep & 1u) ^ 1u)] = 0; }
                for (uint32_t idx = gt; idx < len; idx += gstride) {
                    const uint32_t i = L[idx], r = rk2[i], j = next_live(i), x = ids2[i], y = ids2[j];
                    bool head = false;
                    if (x != y) {
                        const uint32_t wv = win2[i], wl = wv & 0xFFu, wr = wv >> 8;
                        head = true;
                        uint32_t q = i;
                        for (uint32_t c = 0; c < wl && head; c++) { q = prev_live(q); if (q == TKZ_NONE) break; const uint32_t rq = rk2[q]; if (rq == TKZ_BOUNDARY) break; head = rq >= r; }
                        q = i;
                        for (uint32_t c = 0; c < wr && head; c++) { q = next_live(q); if (q >= n) break; const uint32_t rq = rk2[q]; if (rq == TKZ_BOUNDARY) break; head = rq >= r; }
                    } else {
                        // (A, A): run-window rule for runs that end within BG_WALK symbols on both sides, else the word's round
                        uint32_t s0 = i, last = j, c = 0, c2 = 0;
                        bool lopen = false, ropen = false;
                        for (;;) {
                            const uint32_t pq = prev_live(s0);
                            if (pq == TKZ_NONE || rk2[pq] == TKZ_BOUNDARY || ids2[pq] != x) break;
                            if (c == BG_WALK) { lopen = true; break; }
                            s0 = pq; c++;
                        }
                        for (;;) {
                            if (rk2[last] == TKZ_BOUNDARY) break;
                            const uint32_t nq = next_live(last);
                            if (nq >= n || ids2[nq] != x) break;
                            if (c2 == BG_WALK) { ropen = true; break; }
                            last = nq; c2++;
                        }
                        if (!lopen && !ropen) {
                            if ((c & 1u) == 0) {
                                const uint32_t wv = win2[i], wl = wv & 0xFFu, wr = wv >> 8;
                                head = true;
                                uint32_t q = s0;
                                for (uint32_t d = 0; d < wl && head; d++) { q = prev_live(q); if (q == TKZ_NONE) break; const uint32_t rq = rk2[q]; if (rq == TKZ_BOUNDARY) break; head = rq >= r; }
                                q = last;
                                for (uint32_t d = 0; d < wr && head; d++) { const uint32_t rq = rk2[q]; if (rq == TKZ_BOUNDARY) break; head = rq >= r; q = next_live(q); if (q >= n) break; }
                            }
                        } else if (r == a.wmin[sp][wd2[i]]) {
                            // the reference round of this word; the parity of a long run needs the whole distance to its start
                            uint32_t q = s0;
                            for (;;) {
                                const uint32_t pq = prev_live(q);
                                if (pq == TKZ_NONE || rk2[pq] == TKZ_BOUNDARY || ids2[pq] != x) break;
                                q = pq;
                                if (++c > a.sparse_walk) { *(volatile uint32_t*)(a.gs + 16 + (gstep & 1u)) = 1u; break; }
                            }
                            head = (c & 1u) == 0;
                        }
                    }
                    uint32_t hv = TKZ_NONE;
                    if (head) merge_rank_lookup(m, x, y, &hv);
                    a.hn[i] = hv; hstep[i] = gstep;
                }
                grid.sync();
                if (*(volatile uint32_t*)(a.gs + 16 + (gstep & 1u)) != 0u) break;
                // A. apply the merges in place, ranks of the pairs they touch, next list + the word minima of the next step
                for (uint32_t c0 = 0; c0 < len; c0 += gstride) {
                    const uint32_t idx = c0 + gt;
                    uint32_t add0 = TKZ_NONE, add1 = TKZ_NONE;                   // pairs with a rank for the next list
                    uint32_t rmin = TKZ_NONE, w = TKZ_NONE;                      // smallest rank among them, their word
                    if (idx < len) {
                        const uint32_t i = L[idx];
                        const uint32_t nid = head_id(i);
                        w = wd2[i];
                        if (nid != TKZ_NONE) {
                            const uint32_t j = next_live(i), k2 = next_live(j);
                            uint32_t r1 = TKZ_BOUNDARY, w1 = 0;
                            if (k2 < n && wd2[k2] == w) { const uint32_t hk = head_id(k2); uint32_t tmp; r1 = merge_lookup_win(m, nid, hk != TKZ_NONE ? hk : ids2[k2], &tmp, &w1); }
                            const uint32_t pl = prev_live(i);
                            if (pl != TKZ_NONE && wd2[pl] == w) {
                                const uint32_t pp = prev_live(pl);
                                if (!(pp != TKZ_NONE && head_id(pp) != TKZ_NONE)) {              // pl itself survives this step
                                    uint32_t tmp, w0 = 0;
                                    const uint32_t r0 = merge_lookup_win(m, ids2[pl], nid, &tmp, &w0);
                                    rk2[pl] = r0; win2[pl] = (uint16_t)w0;
                                    if (r0 < TKZ_BOUNDARY) { add1 = pl; rmin = r0; }
                                }
                            }
                            ids2[i] = nid; ev2[i] = ev2[j]; rk2[i] = r1; win2[i] = (uint16_t)w1; dstep[j] = gstep;
                            if (r1 < TKZ_BOUNDARY) { add0 = i; rmin = r1 < rmin ? r1 : rmin; }
                        } else {
                            const uint32_t pl = prev_live(i);
                            const bool removed = pl != TKZ_NONE && head_id(pl) != TKZ_NONE;
                            if (!removed && head_id(next_live(i)) == TKZ_NONE) { add0 = i; rmin = rk2[i]; }   // (a head to the right re-ranks and lists this pair)
                        }
                    }
                    const uint32_t m0 = __ballot_sync(FULL, add0 != TKZ_NONE), m1 = __ballot_sync(FULL, add1 != TKZ_NONE);
                    if (m0 | m1) {
                        uint32_t base = 0;
                        if (lane == 0) base = atomicAdd(a.gs + 18 + (li ^ 1u), (uint32_t)(__popc(m0) + __popc(m1)));
                        base = __shfl_sync(FULL, base, 0);
                        const uint32_t lt = (1u << lane) - 1u;
                        if (add0 != TKZ_NONE) Ln[base + __popc(m0 & lt)] = add0;
                        if (add1 != TKZ_NONE) Ln[base + __popc(m0) + __popc(m1 & lt)] = add1;
                        // one atomic per warp when all its listed pairs belong to the same word (the usual case)
                        const uint32_t w0 = __shfl_sync(FULL, w, __ffs(m0 | m1) - 1);
                        if (__all_sync(FULL, rmin == TKZ_NONE || w == w0)) {
                            for (int d = 16; d > 0; d >>= 1) { const uint32_t y = __shfl_xor_sync(FULL, rmin, d); rmin = y < rmin ? y : rmin; }
                            if (lane == 0) atomicMin(&a.wmin[sp ^ 1u][w0], rmin);
                        } else if (rmin != TKZ_NONE) atomicMin(&a.wmin[sp ^ 1u][w], rmin);
                    }
                }
                grid.sync();
                li ^= 1u; sp ^= 1u;
                n_sparse++;
            }
            // compaction: the dead symbols leave; the other buffer becomes the array again
            {
                const unsigned long long per2 = range(n, lo, hi);
                const uint32_t pw2 = (uint32_t)(per2 / 32);
                const unsigned long long wl64 = per2 * b + (unsigned long long)pw2 * wq;
                const uint32_t wlo = (uint32_t)(wl64 < n ? wl64 : n), whi = (uint32_t)(wl64 + pw2 < n ? wl64 + pw2 : n);
                uint32_t nd = 0;
                for (uint32_t c0 = wlo; c0 < whi; c0 += 32) {
                    const uint32_t i = c0 + lane;
                    if (i < whi) { const bool d = dstep[i] != 0u; a.hn[i] = d ? 1u : 0u; nd += d; }
                }
                for (int d = 16; d > 0; d >>= 1) nd += __shfl_xor_sync(FULL, nd, d);
                if (lane == 0) cnt[b * 32 + wq] = nd;
                for (uint32_t w = gt; w < a.n_huge; w += gstride) { a.wmin[0][w] = TKZ_NONE; a.wmin[1][w] = TKZ_NONE; }
                if (gt == 0) { a.gs[1] = 0; a.gs[2] = 0; }
                grid.sync();
                // (only now: a block may still have been reading the run-scan flag / list length when block 0 got here)
                if (gt == 0) { a.gs[16] = 0; a.gs[17] = 0; a.gs[18] = 0; a.gs[19] = 0; }
                uint32_t before, total;
                bg_prefix_total(cnt, G * 32, b * 32, red, before, total);
                {
                    const uint32_t own = __ldcg(cnt + b * 32 + lane);
                    uint32_t inc = own;
                    for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(FULL, inc, d); if (lane >= (uint32_t)d) inc += y; }
                    before += __shfl_sync(FULL, inc - own, wq);
                }
                uint32_t run = before;
                bool any = false;
                uint32_t* const sv2 = a.s[cur];
                for (uint32_t c0 = wlo; c0 < whi; c0 += 32) {
                    const uint32_t i = c0 + lane;
                    const bool live = i < whi && a.hn[i] == 0u;
                    uint32_t xi = 0, xs = 0, xe = 0, xw = 0, xr = TKZ_NONE, xn = 0;
                    if (live) { xi = ids2[i]; xs = sv2[i]; xe = ev2[i]; xw = wd2[i]; xr = rk2[i]; xn = win2[i]; }
                    const uint32_t lm = __ballot_sync(FULL, live), valid = __ballot_sync(FULL, i < whi);
                    const uint32_t q = i - (run + (uint32_t)__popc(valid & ~lm & ((1u << lane) - 1u)));
                    run += (uint32_t)__popc(valid & ~lm);
                    if (live) {
                        // (the words of this buffer were scratch: all six arrays are written)
                        a.id[nxt][q] = xi; a.s[nxt][q] = xs; a.e[nxt][q] = xe; a.wid[nxt][q] = xw; a.rk[nxt][q] = xr; a.win[nxt][q] = (uint16_t)xn;
                        if (xr < TKZ_BOUNDARY) { atomicMin(&a.wmin[par ^ 1u][xw], xr); any = true; }
                    }
                }
                if (__syncthreads_or(any ? 1 : 0) && t == 0) *(volatile uint32_t*)(a.gs + 1 + (par ^ 1u)) = 1u;
                n -= total;
                cur = nxt;
                n_phases++;
            }
            grid.sync();
            if (gt == 0) ts += now() - t0;
        }
    }
    if (gt == 0) {
        a.gs[5] = step; a.gs[6] = n_scans; a.gs[20] = n_sparse; a.gs[21] = n_phases;
        unsigned long long* g64 = reinterpret_cast<unsigned long long*>(a.gs + 8);
        g64[0] = ts; g64[1] = th; g64[2] = tk;
    }

    // ---------------- tokens (bpe.zig:256-260): first symbol of every word in the final array, then the copy to the pool
    {
        uint32_t* const wd = a.wid[cur];
        range(n, lo, hi);
        if (n == 0) { for (uint32_t w = gt; w <= a.n_huge; w += gstride) a.wstart[w] = 0; }
        for (uint32_t i = lo + t; i < hi; i += BG_NT) {
            const uint32_t w = wd[i];
            if (i == 0) { for (uint32_t x = 0; x <= w; x++) a.wstart[x] = 0; }
            else { const uint32_t pw = wd[i - 1]; for (uint32_t x = pw + 1; x <= w; x++) a.wstart[x] = i; }
            if (i == n - 1) for (uint32_t x = w + 1; x <= a.n_huge; x++) a.wstart[x] = n;
        }
        grid.sync();
        for (uint32_t i = lo + t; i < hi; i += BG_NT) {
            const uint32_t w = wd[i];
            if (a.wbad[w]) continue;
            const uint32_t q = __ldg(a.word_start + __ldg(a.hw + w)) + (i - a.wstart[w]);
            a.pool_id[q] = a.id[cur][i]; a.pool_s[q] = a.s[cur][i]; a.pool_e[q] = a.e[cur][i];
        }
        for (uint32_t w = gt; w < a.n_huge; w += gstride) {
            if (a.wbad[w]) continue;
            const uint32_t wi = __ldg(a.hw + w);
            a.word_ntok[wi] = a.wstart[w + 1] - a.wstart[w];
            a.done[wi] = 1;
        }
    }
}

// the huge words of a word list, in list order, with the prefix sums of their lengths.  One block.
__global__ void __launch_bounds__(1024) huge_list_kernel(const uint32_t* __restrict__ word_start, const uint32_t* __restrict__ word_end, uint32_t n_words,
                                                         uint32_t min_len, uint32_t cap, uint32_t* __restrict__ hw, uint32_t* __restrict__ hbase,
                                                         unsigned long long* __restrict__ out /* [0] n_huge, [1] total bytes */) {
    __shared__ unsigned long long sh64[33];
    __shared__ uint32_t sc[2 * 33];
    const uint32_t t = threadIdx.x;
    uint32_t nh = 0, phase = 0;
    unsigned long long bytes = 0;
    for (uint32_t c0 = 0; c0 < n_words; c0 += 1024, phase ^= 1u) {
        const uint32_t w = c0 + t;
        uint32_t len = 0;
        if (w < n_words) { len = word_end[w] - word_start[w]; if (len < min_len) len = 0; }
        uint32_t tot; unsigned long long tb;
        const uint32_t ex = block_excl_scan32<32>(len ? 1u : 0u, sc, phase, &tot);
        const unsigned long long eb = block_excl_scan64<32>((unsigned long long)len, sh64, &tb);
        if (len && nh + ex < cap) { hw[nh + ex] = w; hbase[nh + ex] = (uint32_t)(bytes + eb); }
        nh += tot; bytes += tb;
    }
    if (t == 0) {
        if (nh <= cap && bytes < 0xFFFFF000ull) hbase[nh] = (uint32_t)bytes;
        out[0] = nh; out[1] = bytes;
    }
}

}  // namespace tkz
