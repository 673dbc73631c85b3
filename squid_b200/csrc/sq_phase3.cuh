// Phase 3 of the path: concordant fragments covering each breakpoint (the BAM pass of ExactBPConcordantSupport,
// SegmentGraph.cpp:3124-3166), two passes:
//   k_cov_gather  : the qualifying records -- right-hand mates that pass the gate (:3136-3142) -- as (fragment start key,
//                   fragment end) pairs in stream order.  The classification kernel (sq_phase1.cuh) writes them per tile;
//                   this pass closes the gaps at offsets that come from a scan of the per-tile counts.  Rank offsets and the
//                   running maximum of the start keys are kept per tile, which is all the indBP threshold search needs.
//   k_cov_count   : one pass over the compacted pairs (12 B each).  A block first intersects the position range of its
//                   fragments with the sorted breakpoint list; most blocks see no breakpoint at all and stop there, the
//                   others count against the few breakpoints in range from shared memory.
#ifndef SQ_PHASE3_CUH
#define SQ_PHASE3_CUH
#include "sq_depth_cover.cuh"
#include "sq_stream.cuh"

namespace sq {

struct CovTile {
    int64_t rank0;       // qualifying records before the tile
    uint64_t incmax;     // running maximum of the start keys up to and including the tile
};

constexpr int kCovTile = 2048, kCovThreads = 256, kCovRPT = kCovTile / kCovThreads, kCovWarps = kCovThreads / 32, kCovChunks = kCovTile / 32;
static_assert(kCovTile % kTile == 0, "a coverage tile is a whole number of classification tiles");
// The qualifying records -- right-hand mates that pass the gate (:3136-3142) -- leave the classification kernel as (fragment start
// key, fragment end) pairs compacted inside each 512-record tile (P1Out::qstage_*), together with the tile's count and maximum key.
// rank0[t] / incmax[t] = qualifying records before classification tile t / maximum start key up to and including it (scans of
// those per-tile values): this kernel only closes the gaps between the tiles -- 12 B read and written per qualifying record where
// a separate compaction pass read 23 B of every record -- and no tile waits for another.
__global__ void __launch_bounds__(kCovThreads) k_cov_gather(const uint64_t *stage_key, const int32_t *stage_end, const uint32_t *nq_tile, const int64_t *rank0, const uint64_t *incmax,
                                                             int32_t n_ctiles, int32_t n_tiles, uint64_t *qkey, int32_t *qend, CovTile *tiles) {
    const int tile = blockIdx.x;
    constexpr int kPer = kCovTile / kTile;
    const int ct0 = tile * kPer;
    int ct1 = ct0 + kPer - 1;
    if (ct1 > n_ctiles - 1) ct1 = n_ctiles - 1;
    for (int ct = ct0; ct <= ct1; ct++) {
        const int32_t cnt = (int32_t)nq_tile[ct];
        const int64_t base = rank0[ct], src = (int64_t)ct * kTile;
        for (int k = threadIdx.x; k < cnt; k += kCovThreads) { qkey[base + k] = stage_key[src + k]; qend[base + k] = stage_end[src + k]; }
    }
    if (threadIdx.x == 0) { CovTile t; t.rank0 = rank0[ct0]; t.incmax = incmax[ct1]; tiles[tile] = t; }
}

// r0[k] = first qualifying rank whose running-maximum start key exceeds (chr, pos + dist) of breakpoint k (nq if none);
// also the breakpoint keys and the max-plus form t[k] = r0[k] - k.
__global__ void k_cov_r0_tiles(const uint64_t *qkey, const CovTile *tiles, int32_t n_tiles, int64_t nq, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K,
                               int32_t dist, uint64_t *bpkey, int64_t *r0, int64_t *t) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= K) return;
    bpkey[k] = chrpos_key(bp_chr[k], bp_pos[k]);
    const uint64_t T = cover_pass_key(bp_chr[k], bp_pos[k], dist);
    int32_t lo = 0, hi = n_tiles;  // first tile whose inclusive maximum exceeds T
    while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (tiles[m].incmax <= T) lo = m + 1; else hi = m; }
    int64_t v = nq;
    if (lo < n_tiles) {
        uint64_t run = lo > 0 ? tiles[lo - 1].incmax : 0ull;
        const int64_t a = tiles[lo].rank0, e = lo + 1 < n_tiles ? tiles[lo + 1].rank0 : nq;
        for (int64_t i = a; i < e; i++) { const uint64_t q = qkey[i]; if (q > run) run = q; if (run > T) { v = i; break; } }
    }
    r0[k] = v;
    t[k] = v - k;
}

constexpr int kCovRanks = 1024;   // ranks per block of k_cov_count
constexpr int kCovWin = 256;      // breakpoints a block counts in shared memory
__global__ void __launch_bounds__(256) k_cov_count_tiles(const uint64_t *qkey, const int32_t *qend, int64_t nq, const uint64_t *bpkey, const int64_t *t, int64_t K, int32_t *cov) {
    __shared__ unsigned long long s_lo[8], s_hi[8];
    __shared__ unsigned long long s_bp[kCovWin];
    __shared__ long long s_t[kCovWin];
    __shared__ int32_t s_c[kCovWin];
    __shared__ long long s_ka, s_kb;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned full = 0xffffffffu;
    const int64_t i0 = (int64_t)blockIdx.x * kCovRanks;
    uint64_t ks[4], ke[4];
    uint64_t mn = ~0ull, mxe = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int64_t i = i0 + j * 256 + tid;
        ks[j] = ~0ull; ke[j] = 0;
        if (i < nq) {
            ks[j] = qkey[i];
            ke[j] = (ks[j] & 0xffffffff00000000ull) | (uint32_t)qend[i];
            if (ks[j] < mn) mn = ks[j];
            if (ke[j] > mxe) mxe = ke[j];
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { const uint64_t o = __shfl_xor_sync(full, mn, d); if (o < mn) mn = o; }
    mxe = warp_max_u64(mxe);
    if (lane == 0) { s_lo[warp] = mn; s_hi[warp] = mxe; }
    __syncthreads();
    if (warp < 2) {  // warp 0: first breakpoint at/after the leftmost fragment start; warp 1: ... the rightmost fragment end
        uint64_t a = ~0ull, e = 0;
        for (int w = 0; w < 8; w++) { if (s_lo[w] < a) a = s_lo[w]; if (s_hi[w] > e) e = s_hi[w]; }
        const uint64_t v = warp == 0 ? a : e;
        int64_t lo = 0, hi = K;  // 32-way search: 4 dependent probes instead of 18
        while (hi - lo > 0) {
            const int64_t step = (hi - lo + 32) / 33;
            const int64_t p = lo + (int64_t)(lane + 1) * step - 1;  // probes lo+step-1, lo+2step-1, ...
            const bool less = p < hi && bpkey[p] < v;
            const unsigned m = __ballot_sync(full, less);
            const int c = __popc(m);  // probes below v form a prefix
            const int64_t nlo = lo + (int64_t)c * step;
            const int64_t nhi = c < 32 ? (lo + (int64_t)(c + 1) * step - 1 < hi ? lo + (int64_t)(c + 1) * step - 1 : hi) : hi;
            lo = nlo < hi ? nlo : hi; hi = nhi;
        }
        if (lane == 0) { if (warp == 0) s_ka = lo; else s_kb = lo; }
    }
    __syncthreads();
    const int64_t ka = s_ka, kb = s_kb;
    if (ka >= kb) return;  // no breakpoint under any fragment of the block
    // The breakpoints [ka, kb) under the block are counted kCovWin at a time in shared memory.  Every warp holds 32 consecutive
    // ranks per slot j, whose fragments overlap almost the same few breakpoints: the warp walks only the breakpoints inside
    // its own [leftmost start, rightmost end) and adds one ballot per breakpoint -- no global atomic per (fragment, breakpoint)
    // pair, which serialises on the handful of breakpoints of a highly expressed gene.
    uint64_t wmn[4], wmx[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint64_t a = ks[j];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { const uint64_t o = __shfl_xor_sync(full, a, d); if (o < a) a = o; }
        wmn[j] = a; wmx[j] = warp_max_u64(ke[j]);
    }
    const int64_t nbp = kb - ka;
    for (int64_t w0 = 0; w0 < nbp; w0 += kCovWin) {
        const int nw = (int)((nbp - w0) < kCovWin ? (nbp - w0) : kCovWin);
        __syncthreads();  // the previous window has been flushed
        for (int w = tid; w < nw; w += 256) { s_bp[w] = bpkey[ka + w0 + w]; s_t[w] = t[ka + w0 + w]; s_c[w] = 0; }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (wmx[j] <= s_bp[0] || wmn[j] > s_bp[nw - 1]) continue;  // warp-uniform
            int lo = 0, hi = nw;  // first breakpoint >= the warp's leftmost start
            while (lo < hi) { const int m = (lo + hi) >> 1; if (s_bp[m] < wmn[j]) lo = m + 1; else hi = m; }
            const int wa = lo;
            hi = nw;              // first breakpoint >= the warp's rightmost end
            while (lo < hi) { const int m = (lo + hi) >> 1; if (s_bp[m] < wmx[j]) lo = m + 1; else hi = m; }
            const int wb = lo;
            const int64_t i = i0 + j * 256 + tid;
            for (int w = wa; w < wb; w++) {
                const unsigned long long bp = s_bp[w];
                const bool hit = ks[j] <= bp && bp < ke[j] && i < s_t[w];
                const unsigned m = __ballot_sync(full, hit);
                if (lane == 0 && m) atomicAdd(&s_c[w], __popc(m));
            }
        }
        __syncthreads();
        for (int w = tid; w < nw; w += 256) if (s_c[w]) atomicAdd(&cov[ka + w0 + w], s_c[w]);
    }
}

}  // namespace sq
#endif
