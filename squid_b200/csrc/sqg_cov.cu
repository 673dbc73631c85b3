// Phase 3: breakpoint coverage, whole or staged across range shards.
#include <cub/cub.cuh>

#include <algorithm>

#include "sq_phase3.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

// ------------------------------------------------------------------------------------------------
// kernels: breakpoint coverage
// ------------------------------------------------------------------------------------------------
__global__ void k_cov_verify(const uint64_t *qkey, int64_t nq, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K, int32_t dist,
                             const int64_t *r0, int64_t *t, int32_t *fail) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= K) return;
    const int64_t c = t[k] + k;  // candidate rank
    t[k] = c;
    if (c != r0[k] && c < nq) {  // lag mode: the qualifying record right after t[k-1] must itself pass breakpoint k
        const uint64_t T = cover_pass_key(bp_chr[k], bp_pos[k], dist);
        if (!(qkey[c] > T)) *fail = 1;
    }
}
// Literal chain (:3157-3158), used when the verification above fails: indBP advances by at most one per qualifying
// record, so t[k] = first rank c > t[k-1] whose key passes breakpoint k.  One warp: the lanes prefetch r0/T of 32
// breakpoints and a 128-wide window of record keys; the steps themselves run on shuffled registers.
// Chunked: the breakpoint list is cut where r0 jumps by more than kChainGap ranks; every chunk is replayed by its own warp
// under the assumption that the chain has caught up at its first breakpoint (t = r0 there).  k_cov_chain_check verifies
// that assumption (t of the previous breakpoint < r0 of the chunk's first); only if it fails somewhere is the whole list
// replayed by one warp (chunk_start == nullptr).
constexpr int64_t kChainGap = 4096;
// (also every 32nd breakpoint at which the max-plus candidate has caught up with r0, t == r0: long stretches without a big
// jump of r0 would otherwise be one chunk, replayed by a single warp; the check / redo rounds make any cut set valid)
struct IsChainCutOp {
    const int64_t *r0, *t;
    __device__ bool operator()(int32_t k) const { return k == 0 || r0[k] - r0[k - 1] > kChainGap || ((k & 31) == 0 && t[k] == r0[k]); }
};
// A chunk was replayed with some incoming t (`used`, -1 = "the chain has caught up": irrelevant).  Given the current t of
// its predecessor it needed `need` = t[k-1] if that reaches r0 of the chunk's first breakpoint, else -1.  Chunks whose used
// and needed carries differ are flagged for another replay; *n_redo counts them.
__global__ void k_cov_chain_check(const int32_t *chunk_start, int32_t n_chunks, const int64_t *r0, const int64_t *t, const int64_t *used, int64_t *need, int32_t *n_redo) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chunks) return;
    int64_t nd = -1;
    if (i > 0) { const int32_t k = chunk_start[i]; if (!(t[k - 1] < r0[k])) nd = t[k - 1]; }
    need[i] = nd;
    if (nd != used[i]) atomicAdd(n_redo, 1);
}
__global__ void k_cov_chain(const uint64_t *qkey, int64_t nq, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K_all, int32_t dist, const int64_t *r0, int64_t *t,
                            const int32_t *chunk_start, int32_t n_chunks, int64_t *used, const int64_t *need) {
    const int lane = threadIdx.x & 31;
    constexpr int W = 4;       // keys per lane
    int64_t k_begin = 0, K = K_all;
    int64_t tp = -1;
    if (chunk_start) {
        const int32_t ci = (int32_t)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
        if (ci >= n_chunks) return;
        if (need) {  // a re-run: only the chunks whose incoming t changed, starting from it
            if (need[ci] == used[ci]) return;
            tp = need[ci];
        }
        __syncwarp();
        if (lane == 0) used[ci] = tp;
        k_begin = chunk_start[ci];
        K = ci + 1 < n_chunks ? chunk_start[ci + 1] : K_all;
    } else if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    int64_t wbase = -1024;     // ranks [wbase, wbase + 32*W) are held in wkey[]
    uint64_t wkey[W];
    for (int q = 0; q < W; q++) wkey[q] = 0;
    for (int64_t kb = k_begin; kb < K; kb += 32) {
        const int64_t k = kb + lane;
        const int64_t my_r0 = k < K ? r0[k] : nq;
        const uint64_t my_T = k < K ? cover_pass_key(bp_chr[k], bp_pos[k], dist) : ~0ull;
        int64_t my_t = 0;
        const int cnt = (int)((K - kb) < 32 ? (K - kb) : 32);
        for (int j = 0; j < cnt; j++) {
            const int64_t r0j = __shfl_sync(0xffffffffu, my_r0, j);
            const uint64_t Tj = __shfl_sync(0xffffffffu, my_T, j);
            int64_t c;
            if (r0j > tp) c = r0j;
            else {
                c = tp + 1;
                while (c < nq) {
                    if (c < wbase || c >= wbase + 32 * W) {
                        wbase = c;
#pragma unroll
                        for (int q = 0; q < W; q++) { const int64_t rr = c + q * 32 + lane; wkey[q] = rr < nq ? qkey[rr] : ~0ull; }
                    }
                    int64_t found = -1;
#pragma unroll
                    for (int q = 0; q < W; q++) {
                        const unsigned m = __ballot_sync(0xffffffffu, wbase + q * 32 + lane >= c && wkey[q] > Tj);
                        if (found < 0 && m) found = wbase + q * 32 + (__ffs(m) - 1);
                    }
                    if (found >= 0) { c = found; break; }
                    c = wbase + 32 * W;
                }
            }
            if (lane == j) my_t = c;
            tp = c < nq ? c : nq;
        }
        if (k < K) t[k] = my_t;
    }
}


// Phase 3, first pass (sq_phase3.cuh: k_cov_compact): enqueued as soon as the class bytes exist -- it does not depend on the
// segment table, so sqg_build_nodes runs it while the host still waits for the chimeric pre-pass.  The count lands in the
// mirror's cov_nq once the stream has been synchronised.
int run_cov_compact(sqg_ctx *ctx) {
    if (ctx->cov_compacted) return SQG_OK;
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    const int64_t n_tiles = (n + kCovTile - 1) / kCovTile;
    if (n > 0) {
        // forked behind the classification: the seed machine (latency-bound, few resident warps) shares the SMs with it
        cudaStream_t st = ctx->stream_cov;
        CK(cudaEventRecord(ctx->ev_cov_fork, ctx->stream));
        CK(cudaStreamWaitEvent(st, ctx->ev_cov_fork, 0));
        CK(ctx->d_qkey.ensure(n + 1)); CK(ctx->d_qend.ensure(n + 1)); CK(ctx->d_covtile.ensure(n_tiles + 1));  // (allocation synchronises: before the launches)
        // rank offsets and running maxima of the classification tiles: scans of the per-tile counts phase 1 left (no look-back chain)
        const int64_t n_ct = (n + kTile - 1) / kTile;
        CK(ctx->d_cov_rank0.ensure(n_ct + 2)); CK(ctx->d_cov_incmax.ensure(n_ct + 2));
        CK(cudaMemsetAsync(ctx->d_cov_nq.p + n_ct, 0, 4, st));
        CK(cub_call(ctx->d_temp_cov, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, ctx->d_cov_nq.p, ctx->d_cov_rank0.p, (int)(n_ct + 1), st); }));
        CK(cub_call(ctx->d_temp_cov, [&](void *t, size_t &tb) { return cub::DeviceScan::InclusiveScan(t, tb, ctx->d_cov_qmax.p, ctx->d_cov_incmax.p, MaxU64(), (int)n_ct, st); }));
        ctx->launches += 4;
        int rc = phase_begin(ctx, "k_cov_compact", st);
        if (rc) return rc;
        k_cov_gather<<<(unsigned)n_tiles, kCovThreads, 0, st>>>(ctx->d_qstage_key.p, ctx->d_qstage_end.p, ctx->d_cov_nq.p, ctx->d_cov_rank0.p, ctx->d_cov_incmax.p, (int32_t)n_ct, (int32_t)n_tiles,
                                                                ctx->d_qkey.p, ctx->d_qend.p, ctx->d_covtile.p);
        ctx->launches++;
        CK(cudaGetLastError());
        rc = phase_end(ctx, "k_cov_compact", st);
        if (rc) return rc;
        CK(cudaMemcpyAsync(&ctx->cnt.d.p->cov_nq, ctx->d_cov_rank0.p + n_ct, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        CK(ctx->cnt.to_host(st, &ctx->cnt.d.p->cov_nq));
        CK(cudaEventRecord(ctx->ev_cov_done, st));
        ctx->cov_pending = true;
    } else { CK(ctx->d_qkey.ensure(1)); CK(ctx->d_qend.ensure(1)); CK(ctx->d_covtile.ensure(1)); }
    ctx->cov_compacted = true;
    return SQG_OK;
}


// ---- breakpoint coverage, staged: prepare (upload, compaction) -> chain (t of the breakpoints from k_begin on) -> count ----
static int cov_prepare(sqg_ctx *ctx, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K) {
    if (!ctx->have_batch) FAIL(SQG_ESTATE, "load the concordant batch first");
    CK(cudaSetDevice(ctx->device));
    for (int64_t k = 0; k + 1 < K; k++)
        if (bp_chr[k] > bp_chr[k + 1] || (bp_chr[k] == bp_chr[k + 1] && bp_pos[k] > bp_pos[k + 1])) FAIL(SQG_EINVAL, "breakpoints must be sorted by (chr, pos)");
    int rc = run_classify(ctx);
    if (rc) return rc;
    const int64_t n = ctx->batch.n_rec;
    CK(ctx->d_bpchr.ensure(K + 1)); CK(ctx->d_bppos.ensure(K + 1)); CK(ctx->d_bpkey.ensure(K + 1)); CK(ctx->d_r0.ensure(K + 1)); CK(ctx->d_t.ensure(K + 1)); CK(ctx->d_cov.ensure(K + 1));
    CK(cudaMemcpyAsync(ctx->d_bpchr.p, bp_chr, K * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_bppos.p, bp_pos, K * 4, cudaMemcpyHostToDevice, ctx->stream));
    // qualifying records compacted in stream order (done already if sqg_build_nodes ran: it only needs the class bytes)
    rc = run_cov_compact(ctx);
    if (rc) return rc;
    rc = cov_join(ctx);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->stream_cov));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->cov_K = K;
    ctx->cov_nq = n > 0 ? ctx->cnt.h.p->cov_nq : 0;
    return SQG_OK;
}

// t[k] for k in [k_begin, K) from this batch's qualifying ranks alone, the chain starting fresh at breakpoint k_begin.
// Values >= nq mean "not passed by any record of this batch" (everything from the first such breakpoint on is unresolved).
static int cov_chain(sqg_ctx *ctx, int64_t k_begin, int64_t k_end) {  // resolves t for the breakpoints [k_begin, k_end)
    const int64_t n = ctx->batch.n_rec, nq = ctx->cov_nq, K = k_end - k_begin;
    if (K <= 0) return SQG_OK;
    const int64_t n_tiles = (n + kCovTile - 1) / kCovTile;
    const int32_t *bpchr = ctx->d_bpchr.p + k_begin, *bppos = ctx->d_bppos.p + k_begin;
    uint64_t *bpkey = ctx->d_bpkey.p + k_begin;
    int64_t *r0 = ctx->d_r0.p + k_begin, *t = ctx->d_t.p + k_begin;
    LAUNCH(k_cov_r0_tiles, blocks_for(K), kThreads, ctx->d_qkey.p, ctx->d_covtile.p, (int32_t)(n > 0 ? n_tiles : 0), nq, bpchr, bppos, K, ctx->params.concord_dist_pos, bpkey, r0, t);
    {   // t[k] = max(r0[k], t[k-1]+1) whenever the qualifying record right after t[k-1] passes breakpoint k (the common case):
        // a max-plus prefix scan, verified in parallel; the literal one-step-per-record chain runs only if a candidate fails
        Counters *dc = ctx->cnt.d.p;
        const Counters &hc = *ctx->cnt.h.p;
        CK(cub_call(ctx->d_temp, [&](void *tmp, size_t &tb) { return cub::DeviceScan::InclusiveScan(tmp, tb, t, t, MaxI64(), (int)K, ctx->stream); }));
        ctx->launches += 2;
        CK(ctx->cnt.zero(ctx->stream, &dc->cov_fail));
        LAUNCH(k_cov_verify, blocks_for(K), kThreads, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, &dc->cov_fail);
        CK(ctx->cnt.to_host(ctx->stream, &dc->cov_fail));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->cov_chain_fallback = hc.cov_fail != 0;
        if (ctx->cov_chain_fallback) {
            // literal chain, chunked at large jumps of r0 (one warp per chunk), validated; whole-list replay as a last resort
            cub::CountingInputIterator<int32_t> cnt(0);
            IsChainCutOp cop{r0, t};
            CK(ctx->d_chunks.ensure(K + 1));
            int32_t *chunks = ctx->d_chunks.p;
            CK(cub_call(ctx->d_temp, [&](void *tmp, size_t &tb) { return cub::DeviceSelect::If(tmp, tb, cnt, chunks, &dc->n_chunks, (int)K, cop, ctx->stream); }));
            CK(ctx->cnt.to_host(ctx->stream, &dc->n_chunks));
            CK(cudaStreamSynchronize(ctx->stream));
            const int32_t n_chunks = hc.n_chunks;
            ctx->launches += 2;
            CK(ctx->d_chain_used.ensure(2 * (size_t)n_chunks + 2));
            int64_t *used = ctx->d_chain_used.p, *need = ctx->d_chain_used.p + n_chunks + 1;
            LAUNCH(k_cov_chain, blocks_for((int64_t)n_chunks * 32, 128), 128, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, chunks, n_chunks,
                   used, (const int64_t *)nullptr);
            // chunks whose predecessor's chain runs into them are replayed from its t; a few rounds settle runs of such chunks
            ctx->cov_chain_chunks = n_chunks;
            bool settled = false;
            for (int round = 0; round < 16 && !settled; round++) {
                CK(ctx->cnt.zero(ctx->stream, &dc->cov_redo));
                LAUNCH(k_cov_chain_check, blocks_for(n_chunks), kThreads, chunks, n_chunks, r0, t, used, need, &dc->cov_redo);
                CK(ctx->cnt.to_host(ctx->stream, &dc->cov_redo));
                CK(cudaStreamSynchronize(ctx->stream));
                if (hc.cov_redo == 0) { settled = true; break; }
                LAUNCH(k_cov_chain, blocks_for((int64_t)n_chunks * 32, 128), 128, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, chunks, n_chunks,
                       used, (const int64_t *)need);
            }
            if (!settled) {  // a lagging chain through very many chunks: literal replay of the whole list by one warp
                ctx->cov_chain_chunks = 1;
                LAUNCH(k_cov_chain, 1, 32, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, (const int32_t *)nullptr, 0,
                       (int64_t *)nullptr, (const int64_t *)nullptr);
            }
        }
    }
    return SQG_OK;
}

// Coverages[k] += #{qualifying rank i < t[k] : start_i <= pos_k < end_i} over this batch's ranks (t = ctx->d_t, local ranks)
static int cov_count(sqg_ctx *ctx, int32_t *cov_out) {
    const int64_t K = ctx->cov_K, nq = ctx->cov_nq;
    CK(cudaMemsetAsync(ctx->d_cov.p, 0, K * 4, ctx->stream));
    PHASE_BEGIN("k_cov_count");
    if (nq > 0) LAUNCH(k_cov_count_tiles, blocks_for(nq, kCovRanks), 256, ctx->d_qkey.p, ctx->d_qend.p, nq, ctx->d_bpkey.p, ctx->d_t.p, K, ctx->d_cov.p);
    PHASE_END("k_cov_count");
    CK(cudaMemcpyAsync(cov_out, ctx->d_cov.p, K * 4, cudaMemcpyDeviceToHost, ctx->stream));
    return SQG_OK;
}

extern "C" int sqg_bp_coverage(sqg_ctx *ctx, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K, int32_t *cov_out) {
    if (!ctx || K < 0 || (K > 0 && (!bp_chr || !bp_pos || !cov_out))) return SQG_EINVAL;
    if (ctx->shard_count > 1) FAIL(SQG_ESTATE, "this context is a range shard: use sqg_shard_cov_*");
    if (K == 0) { if (!ctx->have_batch) FAIL(SQG_ESTATE, "load the concordant batch first"); return SQG_OK; }
    int rc = cov_prepare(ctx, bp_chr, bp_pos, K);
    if (rc) return rc;
    PHASE_BEGIN("coverage");
    rc = cov_chain(ctx, 0, K);
    if (rc) return rc;
    rc = cov_count(ctx, cov_out);
    if (rc) return rc;
    PHASE_END("coverage");
    CK(cudaStreamSynchronize(ctx->stream));
    return SQG_OK;
}

// Range shards: the chain `indBP advances by at most one per qualifying record` (:3157-3158) runs through the shards in
// order.  Every shard resolves the breakpoints [k_in, k_out) -- those whose t falls among its own qualifying ranks when the
// chain enters the shard at breakpoint k_in -- and the caller hands k_out on as the next shard's k_in (shards may run
// speculatively from a guessed k_in and repeat when the guess was wrong).  *n_pass = number of breakpoints that some record
// of this shard passes at all, a guess-free upper bound of every later shard's k_in.
extern "C" int sqg_shard_cov_begin(sqg_ctx *ctx, const int32_t *bp_chr, const int32_t *bp_pos, int64_t K, int64_t *nq, int64_t *n_pass) {
    if (!ctx || K < 0 || (K > 0 && (!bp_chr || !bp_pos)) || !nq || !n_pass) return SQG_EINVAL;
    int rc = cov_prepare(ctx, bp_chr, bp_pos, K);
    if (rc) return rc;
    *nq = ctx->cov_nq; *n_pass = 0;
    if (K == 0) return SQG_OK;
    const int64_t n = ctx->batch.n_rec, n_tiles = (n + kCovTile - 1) / kCovTile;
    LAUNCH(k_cov_r0_tiles, blocks_for(K), kThreads, ctx->d_qkey.p, ctx->d_covtile.p, (int32_t)(n > 0 ? n_tiles : 0), ctx->cov_nq, ctx->d_bpchr.p, ctx->d_bppos.p, K, ctx->params.concord_dist_pos,
           ctx->d_bpkey.p, ctx->d_r0.p, ctx->d_t.p);
    CK(ctx->h_t.ensure(K + 1));
    CK(cudaMemcpyAsync(ctx->h_t.p, ctx->d_r0.p, K * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int64_t lo = 0, hi = K;  // r0 is non-decreasing in k: first breakpoint no record of this shard passes
    while (lo < hi) { const int64_t m = (lo + hi) >> 1; if (ctx->h_t.p[m] < ctx->cov_nq) lo = m + 1; else hi = m; }
    *n_pass = lo;
    ctx->cov_n_pass = lo;
    return SQG_OK;
}
extern "C" int sqg_shard_cov_chain(sqg_ctx *ctx, int64_t k_in, int64_t *k_out) {
    if (!ctx || !k_out || k_in < 0 || k_in > ctx->cov_K) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    // No record of this shard passes a breakpoint from cov_n_pass on (r0 is non-decreasing along the sorted list), so the chain
    // cannot resolve any of them here: only [k_in, cov_n_pass) is walked.  (Walking the unresolvable tail as well made the
    // verification fail on it and sent the whole list through the literal replay: 9 ms on the first of two shards.)
    const int64_t k_end = ctx->cov_n_pass < ctx->cov_K ? ctx->cov_n_pass : ctx->cov_K;
    *k_out = k_in;
    if (k_in >= k_end) return SQG_OK;
    int rc = cov_chain(ctx, k_in, k_end);
    if (rc) return rc;
    CK(ctx->h_t.ensure(ctx->cov_K + 1));
    CK(cudaMemcpyAsync(ctx->h_t.p + k_in, ctx->d_t.p + k_in, (k_end - k_in) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int64_t k = k_in;
    while (k < k_end && ctx->h_t.p[k] < ctx->cov_nq) k++;
    *k_out = k;
    return SQG_OK;
}
// t_global[k] = rank_offset + t[k] for the breakpoints [k_in, k_out) of the last sqg_shard_cov_chain call; other entries untouched
extern "C" int sqg_shard_cov_owned_t(sqg_ctx *ctx, int64_t rank_offset, int64_t k_in, int64_t k_out, int64_t *t_global) {
    if (!ctx || !t_global || k_in < 0 || k_out < k_in || k_out > ctx->cov_K) return SQG_EINVAL;
    for (int64_t k = k_in; k < k_out; k++) t_global[k] = rank_offset + ctx->h_t.p[k];
    return SQG_OK;
}
// cov_partial[k] = this shard's share of Coverages[k] given the global t (unresolved breakpoints: t = total number of ranks)
extern "C" int sqg_shard_cov_count(sqg_ctx *ctx, int64_t rank_offset, const int64_t *t_global, int32_t *cov_partial) {
    if (!ctx || (ctx->cov_K > 0 && (!t_global || !cov_partial))) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    const int64_t K = ctx->cov_K, nq = ctx->cov_nq;
    if (K == 0) return SQG_OK;
    CK(ctx->h_t.ensure(K + 1));
    for (int64_t k = 0; k < K; k++) { int64_t v = t_global[k] - rank_offset; ctx->h_t.p[k] = v < 0 ? 0 : (v > nq ? nq : v); }
    CK(cudaMemcpyAsync(ctx->d_t.p, ctx->h_t.p, K * 8, cudaMemcpyHostToDevice, ctx->stream));
    PHASE_BEGIN("coverage");
    int rc = cov_count(ctx, cov_partial);
    if (rc) return rc;
    PHASE_END("coverage");
    CK(cudaStreamSynchronize(ctx->stream));
    return SQG_OK;
}
