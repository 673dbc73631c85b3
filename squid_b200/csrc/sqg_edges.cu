// Phase 2: per-segment depth, the read-to-segment assignment and the raw edges, reduced to the edge table.
#include <cub/cub.cuh>

#include <algorithm>
#include <cstddef>
#include <cstdlib>
#include <vector>

#include "sq_phase2.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

// ------------------------------------------------------------------------------------------------
// kernels: depth
// ------------------------------------------------------------------------------------------------
__global__ void k_depth_disc(NodeTable nt, const DiscBlock *D, int32_t nD, int32_t *cnt, int32_t *sum) {
    const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nD) return;
    const DiscBlock d = D[k];
    if (d.chr < 0 || d.chr >= nt.n_ref) return;
    const ChrHead h = chr_head(nt, d.chr);
    if (h.c1 <= h.c0) return;
    const SegHit j = seg_at(nt, h, d.pos);  // segment whose turn consumes this block (:774): the last with Position <= pos
    if (d.pos >= j.pos && d.pos + d.len <= j.end) { atomicAdd(&cnt[j.s], 1); atomicAdd(&sum[j.s], d.len); }
}

// ------------------------------------------------------------------------------------------------
// kernels: assignment + raw edges
// ------------------------------------------------------------------------------------------------
// res0 codes: >= 0 segment of the read's first block; -1 located nowhere; -2 read does not touch the hint; -3 hint-sensitive
struct ChimDev {
    int64_t n_reads;
    const uint32_t *read_off; const uint16_t *n_first;
    const int32_t *first_total, *second_total;
    int32_t *ref_id, *ref_pos, *read_pos, *match_ref, *match_read;
    const uint8_t *rev;
};
__device__ __forceinline__ void chim_load_read(const ChimDev &c, int64_t i, ReadView &rv) {
    const uint32_t o = c.read_off[i], e = c.read_off[i + 1], nf = c.n_first[i];
    rv.nF = 0; rv.nS = 0;
    for (uint32_t k = o; k < e; k++) {
        Blk x;
        x.ref_id = c.ref_id[k]; x.ref_pos = c.ref_pos[k]; x.match_ref = c.match_ref[k]; x.read_pos = c.read_pos[k]; x.match_read = c.match_read[k]; x.rev = c.rev[k];
        if (k - o < nf) { if (rv.nF < kMaxBlocks) rv.F[rv.nF++] = x; } else { if (rv.nS < kMaxBlocks) rv.S[rv.nS++] = x; }
    }
    rv.first_total = c.first_total[i]; rv.second_total = c.second_total[i];
}
__device__ __forceinline__ void chim_store_read(const ChimDev &c, int64_t i, const ReadView &rv) {
    uint32_t k = c.read_off[i];
    for (int m = 0; m < 2; m++)
        for (int q = 0; q < (m ? rv.nS : rv.nF); q++, k++) {
            const Blk &x = m ? rv.S[q] : rv.F[q];
            c.ref_pos[k] = x.ref_pos; c.match_ref[k] = x.match_ref; c.read_pos[k] = x.read_pos; c.match_read[k] = x.match_read;
        }
}
__global__ void k_chim_edges(ChimDev c, Params p, NodeTable nt, int32_t *res0, PairSink sink, int32_t *sens, int32_t *n_sens) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= c.n_reads) return;
    Blk F[kMaxBlocks + 1], S[kMaxBlocks + 1];
    int32_t node[2 * kMaxBlocks + 2];
    ReadView rv; rv.F = F; rv.S = S;
    chim_load_read(c, i, rv);
    int32_t out = -2;
    if (rv.nF + rv.nS > 0) {
        if (read_edges(nt, p, rv, MODE_CHIM, true, false, 0, node, sink)) { out = node[0]; chim_store_read(c, i, rv); }
        else { out = -3; sens[atomicAdd(n_sens, 1)] = (int32_t)i; }  // sens holds n_reads entries
    }
    res0[i] = out;
}
// Hint-sensitive reads are replayed with the true hint = segment of the first block of the nearest earlier read that
// located one (res0 >= 0), in stream order.  A run of sensitive reads with no located read in between is a chain: its first
// read (the head) knows its hint from the untouched part of res0, and the head's thread replays the whole chain in order.
// `init_hint`: firstfrontindex before the first read (0 at the start of the stream, :1395, :1568; a range shard gets the
// value its predecessor left); *used_init is set when some chain had to start from it.
__global__ void k_fix_heads(const int32_t *res0, const int32_t *sens, const int32_t *n_sens, int32_t cap, int32_t *head_hint, int32_t init_hint, int32_t *used_init) {
    const int32_t n = *n_sens < cap ? *n_sens : cap;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int32_t hint = init_hint;
        bool from_init = true;
        for (int64_t q = (int64_t)sens[i] - 1; q >= 0; q--) {
            const int32_t v = res0[q];
            if (v >= 0) { hint = v; from_init = false; break; }
            if (v == -3) { hint = -1; from_init = false; break; }  // not a head
        }
        head_hint[i] = hint;
        if (from_init && used_init) *used_init = 1;
    }
}
// firstfrontindex after the last read of the batch: res0 of the last read that located its first block (-1: none)
__global__ void k_last_located(const int32_t *res0, int64_t n, int32_t *out) {
    int32_t v = -1;
    for (int64_t q = n - 1; q >= 0; q--) if (res0[q] >= 0) { v = res0[q]; break; }
    *out = v;
}
template <bool CHIM>
__global__ void k_fix_chains(DevBatch b, ChimDev c, Params p, NodeTable nt, int32_t *res0, int64_t n_items, const int32_t *sens, const int32_t *n_sens, int32_t cap,
                             const int32_t *head_hint, PairSink sink) {
    const int32_t n = *n_sens < cap ? *n_sens : cap;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int32_t hint = head_hint[i];
        if (hint < 0 || hint >= nt.n) continue;  // (>= nt.n: only in an attempt whose lists overflowed and that is repeated anyway)
        int64_t q = sens[i];
        for (;;) {
            Blk F[kMaxBlocks + 1], S[kMaxBlocks + 1];
            int32_t node[2 * kMaxBlocks + 2];
            ReadView rv; rv.F = F; rv.S = S;
            bool is_first = true;
            if (CHIM) chim_load_read(c, q, rv); else conc_load_read(b, q, rv, is_first);
            read_edges(nt, p, rv, CHIM ? MODE_CHIM : MODE_OTHER, is_first, true, hint, node, sink);
            if (CHIM) chim_store_read(c, q, rv);
            res0[q] = node[0] >= 0 ? node[0] : -1;
            if (node[0] >= 0) hint = node[0];
            int64_t q2 = q + 1;
            int32_t v = -2;
            while (q2 < n_items && (v = res0[q2]) < 0 && v != -3) q2++;
            if (q2 >= n_items || v != -3) break;  // the next read that matters located on its own: the chain ends
            q = q2;
        }
    }
}
// blocks of the chimeric reads that LocateRead trimmed (:1229-1248): (index, RefPos, ReadPos, MatchRef, MatchRead) rows -- a few
// thousand of a million, so the caller's arrays are patched on the host instead of copying four whole arrays back
__global__ void k_chim_diff(const int32_t *p0, const int32_t *r0, const int32_t *m0, const int32_t *q0, const int32_t *p1, const int32_t *r1, const int32_t *m1, const int32_t *q1,
                            int64_t n, int32_t *rows5, int32_t cap, int32_t *count) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (p0[k] == p1[k] && r0[k] == r1[k] && m0[k] == m1[k] && q0[k] == q1[k]) return;
    const int32_t at = atomicAdd(count, 1);
    if (at < cap) { int32_t *row = rows5 + 5 * (int64_t)at; row[0] = (int32_t)k; row[1] = p1[k]; row[2] = r1[k]; row[3] = m1[k]; row[4] = q1[k]; }
}
__global__ void k_unpack_edges(const uint64_t *keys, const int32_t *counts, int64_t n, int32_t *ind1, int32_t *ind2, uint8_t *heads, int32_t *w) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t a, c; bool h1, h2;
    edge_unpack(keys[i], a, h1, c, h2);
    ind1[i] = a; ind2[i] = c; heads[i] = (uint8_t)((h1 ? 1 : 0) | (h2 ? 2 : 0)); w[i] = counts[i];
}


static int reduce_edges(sqg_ctx *ctx, int64_t n_raw, const int32_t *d_weights_in);

// ReadsOther blocks of <= 3 bp (sq_depth_cover.cuh).  Their segments are known from the start masks unless some of them tie with
// an entry of the same (chr, start) that would move them: the reference's answer is then the order in which its unstable
// std::sort leaves ReadsOther (SegmentGraph.cpp:781), so the sort is replayed -- std::sort's exact permutation, on the device
// (sq_gpusort.cuh), on the CPU twin if the device declines -- and the merge loop's cursor walked as a running maximum.
static int count_short_other(sqg_ctx *ctx, int64_t n_short, int64_t n_unstable) {
    if (n_short <= 0) return SQG_OK;
    const int32_t N = ctx->nt.n;
    int32_t *cnt_other = ctx->d_cnt3.p + 2 * (size_t)N, *sum_other = ctx->d_sum3.p + 2 * (size_t)N;
    static const bool force_sort = getenv("SQG_OTHER_SORT") && atoi(getenv("SQG_OTHER_SORT")) == 1;  // test hook: the sort path even without order-dependent ties
    if (n_unstable == 0 && !force_sort) {
        LAUNCH(k_depth_short_apply, 64, 128, ctx->d_shorts.p, (int32_t)n_short, cnt_other, sum_other);
        return SQG_OK;
    }
    if (ctx->shard_count > 1 && n_unstable > 0)
        FAIL(SQG_EUNSUPPORTED, "a ReadsOther block of <= 3 bp ties with another block at the same start: its segment depends on the tie order of the reference's "
                               "std::sort over the WHOLE stream (SegmentGraph.cpp:781), which a range shard cannot replay -- run this stream on one context");
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    OtherCountOp op{b.blk_off, ctx->d_cls.p, ctx->r_break};
    cub::CountingInputIterator<int64_t> cnt(0);
    cub::TransformInputIterator<int32_t, OtherCountOp, cub::CountingInputIterator<int64_t>> it(cnt, op);
    CK(ctx->d_other_off.ensure((size_t)n + 2));
    CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, it, ctx->d_other_off.p, (int)(n + 1), ctx->stream); }));
    ctx->launches += 2;
    int32_t m32 = 0;
    CK(cudaMemcpyAsync(&m32, ctx->d_other_off.p + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int64_t M = m32;
    if (M <= 0) return SQG_OK;
    CK(ctx->d_other_key.ensure((size_t)M + 1)); CK(ctx->d_other_idx.ensure((size_t)M + 1)); CK(ctx->d_other_len.ensure((size_t)M + 1)); CK(ctx->d_other_own.ensure((size_t)M + 1));
    LAUNCH(k_other_fill, blocks_for(n), kThreads, b, ctx->d_cls.p, ctx->r_break, ctx->d_other_off.p, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p);
    int rc = 0;
    const cudaError_t se = replay_std_sort(ctx->d_other_key.p, ctx->d_other_idx.p, (size_t)M, ctx->d_gs_scratch, ctx->stream, &ctx->launches, 16, [&]() {
        k_other_fill<<<blocks_for(n), kThreads, 0, ctx->stream>>>(b, ctx->d_cls.p, ctx->r_break, ctx->d_other_off.p, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p);
        ctx->launches++;
        return cudaGetLastError();
    }, &rc);
    if (rc < 0) { ctx->err = std::string("ReadsOther sort: ") + cudaGetErrorString(se); return SQG_ECUDA; }
    ctx->other_sort_status = rc;
    if (se != cudaSuccess) { ctx->err = std::string("ReadsOther sort fallback: ") + cudaGetErrorString(se); return SQG_ECUDA; }
    LAUNCH(k_other_own, blocks_for(M), kThreads, ctx->nt, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p, M, ctx->d_other_own.p);
    CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::InclusiveScan(t, tb, ctx->d_other_own.p, ctx->d_other_own.p, MaxI32(), (int)M, ctx->stream); }));
    ctx->launches += 2;
    LAUNCH(k_other_apply, blocks_for(M), kThreads, ctx->nt, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p, ctx->d_other_own.p, M, cnt_other, sum_other);
    return SQG_OK;
}

// Phase 2 (sq_phase2.cuh): one pass over the batch for the depth numerators (do_depth) and the raw edges of the chimeric
// reads + the concordant stream (do_edges); then the hint fix-up chains and the sort + reduce of the (key, count) pairs.
int run_assign(sqg_ctx *ctx, bool do_depth, bool do_edges) {
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    const int32_t N = ctx->nt.n;
    const int32_t nD = ctx->pre_nD;
    const int64_t n_tiles = (n + kTile - 1) / kTile;
    ChimDev cd;
    cd.n_reads = ctx->c_n_reads; cd.read_off = ctx->dc_read_off.p; cd.n_first = ctx->dc_n_first.p;
    cd.first_total = ctx->dc_first_total.p; cd.second_total = ctx->dc_second_total.p;
    cd.ref_id = ctx->dc_ref_id.p; cd.ref_pos = ctx->dc_ref_pos.p; cd.read_pos = ctx->dc_read_pos.p; cd.match_ref = ctx->dc_match_ref.p; cd.match_read = ctx->dc_match_read.p;
    cd.rev = ctx->dc_rev.p;
    if (do_depth) { CK(ctx->d_cnt3.ensure(3 * (size_t)N + 4)); CK(ctx->d_sum3.ensure(3 * (size_t)N + 4)); CK(ctx->d_dtile.ensure(n_tiles + 1)); }
    int64_t cap = std::max<int64_t>({(int64_t)ctx->d_ekeys.cap, n / 8 + 4 * ctx->c_n_blk + 2 * ctx->c_n_reads + 4096, (int64_t)1 << 20});
    int64_t sens_cap = std::max<int64_t>({(int64_t)ctx->d_sens.cap, n / 64 + 4096, ctx->c_n_reads + 1});
    int64_t slow_cap = std::max<int64_t>({(int64_t)ctx->d_slow.cap, n / 8 + 4096});
    int64_t short_cap = std::max<int64_t>({(int64_t)ctx->d_shorts.cap, n / 256 + 4096});
    CK(ctx->dc_res0.ensure(ctx->c_n_reads + 1)); CK(ctx->d_scratch32.ensure(n + 1));
    Counters *dc = ctx->cnt.d.p;
    const Counters &hc = *ctx->cnt.h.p;
    int64_t n_raw = 0;
    int64_t n_short = 0, n_unstable = 0;
    if (ctx->chim_upload_pending) {  // the chimeric arrays: uploaded by the pre-pass thread behind its own work
        ctx->prepass_worker.wait();
        if (ctx->chim_upload_err) { ctx->err = std::string("upload of the chimeric reads: ") + cudaGetErrorString((cudaError_t)ctx->chim_upload_err); return SQG_ECUDA; }
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_chim, 0));
        ctx->chim_upload_pending = false;
    }
    PHASE_BEGIN(do_depth ? "depth_edges" : "edges_only");
    // Capacity retries.  A list that overflows makes the pass run again with room for what it counted, but an attempt whose slow
    // list overflowed never ran the records past its capacity, and one whose sensitive list overflowed never replayed the
    // chains past it: their raw pairs (and, for deferred records, their sensitive reads) are missing from the counts, so the
    // next attempt can overflow again.  The counts firm up one list at a time -- the slow-list count is always complete, so
    // the second attempt runs every record; its sensitive count is then complete, so the third replays every chain; the raw
    // count of the third is complete -- and the fourth attempt always fits.
    constexpr int kEdgeAttempts = 4;
    for (int attempt = 0; attempt < kEdgeAttempts; attempt++) {
        if (do_edges) ctx->edge_pass_attempts = attempt + 1;
        if (do_edges) { CK(ctx->d_ekeys.ensure(cap)); CK(ctx->d_ew.ensure(cap)); CK(ctx->d_sens.ensure(sens_cap)); CK(ctx->d_head.ensure(sens_cap)); }
        cap = do_edges ? (int64_t)std::min(ctx->d_ekeys.cap, ctx->d_ew.cap) : 0;
        sens_cap = do_edges ? (int64_t)std::min(ctx->d_sens.cap, ctx->d_head.cap) : 0;
        CK(ctx->cnt.zero(ctx->stream, &dc->n_raw, &dc->n_sens));
        int32_t *d_nsens = dc->n_sens;
        PairSink sink{ctx->d_ekeys.p, ctx->d_ew.p, cap, &dc->n_raw};
        if (do_depth) {
            CK(cudaMemsetAsync(ctx->d_cnt3.p, 0, (3 * (size_t)N + 4) * 4, ctx->stream));
            CK(cudaMemsetAsync(ctx->d_sum3.p, 0, (3 * (size_t)N + 4) * 4, ctx->stream));
            if (nD > 0 && ctx->shard_index == 0) LAUNCH(k_depth_disc, blocks_for(nD), kThreads, ctx->nt, ctx->d_disc.p, nD, ctx->d_cnt3.p, ctx->d_sum3.p);
        }
        CK(ctx->cnt.zero(ctx->stream, &dc->used_init, &dc->out_hint));
        if (do_edges && ctx->c_n_blk > 0) {  // every pass trims the ORIGINAL blocks (a trimmed block can fit another segment)
            const size_t nbb = (size_t)ctx->c_n_blk * 4;
            CK(cudaMemcpyAsync(ctx->dc_ref_pos.p, ctx->dc0_ref_pos.p, nbb, cudaMemcpyDeviceToDevice, ctx->stream));
            CK(cudaMemcpyAsync(ctx->dc_read_pos.p, ctx->dc0_read_pos.p, nbb, cudaMemcpyDeviceToDevice, ctx->stream));
            CK(cudaMemcpyAsync(ctx->dc_match_ref.p, ctx->dc0_match_ref.p, nbb, cudaMemcpyDeviceToDevice, ctx->stream));
            CK(cudaMemcpyAsync(ctx->dc_match_read.p, ctx->dc0_match_read.p, nbb, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        if (do_edges && cd.n_reads > 0 && ctx->shard_index == 0) {  // (range shards: the chimeric reads are replicated, shard 0 owns their edges)  // RawEdgesChim: chimeric reads, their sensitive ones replayed in chains
            // (the chimeric sensitive list lives behind the concordant one)
            int32_t *csens = ctx->d_sens.p + (sens_cap - ctx->c_n_reads - 1), *chead = ctx->d_head.p + (sens_cap - ctx->c_n_reads - 1);
            LAUNCH(k_chim_edges, blocks_for(cd.n_reads), kThreads, cd, ctx->params, ctx->nt, ctx->dc_res0.p, sink, csens, d_nsens + 1);
            LAUNCH(k_fix_heads, 64, 128, ctx->dc_res0.p, csens, d_nsens + 1, (int32_t)ctx->c_n_reads, chead, 0, (int32_t *)nullptr);
            LAUNCH(k_fix_chains<true>, 64, 128, b, cd, ctx->params, ctx->nt, ctx->dc_res0.p, cd.n_reads, csens, d_nsens + 1, (int32_t)ctx->c_n_reads, chead, sink);
        }
        const int32_t conc_sens_cap = (int32_t)std::max<int64_t>(0, sens_cap - ctx->c_n_reads - 1);
        if (n > 0) {
            P2Args a;
            a.cls = ctx->d_cls.p; a.nt = ctx->nt; a.p = ctx->params; a.r_break = ctx->r_break; a.do_depth = do_depth; a.do_edges = do_edges;
            a.cnt_main = ctx->d_cnt3.p + (size_t)N; a.sum_main = ctx->d_sum3.p + (size_t)N;
            a.cnt_other = ctx->d_cnt3.p + 2 * (size_t)N; a.sum_other = ctx->d_sum3.p + 2 * (size_t)N;
            a.other_nonempty = do_depth ? ctx->d_cnt3.p + 3 * (size_t)N : nullptr;
            a.dtile = ctx->d_dtile.p; a.res0 = ctx->d_scratch32.p; a.sink = sink;
            a.sens = ctx->d_sens.p; a.n_sens = d_nsens; a.sens_cap = conc_sens_cap;
            CK(ctx->cnt.zero(ctx->stream, &dc->path_counts, &dc->n_short));
            CK(ctx->d_slow.ensure(slow_cap));
            a.path_counts = dc->path_counts;
            a.slow_list = ctx->d_slow.p; a.n_slow = &dc->n_slow; a.slow_cap = (int32_t)std::min<int64_t>(ctx->d_slow.cap, 0x7fffffff);
            CK(ctx->d_omask.ensure((size_t)N + 2)); CK(ctx->d_shorts.ensure((size_t)short_cap));
            a.omask = ctx->d_omask.p; a.shorts = ctx->d_shorts.p; a.n_short = dc->n_short; a.short_cap = (int32_t)std::min<int64_t>(short_cap, 0x7fffffff);
            if (do_depth) CK(cudaMemsetAsync(ctx->d_omask.p, 0, ((size_t)N + 2) * 4, ctx->stream));
            {
                struct { BatchDesc d; NodeTable nt; } hd;
                hd.d.b = b; hd.d.p = ctx->params; hd.nt = ctx->nt;
                CK(ctx->d_desc.ensure(sizeof(hd)));
                CK(cudaMemcpyAsync(ctx->d_desc.p, &hd, sizeof(hd), cudaMemcpyHostToDevice, ctx->stream));
                a.desc = (const BatchDesc *)ctx->d_desc.p; a.nt_dev = (const NodeTable *)(ctx->d_desc.p + offsetof(decltype(hd), nt));
            }
            // two launches of the same tile kernel, one per job: each half is small enough for the instruction cache, and
            // reading the batch twice is cheap next to that
            CK(cudaFuncSetAttribute(k_assign_tiles<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmemBytes));
            CK(cudaFuncSetAttribute(k_assign_tiles<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmemBytes));
            // multi-block records that leave their tile's segment all go to k_edges_generic.  Processing them in the tile kernel from
            // shared memory was measured and dropped: at the App. C block mix, 100 M pairs, 4.6 + 8.3 ms against 21.3 ms -- inside
            // the tile kernel the generic rules stall on instruction fetch (ncu: no_instruction is the top stall) and the tile's warps
            // wait at the barrier behind the one that drew the longest records (profiles/r2_ncu_summary.txt).
            // The depth pass and the edge pass are independent, but running the depth tile kernel on a second stream beside
            // k_edges_generic was measured and dropped (100 M pairs): no gain, 21.6 ms against 20.2 ms for the two passes together --
            // the two kernels compete for the same issue slots and L2 -- so they run in sequence.
            PHASE_BEGIN("k_assign");
            if (do_depth) {
                PHASE_BEGIN("k_assign_depth");
                k_assign_tiles<true, false><<<(unsigned)n_tiles, kTileThreads, kTileSmemBytes, ctx->stream>>>(b, a, batch_bulk_ok(b) ? 1 : 0);
                ctx->launches++;
                CK(cudaGetLastError());
                PHASE_END("k_assign_depth");
                LAUNCH(k_depth_scan, 1, 1024, ctx->d_dtile.p, (int32_t)n_tiles);
                LAUNCH(k_depth_fix, blocks_for(n_tiles), kThreads, b, ctx->d_cls.p, ctx->nt, ctx->r_break, ctx->d_dtile.p, (int32_t)n_tiles, a.cnt_main, a.sum_main);
                LAUNCH(k_depth_short_nodes, 64, 128, ctx->nt, ctx->d_omask.p, ctx->d_shorts.p, a.n_short, a.short_cap, a.n_short + 1);
            }
            if (do_edges) {
                PHASE_BEGIN("k_assign_edges");
                k_assign_tiles<false, true><<<(unsigned)n_tiles, kTileThreads, kTileSmemBytes, ctx->stream>>>(b, a, batch_bulk_ok(b) ? 1 : 0);
                ctx->launches++;
                CK(cudaGetLastError());
                PHASE_END("k_assign_edges");
                PHASE_BEGIN("k_edges_generic");
                // the generic kernel is compiled for 8 resident blocks per SM (64 registers): it is bound by the latency of dependent
                // loads, and more warps with fewer registers each beat fewer warps without local-memory traffic -- measured at 100 M
                // pairs: 7 blocks (72 registers) 6.7 ms, 8 blocks 5.4 ms, 10 and 12 blocks (48 / 40 registers) 5.5 ms
                LAUNCH(k_edges_generic<8>, 148 * 16, 128, a);
                PHASE_END("k_edges_generic");
                LAUNCH(k_fix_heads, 256, 128, ctx->d_scratch32.p, ctx->d_sens.p, d_nsens, conc_sens_cap, ctx->d_head.p, ctx->shard_init_hint, &dc->used_init);
                LAUNCH(k_fix_chains<false>, 256, 128, b, cd, ctx->params, ctx->nt, ctx->d_scratch32.p, n, ctx->d_sens.p, d_nsens, conc_sens_cap, ctx->d_head.p, sink);
                if (ctx->shard_count > 1) LAUNCH(k_last_located, 1, 1, ctx->d_scratch32.p, n, &dc->out_hint);
            }
            PHASE_END("k_assign");
        }
        CK(ctx->cnt.to_host(ctx->stream, &dc->n_raw, &dc->out_hint));
        CK(cudaStreamSynchronize(ctx->stream));
        n_short = do_depth && n > 0 ? hc.n_short[0] : 0;
        n_unstable = do_depth && n > 0 ? hc.n_short[1] : 0;
        ctx->shard_lead_sensitive = hc.used_init != 0;
        ctx->shard_out_hint = (ctx->shard_count > 1 && do_edges && n > 0) ? hc.out_hint : -1;
        n_raw = (int64_t)hc.n_raw;
        const int32_t ns_conc = hc.n_sens[0], ns_chim = hc.n_sens[1];
        ctx->n_sensitive = (int64_t)ns_conc + ns_chim;
        const int64_t n_slow = hc.n_slow;
        if (n_short <= short_cap && (!do_edges || (n_raw <= cap && ns_conc <= conc_sens_cap && n_slow <= slow_cap))) break;
        slow_cap = std::max(slow_cap, n_slow + 4096);
        short_cap = std::max(short_cap, n_short + 4096);
        if (attempt + 1 == kEdgeAttempts) FAIL(SQG_ENOMEM, "raw edge / sensitive read / short block buffer overflow");
        cap = std::max(cap, n_raw + 4096);  // rerun with room for everything (counters are reset, the chimeric blocks restored from their pristine copies)
        sens_cap = std::max<int64_t>(sens_cap, (int64_t)ns_conc + ctx->c_n_reads + 4096);
    }
    if (do_depth) {
        ctx->n_short_other = n_short; ctx->n_unstable_other = n_unstable;
        const int rc = count_short_other(ctx, n_short, n_unstable);
        if (rc) return rc;
    }
    PHASE_END(do_depth ? "depth_edges" : "edges_only");
    if (do_edges) {
        ctx->n_raw_edges = n_raw;
        PHASE_BEGIN("edge_sort");
        const int rc = reduce_edges(ctx, n_raw, ctx->d_ew.p);
        if (rc) return rc;
        PHASE_END("edge_sort");
    }
    return SQG_OK;
}

extern "C" int sqg_shard_hint_state(sqg_ctx *ctx, int32_t *lead_sensitive, int32_t *out_hint) {
    if (!ctx || !lead_sensitive || !out_hint) return SQG_EINVAL;
    if (!ctx->have_edge_table) FAIL(SQG_ESTATE, "no edge table yet");
    *lead_sensitive = ctx->shard_lead_sensitive; *out_hint = ctx->shard_out_hint;
    return SQG_OK;
}
extern "C" int sqg_shard_redo_edges(sqg_ctx *ctx, int32_t init_hint) {
    if (!ctx) return SQG_EINVAL;
    if (!ctx->have_nodes || !ctx->shard_seeded) FAIL(SQG_ESTATE, "sqg_shard_build must run first");
    CK(cudaSetDevice(ctx->device));
    ctx->shard_init_hint = init_hint;
    return run_assign(ctx, false, true);
}


// sort raw keys, run-length reduce, unpack
static int reduce_edges(sqg_ctx *ctx, int64_t n_raw, const int32_t *d_weights_in) {
    ctx->n_unique_edges = 0;
    CK(ctx->d_ekeys2.ensure(n_raw + 1)); CK(ctx->d_ukeys.ensure(n_raw + 1)); CK(ctx->d_ecount.ensure(n_raw + 1));
    if (n_raw > 0) {
        int32_t *d_nu = &ctx->cnt.d.p->n_unique;
        if (!d_weights_in) {
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortKeys(t, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, (int)n_raw, 0, 64, ctx->stream); }));
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRunLengthEncode::Encode(t, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_ecount.p, d_nu, (int)n_raw, ctx->stream); }));
        } else {
            CK(ctx->d_sens.ensure(n_raw + 1));
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortPairs(t, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, d_weights_in, ctx->d_sens.p, (int)n_raw, 0, 64, ctx->stream); }));
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceReduce::ReduceByKey(t, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_sens.p, ctx->d_ecount.p, d_nu, cub::Sum(), (int)n_raw, ctx->stream); }));
        }
        ctx->launches += 5;
        CK(ctx->cnt.to_host(ctx->stream, d_nu));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->n_unique_edges = ctx->cnt.h.p->n_unique;
    }
    ctx->have_edge_table = true;
    return SQG_OK;
}

static int export_edges(sqg_ctx *ctx, int32_t **ind1, int32_t **ind2, uint8_t **heads, int32_t **weight, int64_t *n_edges) {
    const int64_t m = ctx->n_unique_edges;
    CK(ctx->d_e_ind1.ensure(m + 1)); CK(ctx->d_e_ind2.ensure(m + 1)); CK(ctx->d_e_w.ensure(m + 1)); CK(ctx->d_e_heads.ensure(m + 1));
    CK(ctx->h_ind1.ensure(m + 1)); CK(ctx->h_ind2.ensure(m + 1)); CK(ctx->h_w.ensure(m + 1)); CK(ctx->h_heads.ensure(m + 1));
    if (m > 0) {
        LAUNCH(k_unpack_edges, blocks_for(m), kThreads, ctx->d_ukeys.p, ctx->d_ecount.p, m, ctx->d_e_ind1.p, ctx->d_e_ind2.p, ctx->d_e_heads.p, ctx->d_e_w.p);
        CK(cudaMemcpyAsync(ctx->h_ind1.p, ctx->d_e_ind1.p, m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_ind2.p, ctx->d_e_ind2.p, m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_w.p, ctx->d_e_w.p, m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_heads.p, ctx->d_e_heads.p, m, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    // BuildEdges drops Weight <= 0 (:1953-1957): weights here are run lengths, always > 0
    *ind1 = ctx->h_ind1.p; *ind2 = ctx->h_ind2.p; *heads = ctx->h_heads.p; *weight = ctx->h_w.p; *n_edges = m;
    return SQG_OK;
}

extern "C" int sqg_build_edges(sqg_ctx *ctx, int32_t **ind1, int32_t **ind2, uint8_t **heads, int32_t **weight, int64_t *n_edges, sqg_chimeric *chim_inout) {
    if (!ctx || !ind1 || !ind2 || !heads || !weight || !n_edges) return SQG_EINVAL;
    if (!ctx->have_batch || !ctx->have_chim || !ctx->have_nodes) FAIL(SQG_ESTATE, "build_edges needs the concordant batch, the chimeric reads and a segment table");
    if (chim_inout && (chim_inout->n_reads != ctx->c_n_reads || chim_inout->n_blk != ctx->c_n_blk)) FAIL(SQG_EINVAL, "chim_inout does not match the loaded chimeric reads");
    CK(cudaSetDevice(ctx->device));
    int rc = run_classify(ctx);
    if (rc) return rc;
    rc = finish_prepass(ctx);
    if (rc) return rc;
    if (!ctx->have_edge_table) {  // sqg_build_nodes computes the table eagerly; sqg_set_nodes invalidates it
        rc = run_assign(ctx, false, true);
        if (rc) return rc;
    }
    if (chim_inout && ctx->c_n_blk > 0) {  // LocateRead trimmed Chimrecord in place (:1229-1248): patch the caller's arrays
        const int64_t nb = ctx->c_n_blk;
        // an earlier call on this context may have patched the same arrays for another segment table: back to the loaded values
        for (const sqg_ctx::ChimPatch &u : ctx->chim_undo) {
            chim_inout->blk_ref_pos[u.k] = u.v[0]; chim_inout->blk_read_pos[u.k] = u.v[1]; chim_inout->blk_match_ref[u.k] = u.v[2]; chim_inout->blk_match_read[u.k] = u.v[3];
        }
        ctx->chim_undo.clear();
        int64_t cap = std::max<int64_t>((int64_t)ctx->d_chimdiff.cap / 5, 4096);
        for (int attempt = 0; attempt < 2; attempt++) {
            CK(ctx->d_chimdiff.ensure((size_t)cap * 5));
            int32_t *d_nd = &ctx->cnt.d.p->n_chim_diff;
            CK(ctx->cnt.zero(ctx->stream, d_nd));
            LAUNCH(k_chim_diff, blocks_for(nb), kThreads, ctx->dc0_ref_pos.p, ctx->dc0_read_pos.p, ctx->dc0_match_ref.p, ctx->dc0_match_read.p,
                   ctx->dc_ref_pos.p, ctx->dc_read_pos.p, ctx->dc_match_ref.p, ctx->dc_match_read.p, nb, ctx->d_chimdiff.p, (int32_t)std::min<int64_t>(cap, 0x7fffffff), d_nd);
            CK(ctx->cnt.to_host(ctx->stream, d_nd));
            CK(cudaStreamSynchronize(ctx->stream));
            const int64_t nd = ctx->cnt.h.p->n_chim_diff;
            if (nd <= cap) {
                CK(ctx->h_chimdiff.ensure((size_t)nd * 5 + 1));
                if (nd > 0) {
                    CK(cudaMemcpyAsync(ctx->h_chimdiff.p, ctx->d_chimdiff.p, (size_t)nd * 5 * 4, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                }
                ctx->chim_undo.reserve((size_t)nd);
                for (int64_t i = 0; i < nd; i++) {
                    const int32_t *row = ctx->h_chimdiff.p + 5 * i;
                    const int32_t k = row[0];
                    ctx->chim_undo.push_back(sqg_ctx::ChimPatch{k, {chim_inout->blk_ref_pos[k], chim_inout->blk_read_pos[k], chim_inout->blk_match_ref[k], chim_inout->blk_match_read[k]}});
                    chim_inout->blk_ref_pos[k] = row[1]; chim_inout->blk_read_pos[k] = row[2]; chim_inout->blk_match_ref[k] = row[3]; chim_inout->blk_match_read[k] = row[4];
                }
                break;
            }
            cap = nd + 16;
        }
    }
    return export_edges(ctx, ind1, ind2, heads, weight, n_edges);
}

extern "C" int sqg_edges_device_table(sqg_ctx *ctx, uint64_t **d_keys, int32_t **d_weights, int64_t *n) {
    if (!ctx || !d_keys || !d_weights || !n) return SQG_EINVAL;
    if (!ctx->have_edge_table) FAIL(SQG_ESTATE, "no edge table: call sqg_build_edges first");
    *d_keys = ctx->d_ukeys.p; *d_weights = ctx->d_ecount.p; *n = ctx->n_unique_edges;
    return SQG_OK;
}

extern "C" int sqg_merge_edge_tables(sqg_ctx *ctx, const uint64_t *d_keys, const int32_t *d_weights, int64_t n,
                                     int32_t **ind1, int32_t **ind2, uint8_t **heads, int32_t **weight, int64_t *n_edges) {
    if (!ctx || n < 0 || !ind1 || !ind2 || !heads || !weight || !n_edges) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    PHASE_BEGIN("edge_merge");
    CK(ctx->d_ekeys.ensure(n + 1));
    if (n > 0) CK(cudaMemcpyAsync(ctx->d_ekeys.p, d_keys, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    int rc = reduce_edges(ctx, n, d_weights);
    if (rc) return rc;
    PHASE_END("edge_merge");
    return export_edges(ctx, ind1, ind2, heads, weight, n_edges);
}
