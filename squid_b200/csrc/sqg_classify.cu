// Phase 1: the classification pass over the resident batch.
#include <cub/cub.cuh>

#include <algorithm>

#include "sq_phase1.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

// classify stage (phase 1): class bytes, gap / partial / displaced lists, first kept record, lmax; validates the batch
// Classification, part 1: buffers, counters and the kernel's argument block for a batch of n records (cand_cap candidates).
int classify_setup(sqg_ctx *ctx, int64_t cand_cap, P1Out &o) {
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec, n_tiles = (n + kTile - 1) / kTile;
    CK(ctx->d_cls.ensure(n + 4)); CK(ctx->d_flen.ensure(n + 4)); CK(ctx->d_scratch32.ensure(n + 1));
    CK(ctx->d_qstage_key.ensure((size_t)n + 1)); CK(ctx->d_qstage_end.ensure((size_t)n + 1));
    CK(ctx->d_tileagg.ensure(n_tiles + 1)); CK(ctx->d_chain64.ensure(n_tiles + 8)); CK(ctx->d_ccmax.ensure(n_tiles + 1)); CK(ctx->d_cov_nq.ensure(n_tiles + 2)); CK(ctx->d_cov_qmax.ensure(n_tiles + 2));
    CK(ctx->d_cand_key.ensure(cand_cap));
    o.cls = ctx->d_cls.p; o.first_len = ctx->d_flen.p; o.agg = ctx->d_tileagg.p; o.ccmax = ctx->d_ccmax.p; o.cov_nq = ctx->d_cov_nq.p; o.cov_qmax = ctx->d_cov_qmax.p; o.qstage_key = ctx->d_qstage_key.p; o.qstage_end = ctx->d_qstage_end.p; o.gate_word = ctx->d_chain64.p; o.n_tiles = (int32_t)n_tiles;
    o.cand_rec = ctx->d_scratch32.p; o.cand_key = ctx->d_cand_key.p; o.cand_cap = (int32_t)cand_cap;
    Counters *dc = ctx->cnt.d.p;
    CK(ctx->cnt.zero(ctx->stream, &dc->totals, &dc->bad_flags));
    CK(cudaMemsetAsync(ctx->d_chain64.p, 0, n_tiles * sizeof(uint64_t), ctx->stream));
    CK(cudaMemcpyAsync(&dc->first_kept, &n, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    o.first_kept = &dc->first_kept; o.lmax = &dc->lmax; o.n_cand = &dc->n_cand; o.ticket = &dc->ticket; o.bad_flags = &dc->bad_flags;
    {
        BatchDesc hd; hd.b = b; hd.p = ctx->params;
        CK(ctx->d_desc.ensure(sizeof(BatchDesc)));
        CK(cudaMemcpyAsync(ctx->d_desc.p, &hd, sizeof(BatchDesc), cudaMemcpyHostToDevice, ctx->stream));  // pageable source: staged before the call returns
        o.desc = (const BatchDesc *)ctx->d_desc.p;
    }
    CK(cudaFuncSetAttribute(k_classify_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmemBytes));
    return SQG_OK;
}
// part 2: the next `tiles` tiles of the batch (a tile takes its index from a ticket, so consecutive launches continue each other)
int classify_launch(sqg_ctx *ctx, const P1Out &o, int64_t tiles) {
    if (tiles <= 0) return SQG_OK;
    const DevBatch &b = ctx->batch;
    k_classify_tiles<<<(unsigned)tiles, kTileThreads, kTileSmemBytes, ctx->stream>>>(b, ctx->params, o, batch_bulk_ok(b) ? 1 : 0);
    ctx->launches++;
    CK(cudaGetLastError());
    return SQG_OK;
}

int run_classify(sqg_ctx *ctx) {
    if (ctx->classified) return SQG_OK;
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    PHASE_BEGIN("classify");
    CK(ctx->cnt.ensure());
    Counters *dc = ctx->cnt.d.p;
    const Counters &hc = *ctx->cnt.h.p;
    ctx->n_gap = 0; ctx->n_pc = 0; ctx->n_dp = 0; ctx->lmax = 0; ctx->first_kept = n; ctx->end_other = 0; ctx->classify_attempts = 0;
    if (n > 0) {
        const int64_t n_tiles = (n + kTile - 1) / kTile;
        int64_t cand_cap = std::max<int64_t>({(int64_t)ctx->d_cand_key.cap, n / 16, (int64_t)1 << 20});
        int32_t n_cand = 0;
        for (int attempt = 0; attempt < 2; attempt++) {
            cand_cap = std::min<int64_t>(cand_cap, n + 1);
            if (attempt == 0 && ctx->classify_prelaunched) {
                // the tile kernel already ran, chunk by chunk, behind the widening kernels of the wire upload
                cand_cap = ctx->pre_cand_cap;
                ctx->classify_prelaunched = false;
            } else {
                P1Out o;
                { const int rc_ = classify_setup(ctx, cand_cap, o); if (rc_) return rc_; }
                PHASE_BEGIN("k_classify");
                { const int rc_ = classify_launch(ctx, o, n_tiles); if (rc_) return rc_; }
                PHASE_END("k_classify");
            }
            LAUNCH(k_tile_scan, 1, 1024, ctx->d_tileagg.p, (int32_t)n_tiles, dc->totals, &dc->end_other);
            CK(ctx->cnt.to_host(ctx->stream, &dc->totals, &dc->end_other));
            if (ctx->wire_loaded) CK(ctx->cnt.to_host(ctx->stream, &dc->wire_bad));
            CK(cudaStreamSynchronize(ctx->stream));
            { const int rc_ = wire_check(ctx); if (rc_) return rc_; }
            const int32_t flags = hc.bad_flags;
            if (flags & 1) FAIL(SQG_EINVAL, "record with ref_id outside [-1, n_ref)");
            if (flags & 2) FAIL(SQG_EUNSUPPORTED, "mapped record with ref_id -1");
            if (flags & 4) FAIL(SQG_EUNSUPPORTED, "record with more than 16 aligned blocks or a decreasing blk_off");
            if (flags & 8) FAIL(SQG_EINVAL, "batch is not sorted by (ref_id, pos)");
            n_cand = hc.n_cand;
            ctx->classify_attempts = attempt + 1;
            if (!(flags & 16)) break;
            if (attempt == 1) FAIL(SQG_ENOMEM, "coverage-gap candidate buffer overflow");
            cand_cap = n + 1;  // every record can be a candidate at worst
        }
        ctx->n_pc = hc.totals[1]; ctx->n_dp = hc.totals[2]; ctx->first_kept = hc.first_kept; ctx->lmax = hc.lmax; ctx->end_other = hc.end_other;
        CK(ctx->d_gap.ensure((size_t)n_cand + 1)); CK(ctx->d_other.ensure((size_t)n_cand + 1));
        CK(ctx->d_pc.ensure((size_t)ctx->n_pc + 1)); CK(ctx->d_dp.ensure((size_t)ctx->n_dp + 1));
        if (n_cand > 0) {
            LAUNCH(k_finish_gaps, blocks_for(n_cand), kThreads, b, ctx->d_tileagg.p, ctx->d_scratch32.p, ctx->d_cand_key.p, n_cand, ctx->params.read_len, dc->totals);
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortPairs(t, tb, ctx->d_scratch32.p, ctx->d_gap.p, ctx->d_cand_key.p, ctx->d_other.p, n_cand, 0, 32, ctx->stream); }));
            ctx->launches += 3;
        }
        if (ctx->n_pc + ctx->n_dp > 0) LAUNCH(k_compact_lists, (unsigned)n_tiles, kTileThreads, ctx->d_cls.p, n, ctx->d_tileagg.p, ctx->d_pc.p, ctx->d_dp.p);
        CK(ctx->cnt.to_host(ctx->stream, &dc->totals));
        PHASE_END("classify");
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->n_gap = hc.totals[0];
    } else {
        PHASE_END("classify");
        CK(ctx->d_gap.ensure(1)); CK(ctx->d_other.ensure(1)); CK(ctx->d_pc.ensure(1)); CK(ctx->d_dp.ensure(1));
    }
    ctx->classified = true;
    return SQG_OK;
}

// Test seam of phase 1: one named output of the classification (run first if it has not run on the resident batch) copied to
// host memory.  Valid before sqg_build_nodes, which reuses some of these buffers.
extern "C" int sqg_classify_dump(sqg_ctx *ctx, const char *name, void *out, int64_t cap, int64_t *n_out) {
    if (!ctx || !name || !n_out || cap < 0) return SQG_EINVAL;
    if (!ctx->have_batch) FAIL(SQG_ESTATE, "no concordant batch");
    CK(cudaSetDevice(ctx->device));
    { const int rc = run_classify(ctx); if (rc) return rc; }
    const std::string k(name);
    const int64_t n = ctx->batch.n_rec, n_tiles = (n + kTile - 1) / kTile;
    const void *src = nullptr;
    int64_t cnt = 0;
    size_t elem = 0;
    if (k == "cls") { src = ctx->d_cls.p; cnt = n; elem = 1; }
    else if (k == "first_len") { src = ctx->d_flen.p; cnt = n; elem = 2; }
    else if (k == "gap_rec") { src = ctx->d_gap.p; cnt = ctx->n_gap; elem = 4; }
    else if (k == "gap_key") { src = ctx->d_other.p; cnt = ctx->n_gap; elem = 8; }
    else if (k == "pc_rec") { src = ctx->d_pc.p; cnt = ctx->n_pc; elem = 4; }
    else if (k == "dp_rec") { src = ctx->d_dp.p; cnt = ctx->n_dp; elem = 4; }
    else if (k == "okmax_excl") { cnt = n_tiles; elem = 8; }
    else if (k == "ccmax") { src = ctx->d_ccmax.p; cnt = n_tiles; elem = 4; }
    else if (k == "cov_nq") { src = ctx->d_cov_nq.p; cnt = n_tiles; elem = 4; }
    else if (k == "cov_qmax") { src = ctx->d_cov_qmax.p; cnt = n_tiles; elem = 8; }
    else if (k == "qstage_key") { src = ctx->d_qstage_key.p; cnt = n; elem = 8; }
    else if (k == "qstage_end") { src = ctx->d_qstage_end.p; cnt = n; elem = 4; }
    else FAIL(SQG_EINVAL, "sqg_classify_dump: unknown array " + k);
    *n_out = cnt;
    if (!out || cap < cnt || cnt == 0) return SQG_OK;
    if (k == "okmax_excl") {  // the okmax member of the tile aggregates (exclusive maxima after k_tile_scan)
        std::vector<TileAgg> agg((size_t)cnt);
        CK(cudaMemcpyAsync(agg.data(), ctx->d_tileagg.p, (size_t)cnt * sizeof(TileAgg), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int64_t t = 0; t < cnt; t++) ((uint64_t *)out)[t] = agg[(size_t)t].okmax;
        return SQG_OK;
    }
    CK(cudaMemcpyAsync(out, src, (size_t)cnt * elem, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SQG_OK;
}
