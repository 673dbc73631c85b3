// Making a concordant batch resident (host arrays, wire form, caller-owned device arrays), its download, the shard planner on the
// resident batch and cutting the batch down to one shard's records.
#include <cub/cub.cuh>

#include <algorithm>
#include <cstdlib>

#include "sq_plan.cuh"
#include "sq_wire.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

// ctx->batch = the context's own arrays (o_*) holding n_rec records and n_blk blocks
void point_batch_at_own_arrays(sqg_ctx *ctx, int64_t n_rec, int64_t n_blk) {
    DevBatch &b = ctx->batch;
    b.n_rec = n_rec; b.n_blk = n_blk;
#define X(T, name, ext) b.name = ctx->o_##name.p;
    SQ_BATCH_ARRAYS(X)
#undef X
}
// A new batch is resident: nothing computed on the previous one applies (the segment table, have_nodes, still does).  `wire`: its
// arrays come from the wire decode, whose consistency flag run_classify checks and whose classification may already be running
// (classify_prelaunched, set during that upload, stands); every other batch starts unclassified.
void reset_batch_state(sqg_ctx *ctx, bool owned, int64_t first_record_index, bool wire) {
    ctx->have_batch = true; ctx->batch_owned = owned; ctx->batch_restricted = false; ctx->first_record_index = first_record_index;
    ctx->classified = false; ctx->cov_compacted = false; ctx->have_edge_table = false; ctx->wire_loaded = wire;
    if (!wire) ctx->classify_prelaunched = false;
}
// A batch from the wire decode is refused when the decode flagged it; the caller has copied the flag to the mirror and synchronised.
int wire_check(sqg_ctx *ctx) {
    if (ctx->wire_loaded && ctx->cnt.h.p->wire_bad) FAIL(SQG_EINVAL, "wire batch is inconsistent (escape without an exception entry, or block counts that contradict the tile table)");
    return SQG_OK;
}

extern "C" int sqg_load_concordant(sqg_ctx *ctx, const sqg_batch *hb, int64_t first_record_index) {
    if (!ctx || !hb || hb->n_rec < 0 || hb->n_blk < 0) return SQG_EINVAL;
    if (hb->n_rec >= 0x7fffff00ll) FAIL(SQG_EUNSUPPORTED, "more than 2^31 records per context: shard the stream");
    // end points of the offset array (host memory: checked before anything is indexed with it; monotonicity and the 16-block limit
    // are checked on the device, where an offset is compared with n_blk before it is used)
    if (hb->n_rec > 0 && (hb->blk_off[0] != 0 || (int64_t)hb->blk_off[hb->n_rec] != hb->n_blk)) FAIL(SQG_EINVAL, "batch: blk_off does not span [0, n_blk]");
    if (hb->n_rec == 0 && hb->n_blk != 0) FAIL(SQG_EINVAL, "batch: blocks without records");
    CK(cudaSetDevice(ctx->device));
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    PHASE_BEGIN("h2d");
    const size_t n = (size_t)hb->n_rec, nb = (size_t)hb->n_blk;
#define X(T, name, ext)                                                                                                  \
    {                                                                                                                    \
        const size_t cnt = batch_extent(ext, n, nb);                                                                     \
        CK(ctx->o_##name.ensure(cnt ? cnt : 1));                                                                         \
        if (cnt) CK(cudaMemcpyAsync(ctx->o_##name.p, hb->name, cnt * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));  \
    }
    SQ_BATCH_ARRAYS(X)
#undef X
    point_batch_at_own_arrays(ctx, hb->n_rec, hb->n_blk);
    PHASE_END("h2d");
    reset_batch_state(ctx, true, first_record_index, false);
    return SQG_OK;
}

static_assert(kWireTile == kTile, "a wire tile is a classification tile");
// Wire-form upload: the chunks go down a copy stream; the main stream waits for each chunk's event and widens it
// (sq_wire.cuh) while the following chunks are on the bus.
extern "C" int sqg_load_concordant_wire(sqg_ctx *ctx, const sqg_wire *w, int64_t first_record_index) {
    if (!ctx || !w || w->n_rec < 0 || w->n_blk < 0 || w->n_rec_exc < 0 || w->n_blk_exc < 0 || w->n_wblk < 0 || w->n_wblk > w->n_blk) return SQG_EINVAL;
    if (w->n_rec >= 0x7fffff00ll) FAIL(SQG_EUNSUPPORTED, "more than 2^31 records per context: shard the stream");
    const int64_t n = w->n_rec, nb = w->n_blk, nt = w->n_tiles, nwb = w->n_wblk;
    if (nt != (n + kWireTile - 1) / kWireTile || nb > 0xFFFFFFFFll) return SQG_EINVAL;
    if (nt > 0) {  // the tile tables drive the copies and index the exception lists: checked here, everything else on the device
        if (w->tile_blk_off[0] != 0 || (int64_t)w->tile_blk_off[nt] != nb || w->tile_rec_exc_off[0] != 0 || (int64_t)w->tile_rec_exc_off[nt] != w->n_rec_exc ||
            w->tile_blk_exc_off[0] != 0 || (int64_t)w->tile_blk_exc_off[nt] != w->n_blk_exc || w->tile_wblk_off[0] != 0 || (int64_t)w->tile_wblk_off[nt] != nwb)
            FAIL(SQG_EINVAL, "wire batch: tile tables do not match the counts");
        bool mono = true;
#pragma omp parallel for schedule(static) reduction(&& : mono)
        for (long long t = 0; t < (long long)nt; t++)
            mono = mono && w->tile_blk_off[t] <= w->tile_blk_off[t + 1] && w->tile_rec_exc_off[t] <= w->tile_rec_exc_off[t + 1] && w->tile_blk_exc_off[t] <= w->tile_blk_exc_off[t + 1] &&
                   w->tile_wblk_off[t] <= w->tile_wblk_off[t + 1];
        if (!mono) FAIL(SQG_EINVAL, "wire batch: tile tables are not monotone");
    } else if (nb != 0 || nwb != 0) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    if (!ctx->stream_up) CK(cudaStreamCreateWithFlags(&ctx->stream_up, cudaStreamNonBlocking));
    PHASE_BEGIN("h2d");
    const size_t n1 = n ? (size_t)n : 1, nb1 = nb ? (size_t)nb : 1, nt1 = (size_t)nt + 1, nwb1 = nwb ? (size_t)nwb : 1;
#define X(T, name, ext) CK(ctx->o_##name.ensure(batch_extent(ext, n1, nb1)));
    SQ_BATCH_ARRAYS(X)
#undef X
    CK(ctx->w_dpos.ensure(n1)); CK(ctx->w_span.ensure(n1)); CK(ctx->w_dmate.ensure(n1)); CK(ctx->w_lp.ensure(n1)); CK(ctx->w_an.ensure(n1));
    CK(ctx->w_bdref.ensure(nwb1)); CK(ctx->w_bmref.ensure(nwb1)); CK(ctx->w_brpos.ensure(nwb1)); CK(ctx->w_bmread.ensure(nwb1)); CK(ctx->w_tile_wblk.ensure(nt1));
    CK(ctx->w_tile_ref.ensure(nt1)); CK(ctx->w_tile_pos.ensure(nt1)); CK(ctx->w_tile_blk.ensure(nt1)); CK(ctx->w_tile_rexc.ensure(nt1)); CK(ctx->w_tile_bexc.ensure(nt1));
    CK(ctx->w_rec_exc.ensure(w->n_rec_exc ? (size_t)w->n_rec_exc : 1)); CK(ctx->w_blk_exc.ensure(w->n_blk_exc ? (size_t)w->n_blk_exc : 1));
    CK(ctx->cnt.ensure());
    cudaStream_t up = ctx->stream_up;
    // the copy stream starts after everything the main stream still has queued on the previous batch
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream)); CK(cudaStreamWaitEvent(up, ctx->ev_fork, 0));
    CK(ctx->cnt.zero(ctx->stream, &ctx->cnt.d.p->wire_bad));
#define UPW(dst, src, off, cnt) do { if ((cnt) > 0) CK(cudaMemcpyAsync((dst) + (off), (src) + (off), (size_t)(cnt) * sizeof(*(src)), cudaMemcpyHostToDevice, up)); } while (0)
    if (nt > 0) {
        UPW(ctx->w_tile_ref.p, w->tile_ref_id, 0, nt); UPW(ctx->w_tile_pos.p, w->tile_pos, 0, nt);
        UPW(ctx->w_tile_blk.p, w->tile_blk_off, 0, nt + 1); UPW(ctx->w_tile_rexc.p, w->tile_rec_exc_off, 0, nt + 1); UPW(ctx->w_tile_bexc.p, w->tile_blk_exc_off, 0, nt + 1);
        UPW(ctx->w_tile_wblk.p, w->tile_wblk_off, 0, nt + 1);
        UPW(ctx->w_rec_exc.p, w->rec_exc, 0, w->n_rec_exc); UPW(ctx->w_blk_exc.p, w->blk_exc, 0, w->n_blk_exc);
    }
    WireDev wd;
    wd.n_rec = n; wd.n_blk = nb; wd.n_tiles = nt;
    wd.tile_ref_id = ctx->w_tile_ref.p; wd.tile_pos = ctx->w_tile_pos.p; wd.tile_blk_off = ctx->w_tile_blk.p; wd.tile_rec_exc_off = ctx->w_tile_rexc.p; wd.tile_blk_exc_off = ctx->w_tile_bexc.p;
    wd.dpos = ctx->w_dpos.p; wd.span = ctx->w_span.p; wd.dmate = ctx->w_dmate.p; wd.lowphred_run = ctx->w_lp.p; wd.aux_nblk = ctx->w_an.p;
    wd.blk_dref = ctx->w_bdref.p; wd.blk_match_ref16 = ctx->w_bmref.p; wd.blk_read_pos = ctx->w_brpos.p; wd.blk_match_read = ctx->w_bmread.p; wd.n_wblk = nwb;
    wd.tile_wblk_off = ctx->w_tile_wblk.p; wd.rec_exc = ctx->w_rec_exc.p; wd.blk_exc = ctx->w_blk_exc.p;
    WireOut wo;
    wo.ref_id = ctx->o_ref_id.p; wo.pos = ctx->o_pos.p; wo.mate_ref_id = ctx->o_mate_ref_id.p; wo.mate_pos = ctx->o_mate_pos.p; wo.end_pos = ctx->o_end_pos.p;
    wo.lowphred_run = ctx->o_lowphred_run.p; wo.aux = ctx->o_aux.p; wo.blk_off = ctx->o_blk_off.p; wo.blk_ref_pos = ctx->o_blk_ref_pos.p; wo.blk_match_ref = ctx->o_blk_match_ref.p;
    wo.blk_read_pos = ctx->o_blk_read_pos.p; wo.blk_match_read = ctx->o_blk_match_read.p;
    wo.bad = &ctx->cnt.d.p->wire_bad;
    point_batch_at_own_arrays(ctx, n, nb);
    // The classification tile kernel needs nothing but the batch: it follows every chunk's widening kernel on the main stream, so
    // that it, too, runs while the later chunks are on the bus (run_classify then only finishes: scans, lists).  A tile looks at
    // the first record of the NEXT tile (sortedness), so the last tile of a chunk waits for the next chunk.
    static const bool pre_classify = !(getenv("SQG_WIRE_CLASSIFY") && atoi(getenv("SQG_WIRE_CLASSIFY")) == 0);
    P1Out pre_o;
    ctx->classify_prelaunched = false;
    if (pre_classify && nt > 0) {
        ctx->pre_cand_cap = std::min<int64_t>(std::max<int64_t>({(int64_t)ctx->d_cand_key.cap, n / 16, (int64_t)1 << 20}), n + 1);
        const int rc_ = classify_setup(ctx, ctx->pre_cand_cap, pre_o);
        if (rc_) return rc_;
        ctx->classify_prelaunched = true;
    }
    int64_t tiles_classified = 0;
    static const int n_chunks_env = getenv("SQG_WIRE_CHUNKS") ? atoi(getenv("SQG_WIRE_CHUNKS")) : 16;
    const int64_t n_chunks = std::max<int64_t>(1, std::min<int64_t>(n_chunks_env, nt));
    while ((int64_t)ctx->ev_up.size() < n_chunks) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->ev_up.push_back(e); }
    for (int64_t c = 0; c < n_chunks && nt > 0; c++) {
        const int64_t t0 = nt * c / n_chunks, t1 = nt * (c + 1) / n_chunks;
        if (t1 <= t0) continue;
        const int64_t r0 = t0 * kWireTile, r1 = std::min<int64_t>(n, t1 * kWireTile), k0 = w->tile_wblk_off[t0], k1 = w->tile_wblk_off[t1];  // (explicit blocks only)
        UPW(ctx->w_dpos.p, w->dpos, r0, r1 - r0); UPW(ctx->w_span.p, w->span, r0, r1 - r0); UPW(ctx->w_dmate.p, w->dmate, r0, r1 - r0);
        UPW(ctx->w_lp.p, w->lowphred_run, r0, r1 - r0); UPW(ctx->w_an.p, w->aux_nblk, r0, r1 - r0);
        UPW(ctx->o_flag.p, w->flag, r0, r1 - r0); UPW(ctx->o_total_len.p, w->total_len, r0, r1 - r0); UPW(ctx->o_mapq.p, w->mapq, r0, r1 - r0);
        UPW(ctx->w_bdref.p, w->blk_dref, k0, k1 - k0); UPW(ctx->w_bmref.p, w->blk_match_ref, k0, k1 - k0);
        UPW(ctx->w_brpos.p, w->blk_read_pos, k0, k1 - k0); UPW(ctx->w_bmread.p, w->blk_match_read, k0, k1 - k0);
        CK(cudaEventRecord(ctx->ev_up[(size_t)c], up));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_up[(size_t)c], 0));
        k_wire_decode<<<(unsigned)(t1 - t0), kWireTile, 0, ctx->stream>>>(wd, wo, t0);
        ctx->launches++;
        CK(cudaGetLastError());
        if (ctx->classify_prelaunched) {
            const int64_t upto = t1 == nt ? nt : t1 - 1;
            const int rc_ = classify_launch(ctx, pre_o, upto - tiles_classified);
            if (rc_) return rc_;
            if (upto > tiles_classified) tiles_classified = upto;
        }
    }
#undef UPW
    if (n == 0) CK(cudaMemsetAsync(ctx->o_blk_off.p, 0, sizeof(uint32_t), ctx->stream));
    PHASE_END("h2d");
    reset_batch_state(ctx, true, first_record_index, true);
    return SQG_OK;
}


// (test / diagnostic) the resident batch back into host arrays
extern "C" int sqg_download_concordant(sqg_ctx *ctx, sqg_batch *out) {
    if (!ctx || !out) return SQG_EINVAL;
    if (!ctx->have_batch) FAIL(SQG_ESTATE, "no concordant batch loaded");
    const DevBatch &b = ctx->batch;
    if (out->n_rec != b.n_rec || out->n_blk != b.n_blk) FAIL(SQG_EINVAL, "sqg_download_concordant: n_rec / n_blk do not match the resident batch");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)b.n_rec, nb = (size_t)b.n_blk;
#define X(T, name, ext) if (const size_t cnt = batch_extent(ext, n, nb)) CK(cudaMemcpyAsync((void *)out->name, b.name, cnt * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    SQ_BATCH_ARRAYS(X)
#undef X
    if (ctx->wire_loaded) CK(ctx->cnt.to_host(ctx->stream, &ctx->cnt.d.p->wire_bad));
    CK(cudaStreamSynchronize(ctx->stream));
    return wire_check(ctx);
}

extern "C" int sqg_attach_concordant_device(sqg_ctx *ctx, const sqg_batch *db, int64_t first_record_index) {
    if (!ctx || !db || db->n_rec < 0 || db->n_blk < 0) return SQG_EINVAL;
    if (db->n_rec >= 0x7fffff00ll) FAIL(SQG_EUNSUPPORTED, "more than 2^31 records per context: shard the stream");
    CK(cudaSetDevice(ctx->device));
    if (ctx->cov_pending) { CK(cudaStreamSynchronize(ctx->stream_cov)); ctx->cov_pending = false; }  // the previous batch's arrays belong to the caller again
    DevBatch &b = ctx->batch;
    b.n_rec = db->n_rec; b.n_blk = db->n_blk;
#define X(T, name, ext) b.name = db->name;
    SQ_BATCH_ARRAYS(X)
#undef X
    reset_batch_state(ctx, false, first_record_index, false);
    return SQG_OK;
}


// host/plan.cpp's cuts from the resident batch (sq_plan.cuh): class bytes of the classification pass, groups of the chimeric
// pre-pass, three exclusive scans, one candidate per record, compacted and sent back; the greedy runs on the host.
static int plan_resident(sqg_ctx *ctx, int32_t n_shards, int64_t *cuts, int32_t *n_planned) {
    int rc = run_classify(ctx);
    if (rc) return rc;
    rc = finish_prepass(ctx);
    if (rc) return rc;
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    int64_t n_cand = 0;
    PHASE_BEGIN("plan");
    if (n > 0) {
        CK(ctx->d_plan_reach.ensure((size_t)n)); CK(ctx->d_plan_keep.ensure((size_t)n)); CK(ctx->d_plan_upd.ensure((size_t)n));
        CK(ctx->d_plan_cand.ensure((size_t)n)); CK(ctx->d_plan_sel.ensure((size_t)n));
        LAUNCH(k_plan_prep, blocks_for(n), kThreads, b, ctx->d_cls.p, ctx->d_plan_reach.p, ctx->d_plan_keep.p, ctx->d_plan_upd.p);
        int32_t *d_nsel = &ctx->cnt.d.p->n_plan_cand;
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveScan(t, tb, ctx->d_plan_reach.p, ctx->d_plan_reach.p, MaxU64(), (uint64_t)0, (int)n, ctx->stream); }));
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveScan(t, tb, ctx->d_plan_keep.p, ctx->d_plan_keep.p, MaxI32(), (int32_t)-1, (int)n, ctx->stream); }));
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveScan(t, tb, ctx->d_plan_upd.p, ctx->d_plan_upd.p, MaxI32(), (int32_t)-1, (int)n, ctx->stream); }));
        LAUNCH(k_plan_cands, blocks_for(n), kThreads, b, ctx->params, ctx->d_cls.p, ctx->d_plan_reach.p, ctx->d_plan_keep.p, ctx->d_plan_upd.p,
               ctx->d_groups.p, ctx->d_disc.p, ctx->pre_nG, ctx->d_plan_cand.p);
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceSelect::If(t, tb, ctx->d_plan_cand.p, ctx->d_plan_sel.p, d_nsel, (int)n, PlanIsCand(), ctx->stream); }));
        ctx->launches += 4;
        CK(ctx->cnt.to_host(ctx->stream, d_nsel));
        CK(cudaStreamSynchronize(ctx->stream));
        n_cand = ctx->cnt.h.p->n_plan_cand;
        CK(ctx->h_plan_sel.ensure((size_t)n_cand + 1));
        if (n_cand > 0) CK(cudaMemcpyAsync(ctx->h_plan_sel.p, ctx->d_plan_sel.p, (size_t)n_cand * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    PHASE_END("plan");
    CK(cudaStreamSynchronize(ctx->stream));
    *n_planned = plan_greedy(ctx->h_plan_sel.p, n_cand, n, n_shards, cuts);
    return SQG_OK;
}

extern "C" int sqg_plan_shards_resident(sqg_ctx *ctx, int32_t n_shards, int64_t *cuts, int32_t *n_planned) {
    if (!ctx || !cuts || !n_planned || n_shards < 1) return SQG_EINVAL;
    if (!ctx->have_batch || !ctx->have_chim) FAIL(SQG_ESTATE, "load the concordant batch and the chimeric reads first");
    if (ctx->batch_restricted) FAIL(SQG_ESTATE, "sqg_plan_shards_resident: the batch is one shard's range already (sqg_keep_records); plan on the whole stream");
    CK(cudaSetDevice(ctx->device));
    const int rc = plan_resident(ctx, n_shards, cuts, n_planned);
    // the scratch is as large as the batch and only needed once per load
    ctx->d_plan_reach.release(); ctx->d_plan_keep.release(); ctx->d_plan_upd.release(); ctx->d_plan_cand.release(); ctx->d_plan_sel.release();
    return rc;
}

// Records [lo, hi) of the resident batch become the batch, moved to the front of the context's own arrays: the tile loads of
// the classification pass (cp.async.bulk) need every array to start 16-byte aligned, which an offset pointer would not be.
extern "C" int sqg_keep_records(sqg_ctx *ctx, int64_t lo, int64_t hi) {
    if (!ctx) return SQG_EINVAL;
    if (!ctx->have_batch) FAIL(SQG_ESTATE, "no concordant batch loaded");
    if (!ctx->batch_owned) FAIL(SQG_ESTATE, "sqg_keep_records: the batch is attached (caller-owned device arrays)");
    if (lo < 0 || lo > hi || hi > ctx->batch.n_rec) FAIL(SQG_EINVAL, "sqg_keep_records: need 0 <= lo <= hi <= n_rec");
    CK(cudaSetDevice(ctx->device));
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    cudaStream_t st = ctx->stream;
    uint32_t ends[2];
    CK(cudaMemcpyAsync(&ends[0], ctx->o_blk_off.p + lo, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&ends[1], ctx->o_blk_off.p + hi, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (ends[1] < ends[0] || (int64_t)ends[1] > ctx->batch.n_blk) FAIL(SQG_EINVAL, "sqg_keep_records: blk_off of the batch is not monotone");
    const int64_t nr = hi - lo, b0 = ends[0], nb = (int64_t)ends[1] - b0;
    DBuf<uint8_t> tmp;  // a range that overlaps its destination goes through here
    CK(tmp.ensure((size_t)std::max<int64_t>(4 * (nr + 1), 4 * nb)));
    cudaError_t e = cudaSuccess;
    auto move = [&](void *arr, size_t elem, int64_t first, int64_t count) {
        char *p = (char *)arr;
        const size_t bytes = (size_t)count * elem;
        if (e != cudaSuccess || first == 0 || count == 0) return;
        if (first >= count) { e = cudaMemcpyAsync(p, p + (size_t)first * elem, bytes, cudaMemcpyDeviceToDevice, st); return; }
        e = cudaMemcpyAsync(tmp.p, p + (size_t)first * elem, bytes, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(p, tmp.p, bytes, cudaMemcpyDeviceToDevice, st);
    };
#define X(T, name, ext) if (ext != BX_OFF) move(ctx->o_##name.p, sizeof(T), ext == BX_REC ? lo : b0, ext == BX_REC ? nr : nb);
    SQ_BATCH_ARRAYS(X)  // (blk_off is rebased below)
#undef X
    CK(e);
    CK(cudaMemcpyAsync(tmp.p, ctx->o_blk_off.p + lo, (size_t)(nr + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    LAUNCH(k_keep_offsets, blocks_for(nr + 1), kThreads, ctx->o_blk_off.p, (const uint32_t *)tmp.p, nr + 1, (uint32_t)b0);
    CK(cudaStreamSynchronize(st));
    ctx->batch.n_rec = nr; ctx->batch.n_blk = nb;
    reset_batch_state(ctx, true, ctx->first_record_index + lo, ctx->wire_loaded);
    ctx->batch_restricted = true; ctx->classify_prelaunched = false;  // (a classification launched on the whole batch does not apply)
    return SQG_OK;
}
