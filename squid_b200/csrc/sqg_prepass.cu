// The chimeric reads: their upload and the chimeric pre-pass on the device, and std::sort's permutation reproduced on the device
// (with the CPU twin behind it) for every stage that needs it.
#include <cub/cub.cuh>

#include <algorithm>
#include <vector>

#include "sq_gpusort.cuh"
#include "sq_prepass.cuh"
#include "sqg_ctx.cuh"
#include "host/prepass.h"

using namespace sq;

// test hook: does the device sort reproduce std::sort's permutation (payload included) on n keys drawn from [0,range)?
// 1 yes, 0 no, < 0 CUDA error, 2/3: the device sort declined (depth budget) -- patterns as sqh_selftest_sort
extern "C" int sqg_selftest_gpu_sort(int32_t device, int64_t n, uint64_t seed, uint64_t range, int32_t pattern, float *ms_out) {
    if (cudaSetDevice(device) != cudaSuccess) return -1;
    std::vector<sqh::SortKey> a((size_t)n);
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1;
    for (int64_t i = 0; i < n; i++) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        uint64_t v = range ? x % range : 0;
        if (pattern == 1) v = (uint64_t)i / 3;
        else if (pattern == 2) v = (uint64_t)(n - i) / 3;
        else if (pattern == 3) v = (uint64_t)std::min(i, n - 1 - i);
        a[(size_t)i] = sqh::SortKey{v, (uint32_t)i};
    }
    std::vector<uint64_t> hk((size_t)n); std::vector<uint32_t> hi((size_t)n);
    for (int64_t i = 0; i < n; i++) { hk[(size_t)i] = a[(size_t)i].key; hi[(size_t)i] = a[(size_t)i].k; }
    std::sort(a.begin(), a.end(), [](const sqh::SortKey &p, const sqh::SortKey &q) { return p.key < q.key; });
    DBuf<uint64_t> dk; DBuf<uint32_t> di; DBuf<unsigned char> ds;
    cudaStream_t st;
    int verdict = -1;
    if (cudaStreamCreate(&st) != cudaSuccess) return -1;
    if (dk.ensure((size_t)n + 1) == cudaSuccess && di.ensure((size_t)n + 1) == cudaSuccess && ds.ensure(gsort::bytes_needed((size_t)n)) == cudaSuccess) {
        cudaMemcpy(dk.p, hk.data(), (size_t)n * 8, cudaMemcpyHostToDevice); cudaMemcpy(di.p, hi.data(), (size_t)n * 4, cudaMemcpyHostToDevice);
        cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, st);
        const int rc = gsort::sort_like_std_device(dk.p, di.p, (size_t)n, ds.p, st, nullptr);
        cudaEventRecord(e1, st); cudaEventSynchronize(e1);
        if (ms_out) cudaEventElapsedTime(ms_out, e0, e1);
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        if (rc != 0) verdict = rc;
        else {
            cudaMemcpy(hk.data(), dk.p, (size_t)n * 8, cudaMemcpyDeviceToHost); cudaMemcpy(hi.data(), di.p, (size_t)n * 4, cudaMemcpyDeviceToHost);
            verdict = cudaGetLastError() == cudaSuccess ? 1 : -2;
            for (int64_t i = 0; verdict == 1 && i < n; i++) if (a[(size_t)i].key != hk[(size_t)i] || a[(size_t)i].k != hi[(size_t)i]) verdict = 0;
        }
    }
    cudaStreamDestroy(st);
    return verdict;
}

// The chimeric pre-pass on the device (sq_prepass.cuh), run by the pre-pass thread on stream3 beside the classification: the
// chimeric arrays are in HBM already (this thread uploaded them), the products never touch the host -- only their sizes do.
// Reads without blocks, or no reads, push nothing: the zeroed sentinel alone, no groups, PartAlignPos = n_ref entries (0, 0).
#define PCK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return (int)e_; } while (0)
static int device_prepass(sqg_ctx *ctx, size_t nr) {
    cudaStream_t st = ctx->stream3;
    const int32_t n_ref = ctx->params.n_ref;
    PreChim c;
    c.n_reads = (int64_t)nr; c.read_off = ctx->dc_read_off.p; c.n_first = ctx->dc_n_first.p; c.first_total = ctx->dc_first_total.p; c.second_total = ctx->dc_second_total.p;
    c.first_low = ctx->dc_first_low.p; c.second_low = ctx->dc_second_low.p; c.multi = ctx->dc_multi.p;
    c.chr = ctx->dc_ref_id.p; c.pos = ctx->dc0_ref_pos.p; c.rpos = ctx->dc0_read_pos.p; c.mref = ctx->dc0_match_ref.p; c.mread = ctx->dc0_match_read.p; c.rev = ctx->dc_rev.p;
    PCK(ctx->d_pre_ndis.ensure(nr + 1)); PCK(ctx->d_pre_pusher.ensure(nr + 1)); PCK(ctx->d_pre_lastk.ensure(nr + 1)); PCK(ctx->d_pre_off.ensure(nr + 2));
    PCK(ctx->d_pre_part.ensure(4 * nr + n_ref + 1)); PCK(ctx->d_pre_part2.ensure(4 * nr + n_ref + 1)); PCK(ctx->pre_cnt.ensure());
    PreCounters *dc = ctx->pre_cnt.d.p, *hc = ctx->pre_cnt.h.p;
    int64_t launches = 0;
    PCK(cudaMemsetAsync(ctx->d_pre_ndis.p + nr, 0, 4, st));
    k_pre_count<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_ndis.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p);
    PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, ctx->d_pre_ndis.p, ctx->d_pre_off.p, (int)(nr + 1), st); }));
    PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveScan(t, tb, ctx->d_pre_pusher.p, ctx->d_pre_pusher.p, MaxI32(), (int32_t)-1, (int)nr, st); }));
    PCK(cudaMemcpyAsync(&hc->n_disc, ctx->d_pre_off.p + nr, 8, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
    const int64_t nD = hc->n_disc;
    if (nD >= 0x7fffff00ll) return (int)cudaErrorInvalidValue;
    PCK(ctx->d_gs_keys.ensure((size_t)nD + 1)); PCK(ctx->d_gs_idx.ensure((size_t)nD + 1));
    PCK(ctx->d_disc.ensure((size_t)nD + 1)); PCK(ctx->d_pre_endkey.ensure((size_t)nD + 1)); PCK(ctx->d_pre_excl.ensure((size_t)nD + 1)); PCK(ctx->d_pre_incl.ensure((size_t)nD + 1));
    PCK(ctx->d_pre_opens.ensure((size_t)nD + 1)); PCK(ctx->d_pre_open.ensure((size_t)nD + 1));
    // PartAlignPos is resize()d to n_ref entries (0, 0) and then appended to (:203-204)
    PCK(cudaMemsetAsync(ctx->d_pre_part.p, 0, (size_t)n_ref * 8, st));
    const unsigned long long np0 = (unsigned long long)n_ref;
    PCK(cudaMemcpyAsync(&dc->n_part, &np0, 8, cudaMemcpyHostToDevice, st));
    k_pre_write<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_off.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p, ctx->d_gs_keys.p, ctx->d_gs_idx.p, ctx->d_pre_part.p, &dc->n_part);
    PCK(ctx->pre_cnt.to_host(st, &dc->n_part));
    launches += 6;
    // std::sort's permutation of bamdiscordant (:264): tie order is observable (SURVEY.md App. A-11).  A decline refills the keys
    // by running k_pre_write again, which appends to PartAlignPos again from its n_ref leading entries.
    int rc = 0;
    const cudaError_t se = replay_std_sort(ctx->d_gs_keys.p, ctx->d_gs_idx.p, (size_t)nD, ctx->d_gs_scratch, st, &launches, 8, [&]() {
        const unsigned long long np1 = (unsigned long long)n_ref;
        const cudaError_t e = cudaMemcpyAsync(&dc->n_part, &np1, 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess)
            k_pre_write<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_off.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p, ctx->d_gs_keys.p, ctx->d_gs_idx.p, ctx->d_pre_part.p, &dc->n_part);
        return e;
    }, &rc);
    ctx->gs_last_status = rc;
    PCK(se);
    PCK(cudaStreamSynchronize(st));
    const int64_t nP = (int64_t)hc->n_part;
    PCK(ctx->d_pchr.ensure((size_t)nP + 1)); PCK(ctx->d_ppos.ensure((size_t)nP + 1));
    {   // sort(PartAlignPos) by (chr, pos) (:262): a total order on the values, any stable or unstable sort agrees
        int key_bits = 33;
        while (key_bits < 64 && (1ll << (key_bits - 32)) < (long long)n_ref) key_bits++;
        PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortKeys(t, tb, ctx->d_pre_part.p, ctx->d_pre_part2.p, (int)nP, 0, key_bits, st); }));
        k_pre_split_part<<<blocks_for(nP), kThreads, 0, st>>>(ctx->d_pre_part2.p, nP, ctx->d_pchr.p, ctx->d_ppos.p);
        launches += 4;
    }
    k_pre_gather<<<blocks_for(nD + 1), kThreads, 0, st>>>(c, ctx->d_gs_idx.p, nD, ctx->d_disc.p, ctx->d_pre_endkey.p);
    int32_t nG = 0;
    if (nD > 0) {
        PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveScan(t, tb, ctx->d_pre_endkey.p, ctx->d_pre_excl.p, MaxU64(), (uint64_t)0, (int)nD, st); }));
        PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceScan::InclusiveScan(t, tb, ctx->d_pre_endkey.p, ctx->d_pre_incl.p, MaxU64(), (int)nD, st); }));
        k_pre_opens<<<blocks_for(nD), kThreads, 0, st>>>(ctx->d_disc.p, ctx->d_pre_excl.p, nD, ctx->params.read_len, ctx->d_pre_opens.p);
        cub::CountingInputIterator<int32_t> cnt(0);
        PreOpenOp op{ctx->d_pre_opens.p};
        PCK(cub_call(ctx->d_temp3, [&](void *t, size_t &tb) { return cub::DeviceSelect::If(t, tb, cnt, ctx->d_pre_open.p, &dc->n_groups, (int)nD, op, st); }));
        PCK(ctx->pre_cnt.to_host(st, &dc->n_groups));
        PCK(cudaStreamSynchronize(st));
        nG = hc->n_groups;
        PCK(ctx->d_groups.ensure((size_t)nG + 1));
        k_pre_groups<<<blocks_for(nG), kThreads, 0, st>>>(ctx->d_disc.p, ctx->d_pre_open.p, &dc->n_groups, ctx->d_pre_excl.p, ctx->d_pre_incl.p, nD, ctx->d_groups.p);
        launches += 9;
    } else PCK(ctx->d_groups.ensure(1));
    PCK(cudaGetLastError());
    ctx->pre_nD = (int32_t)nD; ctx->pre_nG = nG; ctx->pre_nP = (int32_t)nP;
    ctx->gs_launches += launches;
    if (ctx->shard_count > 1) {  // a range shard looks its first group up on the host (seed_stage: g_lo)
        ctx->h_groups.resize((size_t)nG);
        if (nG) PCK(cudaMemcpyAsync(ctx->h_groups.data(), ctx->d_groups.p, (size_t)nG * sizeof(Group), cudaMemcpyDeviceToHost, st));
        PCK(cudaStreamSynchronize(st));
    }
    return 0;
}
#undef PCK

extern "C" int sqg_load_chimeric(sqg_ctx *ctx, const sqg_chimeric *c) {
    if (!ctx || !c || c->n_reads < 0 || c->n_blk < 0) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    // the pre-pass and the uploads index the block arrays through read_off: it has to start at 0, never decrease and end at n_blk
    if (c->n_reads > 0 && (c->read_off[0] != 0 || (int64_t)c->read_off[c->n_reads] != c->n_blk)) FAIL(SQG_EINVAL, "chimeric reads: read_off does not span [0, n_blk]");
    if (c->n_reads == 0 && c->n_blk != 0) FAIL(SQG_EINVAL, "chimeric reads: blocks without reads");
    for (int64_t i = 0; i < c->n_reads; i++) {
        if (c->read_off[i + 1] < c->read_off[i]) FAIL(SQG_EINVAL, "chimeric reads: read_off decreases");
        const uint32_t nb = c->read_off[i + 1] - c->read_off[i], nf = c->n_first[i];
        if (nf > nb || nf > (uint32_t)kMaxBlocks || nb - nf > (uint32_t)kMaxBlocks) FAIL(SQG_EUNSUPPORTED, "chimeric read with more than 16 blocks in one mate");
    }
    // The upload of the chimeric reads and their pre-pass (BuildNode_STAR part A) are driven by a host thread on stream3 while the
    // caller's stream copies and classifies the concordant batch; they are joined in sqg_build_nodes / sqg_build_edges.
    ctx->prepass_worker.wait();
    ctx->chim_view = *c;
    ctx->chim_undo.clear();  // fresh arrays: nothing of an earlier patch applies
    ctx->prepass_uploaded = false;
    ctx->c_n_reads = c->n_reads; ctx->c_n_blk = c->n_blk;
    const size_t nr = (size_t)c->n_reads, nb = (size_t)c->n_blk;
    CK(ctx->dc_read_off.ensure(nr + 1)); CK(ctx->dc_n_first.ensure(nr + 1)); CK(ctx->dc_first_total.ensure(nr + 1)); CK(ctx->dc_second_total.ensure(nr + 1));
    CK(ctx->dc_ref_id.ensure(nb + 1)); CK(ctx->dc_ref_pos.ensure(nb + 1)); CK(ctx->dc_read_pos.ensure(nb + 1)); CK(ctx->dc_match_ref.ensure(nb + 1));
    CK(ctx->dc_match_read.ensure(nb + 1)); CK(ctx->dc_rev.ensure(nb + 1));
    CK(ctx->dc0_ref_pos.ensure(nb + 1)); CK(ctx->dc0_read_pos.ensure(nb + 1)); CK(ctx->dc0_match_ref.ensure(nb + 1)); CK(ctx->dc0_match_read.ensure(nb + 1));
    CK(ctx->dc_first_low.ensure(nr + 1)); CK(ctx->dc_second_low.ensure(nr + 1)); CK(ctx->dc_multi.ensure(nr + 1));
    // the previous edge pass may still read the device copies: the uploads are ordered behind everything enqueued so far
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->stream3, ctx->ev_fork, 0));
    ctx->chim_upload_err = 0;
    ctx->chim_upload_pending = true;
    {   // "prepass" phase timer: created here, on the caller's thread (the map is not touched by the pre-pass thread, only its events)
        PhaseTimer &t = ctx->timers["prepass"];
        if (!t.a) { CK(cudaEventCreate(&t.a)); CK(cudaEventCreate(&t.b)); }
        t.done = false;
        ctx->prepass_timer = &t;
    }
    ctx->prepass_worker.submit([ctx, nr, nb]() {
        // the chimeric arrays first, then the pre-pass itself on the device (sq_prepass.cuh): nothing of it runs on the cores
        cudaSetDevice(ctx->device);
        const sqg_chimeric &c = ctx->chim_view;
        cudaError_t e = cudaEventRecord(ctx->prepass_timer->a, ctx->stream3);
#define UPW(buf, src, cnt) do { if (e == cudaSuccess && (cnt)) e = cudaMemcpyAsync(ctx->buf.p, (src), (cnt) * sizeof(*(src)), cudaMemcpyHostToDevice, ctx->stream3); } while (0)
        UPW(dc_read_off, c.read_off, nr + 1); UPW(dc_n_first, c.n_first, nr);
        UPW(dc_first_total, c.first_total_len, nr); UPW(dc_second_total, c.second_total_len, nr);
        UPW(dc_first_low, c.first_lowphred, nr); UPW(dc_second_low, c.second_lowphred, nr); UPW(dc_multi, c.multi_filter, nr);
        UPW(dc_ref_id, c.blk_ref_id, nb); UPW(dc0_ref_pos, c.blk_ref_pos, nb); UPW(dc0_read_pos, c.blk_read_pos, nb);
        UPW(dc0_match_ref, c.blk_match_ref, nb); UPW(dc0_match_read, c.blk_match_read, nb); UPW(dc_rev, c.blk_is_reverse, nb);
#undef UPW
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_chim, ctx->stream3);
        ctx->chim_upload_err = (int)e;
        int rc = e == cudaSuccess ? device_prepass(ctx, nr) : (int)e;
        if (rc == 0) rc = (int)cudaEventRecord(ctx->ev_pre, ctx->stream3);
        if (rc == 0) { rc = (int)cudaEventRecord(ctx->prepass_timer->b, ctx->stream3); ctx->prepass_timer->done = rc == 0; }
        ctx->pre_upload_err = rc;
    });
    ctx->have_chim = true; ctx->have_edge_table = false;
    return SQG_OK;
}

// join the pre-pass thread: the caller's stream waits for the pre-pass products (discordant blocks, groups, PartAlignPos)
int finish_prepass(sqg_ctx *ctx) {
    ctx->prepass_worker.wait();
    if (ctx->prepass_uploaded) return SQG_OK;
    if (ctx->pre_upload_err) { ctx->err = std::string("upload of the pre-pass products: ") + cudaGetErrorString((cudaError_t)ctx->pre_upload_err); return SQG_ECUDA; }
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_pre, 0));
    ctx->prepass_uploaded = true;
    return SQG_OK;
}

// (sqg_ctx.cuh) the sort of bamdiscordant in the pre-pass and the replayed sort(ReadsOther) of the depth pass
cudaError_t replay_std_sort(uint64_t *keys, uint32_t *idx, size_t n, DBuf<unsigned char> &scratch, cudaStream_t st, int64_t *launches, int cpu_threads,
                            const std::function<cudaError_t()> &refill, int *status) {
    cudaError_t e = scratch.ensure(gsort::bytes_needed(n));
    if (e != cudaSuccess) { *status = -(int)e; return e; }
    const int rc = gsort::sort_like_std_device(keys, idx, n, scratch.p, st, launches);
    *status = rc;
    if (rc <= 0) return (cudaError_t)(-rc);
    // std::sort would have left the quicksort path (never seen on alignment data): the CPU twin, from a fresh copy of the keys
    std::vector<uint64_t> hk(n); std::vector<uint32_t> hi(n);
    e = refill();
    if (e == cudaSuccess) e = cudaMemcpyAsync(hk.data(), keys, n * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hi.data(), idx, n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return e;
    std::vector<sqh::SortKey> a(n);
    for (size_t i = 0; i < n; i++) a[i] = sqh::SortKey{hk[i], hi[i]};
    sqh::sort_keys_like_std(a.data(), a.data() + a.size(), cpu_threads);
    for (size_t i = 0; i < n; i++) { hk[i] = a[i].key; hi[i] = a[i].k; }
    e = cudaMemcpyAsync(keys, hk.data(), n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx, hi.data(), n * 4, cudaMemcpyHostToDevice, st);
    return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
}
