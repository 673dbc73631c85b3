// squid_b200 C ABI implementation: kernels for sm_100a + orchestration.  See include/squid_b200.h.
//
// Phase structure (DESIGN.md):
//   load      : batch -> HBM once, stays resident for the three phases
//   classify  : gate + duplicate filter + concordance class + otherrightmost scan  (phase-1 stream pass)
//   seed      : discordant-group state machine over the compacted gap/partial lists -> seed segments
//   tile      : normalise + tile the genome -> segment table
//   depth_edges: per-segment depth + read-to-segment assignment + raw edges        (phase-2 stream pass)
//   edge_sort : radix sort by packed key + run-length reduce
//   coverage  : breakpoint coverage with the reference's indBP lag                 (phase-3 stream pass)
// One translation unit per stage: sqg_load.cu and sqg_bam.cu (load), sqg_prepass.cu (the chimeric reads), sqg_classify.cu,
// sqg_nodes.cu (seed, tile), sqg_edges.cu (depth_edges, edge_sort), sqg_cov.cu (coverage).  This one holds the context's
// lifecycle, its statistics and ConnectedComponent.
#include <cub/cub.cuh>

#include <new>

#include "sq_cc.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

// ------------------------------------------------------------------------------------------------
// API
// ------------------------------------------------------------------------------------------------
extern "C" {

int sqg_create(sqg_ctx **out, const sqg_config *cfg, const int32_t *ref_len, int32_t n_ref, int32_t device) {
    if (!out || !cfg || !ref_len || n_ref <= 0) return SQG_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return SQG_ENODEVICE;
    if (cudaSetDevice(device) != cudaSuccess) return SQG_ENODEVICE;
    sqg_ctx *ctx = new (std::nothrow) sqg_ctx();
    if (!ctx) return SQG_ENOMEM;
    ctx->device = device;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // (numerically lower = more urgent)
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return SQG_ECUDA; }
    if (cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream_cov, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&ctx->ev_cov_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_cov_done, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream3, cudaStreamNonBlocking, prio_hi) != cudaSuccess || cudaEventCreateWithFlags(&ctx->ev_chim, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_pre, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return SQG_ECUDA; }
    ctx->params.min_mapq = cfg->min_mapq; ctx->params.max_lowphred_len = cfg->max_lowphred_len;
    ctx->params.concord_dist_pos = cfg->concord_dist_pos; ctx->params.concord_dist_idx = cfg->concord_dist_idx;
    ctx->params.read_len = cfg->read_len; ctx->params.n_ref = n_ref;
    ctx->ref_len.assign(ref_len, ref_len + n_ref);
    *out = ctx;
    if (!cfg->using_star) { ctx->err = "BWA mode (BuildNode_BWA / RawEdges) is not implemented"; return SQG_EUNSUPPORTED; }
    if (cfg->read_len <= 0) { ctx->err = "read_len must be > 0"; return SQG_EINVAL; }
    return SQG_OK;
}

void sqg_destroy(sqg_ctx *ctx) {
    if (!ctx) return;
    ctx->prepass_worker.stop();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->stream_cov) cudaStreamSynchronize(ctx->stream_cov);
    if (ctx->stream3) cudaStreamSynchronize(ctx->stream3);
    for (cudaEvent_t e : ctx->bam_ev) cudaEventDestroy(e);
    for (auto &kv : ctx->timers) { if (kv.second.a) cudaEventDestroy(kv.second.a); if (kv.second.b) cudaEventDestroy(kv.second.b); }
    cudaStreamDestroy(ctx->stream);
    if (ctx->stream3) cudaStreamDestroy(ctx->stream3);
    if (ctx->ev_chim) cudaEventDestroy(ctx->ev_chim);
    if (ctx->ev_pre) cudaEventDestroy(ctx->ev_pre);
    if (ctx->stream_cov) cudaStreamDestroy(ctx->stream_cov);
    if (ctx->stream_up) cudaStreamDestroy(ctx->stream_up);
    for (cudaEvent_t e : ctx->ev_up) cudaEventDestroy(e);
    if (ctx->ev_cov_fork) cudaEventDestroy(ctx->ev_cov_fork);
    if (ctx->ev_cov_done) cudaEventDestroy(ctx->ev_cov_done);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    delete ctx;  // (the buffers free themselves, on this device)
}

const char *sqg_last_error(const sqg_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

float sqg_phase_ms(const sqg_ctx *ctx, const char *name) {
    if (!ctx || !name) return -1.f;
    const auto acc = ctx->acc_ms.find(name);  // phases of a windowed BAM load: summed over the windows
    if (acc != ctx->acc_ms.end()) return acc->second;
    auto it = ctx->timers.find(name);
    if (it == ctx->timers.end() || !it->second.done) return -1.f;
    if (cudaEventSynchronize(it->second.b) != cudaSuccess) return -1.f;
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, it->second.a, it->second.b) != cudaSuccess) return -1.f;
    return ms;
}
int64_t sqg_launch_count(const sqg_ctx *ctx) { return ctx ? ctx->launches + ctx->gs_launches : 0; }
int64_t sqg_stat(const sqg_ctx *ctx, const char *name) {
    if (!ctx || !name) return -1;
    const std::string n(name);
    const Counters *hc = ctx->cnt.h.p;  // (-1 for its fields until a stage has allocated it)
    if (n == "islands") return ctx->n_islands;
    if (n == "device_sort_status") return ctx->gs_last_status;  // 0: the pre-pass sort ran on the device (also on no discordant blocks); 2/3: it declined, the cores sorted; -100: no pre-pass yet
    if (n == "heavy_islands") return ctx->n_heavy;
    if (n == "giant_islands") return 0;  // every island runs in one block or one warp
    if (n == "cov_chain_fallback") return ctx->cov_chain_fallback;
    if (n == "cov_chain_chunks") return ctx->cov_chain_chunks;
    if (n == "gap_records") return ctx->n_gap;
    if (n == "partial_records") return ctx->n_pc;
    if (n == "displaced_records") return ctx->n_dp;
    if (n == "lmax") return ctx->lmax;
    if (n == "groups") return ctx->pre_nG;
    if (n == "disc_blocks") return ctx->pre_nD;
    if (n == "sensitive_reads") return ctx->n_sensitive;
    if (n == "raw_edges") return ctx->n_raw_edges;
    if (n == "first_kept") return ctx->first_kept;                  // first record that is gate-passing and not a duplicate (n_rec: none)
    if (n == "end_other") return (int64_t)ctx->end_other;            // otherChr/otherrightmost key after the last record
    if (n == "classify_attempts") return ctx->classify_attempts;    // 2: the coverage-gap candidate buffer overflowed and phase 1 ran again
    if (n == "edge_pass_attempts") return ctx->edge_pass_attempts;  // > 1: a list of the last edge pass overflowed and the pass ran again
    if (n == "r_break") return ctx->r_break;
    if (n == "seed_window_records") return hc ? (int64_t)hc->win_count : -1;  // concordant-cluster window sizes summed over the groups
    if (n == "n_rec") return ctx->have_batch ? ctx->batch.n_rec : -1;
    if (n == "n_blk") return ctx->have_batch ? ctx->batch.n_blk : -1;
    if (n == "slow_records") return hc ? hc->n_slow : -1;  // records handled by k_edges_generic
    if (n == "qualifying_records") return ctx->cov_nq;
    if (n == "short_other_blocks") return ctx->n_short_other;        // ReadsOther blocks of <= 3 bp in the last depth pass
    if (n == "unstable_depth_blocks") return ctx->n_unstable_other;  // ... whose segment depends on the tie order of sort(ReadsOther): resolved by replaying that sort
    if (n == "other_sort_status") return ctx->other_sort_status;
    if (n == "edges_single_path") return hc ? (int64_t)hc->path_counts[0] : -1;
    if (n == "bam_members") return ctx->bam_members;                // BGZF members (with data) of the last sqg_load_concordant_bam
    if (n == "bam_windows") return ctx->bam_windows;
    if (n == "bam_repair_rounds") return ctx->bam_repair_rounds;    // rounds of segments walked again from their true entry, summed over the windows
    if (n == "edges_generic_path") return hc ? (int64_t)hc->path_counts[1] : -1;
    return -1;
}

}  // extern "C"


// SegmentGraph_t::ConnectedComponent on the device (sq_cc.cuh)
extern "C" int sqg_connected_components(int32_t device, int64_t n_nodes, const int32_t *ind1, const int32_t *ind2, int64_t n_edges, int32_t *label_out, int32_t *n_components) {
    if (n_nodes < 0 || n_edges < 0 || n_nodes >= 0x7fffff00ll || (n_edges > 0 && (!ind1 || !ind2)) || (n_nodes > 0 && !label_out)) return SQG_EINVAL;
    if (n_components) *n_components = 0;
    if (n_nodes == 0) return n_edges == 0 ? SQG_OK : SQG_EINVAL;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev || cudaSetDevice(device) != cudaSuccess) return SQG_ENODEVICE;
    cudaStream_t st;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return SQG_ECUDA;
    DBuf<int32_t> mem;  // one allocation per call: parent, flag, rank, e1, e2, bad and the scan's scratch, each 256-byte aligned
    int rc = SQG_OK;
    do {
#define CC_CK(x) if ((x) != cudaSuccess) { cudaGetLastError(); rc = SQG_ECUDA; break; }
        size_t tb = 0;
        CC_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, (int32_t *)nullptr, (int32_t *)nullptr, (int)n_nodes, st));
        auto words = [](size_t k) { return (k + 63) & ~(size_t)63; };
        const size_t wn = words((size_t)n_nodes), we = words((size_t)(n_edges ? n_edges : 1));
        CC_CK(mem.ensure(3 * wn + 2 * we + 64 + words(tb / 4 + 1)));
        int32_t *parent = mem.p, *flag = parent + wn, *rank = flag + wn, *e1 = rank + wn, *e2 = e1 + we, *bad = e2 + we;
        void *temp = bad + 64;
        CC_CK(cudaMemsetAsync(bad, 0, 4, st));
        if (n_edges) { CC_CK(cudaMemcpyAsync(e1, ind1, (size_t)n_edges * 4, cudaMemcpyHostToDevice, st)); CC_CK(cudaMemcpyAsync(e2, ind2, (size_t)n_edges * 4, cudaMemcpyHostToDevice, st)); }
        k_cc_init<<<blocks_for(n_nodes), kThreads, 0, st>>>(parent, n_nodes);
        if (n_edges) k_cc_hook<<<blocks_for(n_edges), kThreads, 0, st>>>(parent, e1, e2, n_edges, n_nodes, bad);
        k_cc_flatten<<<blocks_for(n_nodes), kThreads, 0, st>>>(parent, n_nodes, flag);
        CC_CK(cub::DeviceScan::ExclusiveSum(temp, tb, flag, rank, (int)n_nodes, st));
        k_cc_label<<<blocks_for(n_nodes), kThreads, 0, st>>>(parent, rank, n_nodes, flag);  // (flag is free again: the labels)
        CC_CK(cudaGetLastError());
        int32_t hbad = 0, last_rank = 0, last_root = 0;
        CC_CK(cudaMemcpyAsync(label_out, flag, (size_t)n_nodes * 4, cudaMemcpyDeviceToHost, st));
        CC_CK(cudaMemcpyAsync(&hbad, bad, 4, cudaMemcpyDeviceToHost, st));
        CC_CK(cudaMemcpyAsync(&last_rank, rank + (n_nodes - 1), 4, cudaMemcpyDeviceToHost, st));
        CC_CK(cudaMemcpyAsync(&last_root, parent + (n_nodes - 1), 4, cudaMemcpyDeviceToHost, st));
        CC_CK(cudaStreamSynchronize(st));
#undef CC_CK
        if (hbad) { rc = SQG_EINVAL; break; }
        if (n_components) *n_components = last_rank + (last_root == (int32_t)(n_nodes - 1) ? 1 : 0);
    } while (false);
    cudaStreamDestroy(st);
    return rc;
}
