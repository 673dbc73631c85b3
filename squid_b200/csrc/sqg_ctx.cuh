// Context of the C ABI: owns the CUDA stream, the HBM-resident batches, the segment table and all
// scratch.  One context per GPU per run (include/squid_b200.h).
#ifndef SQG_CTX_CUH
#define SQG_CTX_CUH
#include <cuda_runtime.h>

#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "sq_bam.cuh"
#include "sq_common.cuh"
#include "sq_seed.cuh"
#include "sq_phase1.cuh"
#include "sq_phase2.cuh"
#include "sq_phase3.cuh"
#include "sq_plan.cuh"
#include "squid_b200.h"

namespace sq {

// Device / pinned host buffers own their storage: freed by the destructor, or earlier by release().  Moves hand it over.
template <class T> struct DBuf {
    T *p = nullptr;
    size_t cap = 0;
    DBuf() = default;
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
    DBuf(DBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DBuf &operator=(DBuf &&o) noexcept { if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; } return *this; }
    ~DBuf() { release(); }
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 64;
        cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    // capacity for n elements keeping the first `used` (geometric growth: a batch whose size is only known window by window)
    cudaError_t grow(size_t n, size_t used, cudaStream_t st) {
        if (n <= cap) return cudaSuccess;
        const size_t want = n + n / 8 + 64 > 2 * cap ? n + n / 8 + 64 : 2 * cap;
        T *q = nullptr;
        cudaError_t e = cudaMalloc((void **)&q, want * sizeof(T));
        if (e != cudaSuccess) return e;
        if (used && p) e = cudaMemcpyAsync(q, p, used * sizeof(T), cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) { cudaFree(q); return e; }
        if (p) cudaFree(p);  // (waits for the device, so the copy is complete)
        p = q; cap = want;
        return cudaSuccess;
    }
};
template <class T> struct HBuf {  // pinned host
    T *p = nullptr;
    size_t cap = 0;
    HBuf() = default;
    HBuf(const HBuf &) = delete;
    HBuf &operator=(const HBuf &) = delete;
    HBuf(HBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    HBuf &operator=(HBuf &&o) noexcept { if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; } return *this; }
    ~HBuf() { release(); }
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 64;
        cudaError_t e = cudaMallocHost((void **)&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// One persistent host thread that runs one job at a time.
struct Worker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, busy = false, quit = false;
    void submit(std::function<void()> f) {
        wait();
        std::unique_lock<std::mutex> lk(m);
        if (!th.joinable()) th = std::thread([this]() { loop(); });
        job = std::move(f); has_job = true; busy = true;
        cv.notify_all();
    }
    void wait() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [this]() { return !busy; }); }
    void stop() {
        wait();
        { std::unique_lock<std::mutex> lk(m); quit = true; cv.notify_all(); }
        if (th.joinable()) th.join();
    }
    void loop() {
        for (;;) {
            std::function<void()> f;
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [this]() { return has_job || quit; });
                if (quit) return;
                f = std::move(job); has_job = false;
            }
            f();
            { std::unique_lock<std::mutex> lk(m); busy = false; cv.notify_all(); }
        }
    }
};

struct PhaseTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    bool done = false;
};

}  // namespace sq

struct sqg_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_fork = nullptr;
    // the coverage compaction (phase 3, first pass) runs beside the seed machine on its own stream
    cudaStream_t stream_cov = nullptr;
    cudaEvent_t ev_cov_fork = nullptr, ev_cov_done = nullptr;
    bool cov_pending = false;
    std::string err;
    sq::Params params{};
    std::vector<int32_t> ref_len;
    int64_t launches = 0;
    std::map<std::string, sq::PhaseTimer> timers;

    // concordant batch
    bool have_batch = false, batch_owned = false, classified = false, cov_compacted = false;
    bool batch_restricted = false;   // sqg_keep_records has cut the batch down to one shard's range
    int64_t first_record_index = 0;
    sq::DevBatch batch;
    sq::DBuf<int32_t> o_ref_id, o_pos, o_mate_ref_id, o_mate_pos, o_end_pos, o_blk_ref_pos, o_blk_match_ref;
    sq::DBuf<uint16_t> o_flag, o_total_len, o_lowphred_run, o_blk_read_pos, o_blk_match_read;
    sq::DBuf<uint8_t> o_mapq, o_aux;
    sq::DBuf<uint32_t> o_blk_off;
    // wire-form upload (sqg_load_concordant_wire): staging of the delta-coded arrays, the copy stream and one event per chunk
    sq::DBuf<uint16_t> w_dpos, w_span, w_bdref, w_bmref, w_brpos, w_bmread;
    sq::DBuf<int16_t> w_dmate;
    sq::DBuf<uint8_t> w_lp, w_an;
    sq::DBuf<int32_t> w_tile_ref, w_tile_pos;
    sq::DBuf<uint32_t> w_tile_blk, w_tile_rexc, w_tile_bexc, w_tile_wblk;
    sq::DBuf<sqg_wire_rec_exc> w_rec_exc;
    sq::DBuf<sqg_wire_blk_exc> w_blk_exc;
    cudaStream_t stream_up = nullptr;
    std::vector<cudaEvent_t> ev_up;
    bool wire_loaded = false;
    // classification launched chunk by chunk behind the widening kernels of a wire upload (run_classify then only finishes it)
    bool classify_prelaunched = false;
    int64_t pre_cand_cap = 0;

    // device BAM decode (sqg_load_concordant_bam): compressed window, two inflated windows (the tail of one is the head of the
    // next), segment walks, record offsets, per-record block counts, the ChimName hash set, pinned staging of the file
    sq::DBuf<uint8_t> bam_comp, bam_win[2], bam_nblob;
    sq::DBuf<sq::BamMember> bam_mem;
    sq::DBuf<int64_t> bam_seg, bam_start, bam_exit, bam_newstart, bam_recoff, bam_small, bam_noff;
    sq::DBuf<uint32_t> bam_cnt, bam_base, bam_nblk;
    sq::DBuf<uint64_t> bam_incl, bam_nhash;
    sq::DBuf<int32_t> bam_nlen;
    sq::DBuf<uint8_t> bam_bad, bam_redo;
    sq::DBuf<uint16_t> bam_lseq;           // read length from the CIGAR, kept only for the synthesised-quality rule (see sqg_api.cu)
    sq::HBuf<uint8_t> bam_stage[2];
    sq::HBuf<int64_t> bam_hsmall;
    std::vector<cudaEvent_t> bam_ev;       // [0..1]: staging buffer free again
    std::map<std::string, float> acc_ms;   // phases summed over the windows of the last BAM load
    int64_t bam_members = -1, bam_windows = -1, bam_repair_rounds = -1;
    int64_t bam_win_len = 0;               // bytes of the previous window (its unconsumed tail is copied to the front of the next)

    // classify products
    sq::DBuf<uint8_t> d_cls;
    sq::DBuf<uint16_t> d_flen;      // first-block length of every CLS_CONC record (seed machine windows)
    sq::DBuf<uint64_t> d_other;     // running otherChr/otherrightmost key at each coverage-gap record
    sq::DBuf<uint64_t> d_chain64;   // look-back words of the classification tiles (P1Out::gate_word)
    sq::DBuf<sq::TileAgg> d_tileagg;  // per-tile aggregates / exclusive prefixes of phase 1
    sq::DBuf<uint32_t> d_cov_nq; sq::DBuf<uint64_t> d_cov_qmax, d_cov_incmax; sq::DBuf<int64_t> d_cov_rank0; sq::DBuf<uint8_t> d_temp_cov;  // phase 3: per classification tile
    sq::DBuf<uint64_t> d_qstage_key; sq::DBuf<int32_t> d_qstage_end;  // phase 3's pairs as the classification kernel leaves them (per tile)
    sq::DBuf<int32_t> d_ccmax;        // per tile: maximum end of its ConcordantCluster entries (consume_cc of the seed machine)
    sq::DBuf<unsigned char> d_desc;   // device copy of the batch descriptor
    sq::DBuf<uint64_t> d_cand_key;    // coverage-gap candidates (their record indices live in d_scratch32)
    sq::DBuf<int32_t> d_scratch32;  // lastpass / depth targets / res0
    sq::DBuf<int32_t> d_gap, d_pc, d_dp;
    int32_t n_gap = 0, n_pc = 0, n_dp = 0, lmax = 0, n_islands = 0;
    int64_t first_kept = 0;
    uint64_t end_other = 0;      // otherChr/otherrightmost after the last record of the batch
    sq::DBuf<unsigned char> d_temp;  // CUB temp storage
    sq::DBuf<int64_t> d_counters;    // small device counters
    sq::HBuf<int64_t> h_counters;

    // chimeric side
    bool have_chim = false, prepass_uploaded = false;
    std::vector<sq::Group> h_groups;  // the pre-pass's groups on the host, for a range shard only (seed_stage looks up g_lo)
    sqg_chimeric chim_view{};
    sq::Worker prepass_worker;  // persistent host thread of the chimeric pre-pass (keeps its OpenMP team alive between runs)
    int64_t c_n_reads = 0, c_n_blk = 0;
    sq::DBuf<sq::DiscBlock> d_disc;
    sq::DBuf<sq::Group> d_groups;
    sq::DBuf<int32_t> d_pchr, d_ppos;
    sq::DBuf<uint32_t> dc_read_off;
    sq::DBuf<uint16_t> dc_n_first;
    sq::DBuf<int32_t> dc_first_total, dc_second_total, dc_ref_id, dc_ref_pos, dc_read_pos, dc_match_ref, dc_match_read, dc_res0;
    sq::DBuf<uint8_t> dc_rev;
    // pristine copies of the four arrays LocateRead trims in place: every edge pass starts from them (a pass may run twice --
    // buffer overflow, a shard's hint redo -- and a trimmed block can locate differently from the original one)
    sq::DBuf<int32_t> dc0_ref_pos, dc0_read_pos, dc0_match_ref, dc0_match_read;

    // std::sort's permutation of the discordant blocks on the device (sq_gpusort.cuh), driven by the pre-pass thread
    cudaStream_t stream3 = nullptr;
    cudaEvent_t ev_chim = nullptr;       // the chimeric arrays are in HBM (uploaded by the pre-pass thread before its own work)
    bool chim_upload_pending = false;
    int chim_upload_err = 0;
    cudaEvent_t ev_pre = nullptr;        // the pre-pass products (discordant blocks, groups, PartAlignPos) are in HBM
    int pre_upload_err = 0;
    sq::DBuf<uint64_t> d_gs_keys;
    sq::DBuf<uint32_t> d_gs_idx;
    sq::DBuf<unsigned char> d_gs_scratch;
    int64_t gs_launches = 0;
    int gs_last_status = -100;   // status of the most recent device sort (-100: not run)

    // node building
    sq::DBuf<int64_t> d_trigger;
    sq::DBuf<sq::RestBlock> d_rest, d_rest2;
    sq::DBuf<uint32_t> d_restkey, d_restkey2;
    sq::DBuf<int32_t> d_chimdiff; sq::HBuf<int32_t> h_chimdiff;  // rows (block, RefPos, ReadPos, MatchRef, MatchRead) of the trimmed chimeric blocks
    struct ChimPatch { int32_t k; int32_t v[4]; };
    std::vector<ChimPatch> chim_undo;  // loaded values of the blocks the last sqg_build_edges patched in the caller's arrays
    sq::DBuf<uint32_t> d_restbits; sq::DBuf<int32_t> d_restoff, d_reflen;  // bitmap of the 1024-bp bins near discordant groups (k_rest_collect)
    sq::DBuf<uint32_t> d_omask; sq::DBuf<int4> d_shorts;  // ReadsOther blocks of <= 3 bp: per-segment start masks, deferred blocks
    sq::DBuf<int32_t> d_other_off, d_other_len, d_other_own; sq::DBuf<uint64_t> d_other_key; sq::DBuf<uint32_t> d_other_idx;  // the replayed sort(ReadsOther)
    int64_t n_short_other = 0, n_unstable_other = 0; int other_sort_status = -1;
    // the chimeric pre-pass on the device (sq_prepass.cuh)
    sq::DBuf<int32_t> d_pre_ndis, d_pre_pusher, d_pre_lastk, d_pre_open; sq::DBuf<int64_t> d_pre_off; sq::DBuf<uint64_t> d_pre_part, d_pre_part2, d_pre_endkey, d_pre_excl, d_pre_incl;
    sq::DBuf<uint8_t> d_pre_opens, dc_first_low, dc_second_low, dc_multi, d_temp3; sq::DBuf<int64_t> d_pre_cnt; sq::HBuf<int64_t> h_pre_cnt;
    sq::PhaseTimer *prepass_timer = nullptr;
    int32_t pre_nD = 0, pre_nG = 0, pre_nP = 0;   // sizes of the pre-pass products
    sq::DBuf<sq::SeedOp> d_ops;
    sq::DBuf<sq::SeedOp> d_ops_dense;  // the islands' op lists without their unused capacity, island order
    sq::HBuf<sq::SeedOp> h_ops;
    sq::DBuf<uint8_t> d_cutflag;
    sq::DBuf<int32_t> d_isl, d_cap_ops, d_cap_mar, d_isl_nout, d_isl_gdone, d_span, d_heavy, d_light;
    int32_t n_heavy = 0;
    bool cov_chain_fallback = false;
    int64_t n_sensitive = 0, n_raw_edges = 0;
    int32_t classify_attempts = 0;   // passes the last run_classify needed (2: the coverage-gap candidate buffer overflowed)
    int32_t edge_pass_attempts = 0;  // passes the last run_assign needed (1 unless a list overflowed; at most 4)
    sq::DBuf<int64_t> d_off_ops, d_off_mar;
    sq::DBuf<int32_t> d_margin;
    int64_t r_break = 0;

    // the shard planner on the resident batch (sqg_plan_shards_resident): scan inputs / outputs, candidates; released after each plan
    sq::DBuf<uint64_t> d_plan_reach;
    sq::DBuf<int32_t> d_plan_keep, d_plan_upd;
    sq::DBuf<uint64_t> d_plan_cand, d_plan_sel;
    sq::HBuf<uint64_t> h_plan_sel;

    // range shard of one genome (sqg_set_shard, SURVEY.md 8e): index 0 owns the chimeric edges and the discordant depth
    int32_t shard_index = 0, shard_count = 1;
    bool shard_prior_emission = false;   // some earlier shard has emitted a seed segment (k_seed_prefix is skipped)
    int32_t shard_g_lo = 0;              // first discordant group this shard owns
    int32_t shard_init_hint = 0;         // firstfrontindex at the shard's first read
    int32_t shard_lead_sensitive = 0, shard_out_hint = -1;
    bool shard_seeded = false;
    std::vector<sq::SeedOp> shard_ops;   // this shard's seed ops, island order
    int32_t shard_g_done = 0;
    int64_t shard_trig_last = 0;
    int64_t cov_K = 0, cov_nq = 0;       // staged coverage (sqg_shard_cov_*)
    int64_t cov_n_pass = 0;              // range shard: breakpoints [cov_n_pass, cov_K) are passed by no record of this shard
    sq::HBuf<int64_t> h_t;

    // segment table
    bool have_nodes = false;
    std::vector<int32_t> h_nchr, h_npos, h_nend, h_chr_first;
    sq::DBuf<int32_t> d_nchr, d_npos, d_nend, d_chr_first, d_bin_off, d_bin_seg;
    std::vector<int32_t> h_bin_off;
    sq::NodeTable nt;
    sq::DBuf<int32_t> d_cnt3, d_sum3;

    // edges
    sq::DBuf<uint64_t> d_ekeys, d_ekeys2, d_ukeys;
    sq::DBuf<int32_t> d_ecount, d_sens, d_head, d_ew, d_slow;
    sq::DBuf<sq::DepthTile> d_dtile;
    sq::DBuf<int32_t> d_e_ind1, d_e_ind2, d_e_w;
    sq::DBuf<uint8_t> d_e_heads;
    int64_t n_unique_edges = 0;
    bool have_edge_table = false;

    // coverage
    sq::DBuf<uint64_t> d_bpkey, d_covM, d_qkey;
    sq::DBuf<int32_t> d_chunks;
    int32_t cov_chain_chunks = 0;
    sq::DBuf<int64_t> d_r0, d_t, d_chain_used;
    sq::DBuf<int32_t> d_cov, d_bpchr, d_bppos, d_qend;
    sq::DBuf<sq::CovTile> d_covtile;

    // pinned outputs
    sq::HBuf<int32_t> h_chr, h_pos, h_len, h_cnt3, h_sum3, h_ind1, h_ind2, h_w;
    sq::HBuf<uint8_t> h_heads;
};
#endif
