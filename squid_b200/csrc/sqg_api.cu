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
#include <cub/cub.cuh>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "sq_classify.cuh"
#include "sq_depth_cover.cuh"
#include "sq_locate.cuh"
#include "sq_phase1.cuh"
#include "sq_phase2.cuh"
#include "sq_phase3.cuh"
#include "sq_plan.cuh"
#include "sq_seed.cuh"
#include "sq_gpusort.cuh"
#include "sq_prepass.cuh"
#include "sq_wire.cuh"
#include "sq_cc.cuh"
#include "sq_inflate.cuh"
#include "sq_bam.cuh"
#include "sqg_ctx.cuh"
#include "host/bam.h"
#include "host/prepass.h"

using namespace sq;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return SQG_ECUDA;                                                                      \
        }                                                                                          \
    } while (0)
#define FAIL(code, msg) do { ctx->err = (msg); return (code); } while (0)
#define LAUNCH_ON(st, kernel, grid, block, ...)                                                    \
    do {                                                                                           \
        kernel<<<(grid), (block), 0, (st)>>>(__VA_ARGS__);                                         \
        ctx->launches++;                                                                           \
        CK(cudaGetLastError());                                                                    \
    } while (0)
#define LAUNCH(kernel, grid, block, ...) LAUNCH_ON(ctx->stream, kernel, grid, block, __VA_ARGS__)

struct HostLap {  // SQG_TIMING=1: wall-clock laps of the host side of a call, to stderr
    bool on; std::chrono::steady_clock::time_point t0;
    HostLap() : on(getenv("SQG_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void operator()(const char *what) {
        if (!on) return;
        const auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[sqg] %-28s %8.3f ms\n", what, 1e3 * std::chrono::duration<double>(t - t0).count());
        t0 = t;
    }
};
static constexpr int kThreads = 256;
static inline unsigned blocks_for(int64_t n, int threads = kThreads) { return (unsigned)std::max<int64_t>(1, (n + threads - 1) / threads); }

static int phase_begin(sqg_ctx *ctx, const char *name, cudaStream_t st = nullptr) {
    PhaseTimer &t = ctx->timers[name];
    if (!t.a) { CK(cudaEventCreate(&t.a)); CK(cudaEventCreate(&t.b)); }
    t.done = false;
    CK(cudaEventRecord(t.a, st ? st : ctx->stream));
    return SQG_OK;
}
static int phase_end(sqg_ctx *ctx, const char *name, cudaStream_t st = nullptr) {
    PhaseTimer &t = ctx->timers[name];
    CK(cudaEventRecord(t.b, st ? st : ctx->stream));
    t.done = true;
    return SQG_OK;
}
// everything that rewrites what the coverage compaction reads (batch, class bytes, chain scratch) first waits for it
static int cov_join(sqg_ctx *ctx) {
    if (ctx->cov_pending) { CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_cov_done, 0)); ctx->cov_pending = false; }
    return SQG_OK;
}
#define PHASE_BEGIN(name) do { int rc_ = phase_begin(ctx, name); if (rc_) return rc_; } while (0)
#define PHASE_END(name) do { int rc_ = phase_end(ctx, name); if (rc_) return rc_; } while (0)

// ------------------------------------------------------------------------------------------------
// functors / kernels: classify
// ------------------------------------------------------------------------------------------------
struct MaxI32 { __device__ int32_t operator()(int32_t a, int32_t b) const { return a > b ? a : b; } };
struct MaxU64 { __device__ uint64_t operator()(uint64_t a, uint64_t b) const { return a > b ? a : b; } };
struct MaxI64 { __device__ int64_t operator()(int64_t a, int64_t b) const { return a > b ? a : b; } };

// ------------------------------------------------------------------------------------------------
// kernels: node building
// ------------------------------------------------------------------------------------------------
__global__ void k_triggers(DevBatch b, const uint8_t *cls, const Group *G, int32_t nG, int64_t *trig) {
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nG) return;
    const Group grp = G[g];
    int64_t lo = 0, hi = b.n_rec;
    while (lo < hi) {  // first record past (chr, right) of the group (:353)
        const int64_t m = (lo + hi) >> 1;
        const int32_t rid = b.ref_id[m];
        const bool past = rid < 0 || grp.chr < rid || (grp.chr == rid && grp.right < b.pos[m]);
        if (!past) lo = m + 1; else hi = m;
    }
    while (lo < b.n_rec && !(cls[lo] & CLS_KEEP)) lo++;
    trig[g] = lo;
}

// ConcordRest candidates: non-first blocks of concordant records that start inside
// [group start - ReadLen, group right + ReadLen) of some discordant group (:690-699, :387, :471-473).
// The groups cover a tiny part of the genome, so a bitmap over 1024-bp bins (bit set = some group's extended range touches the
// bin) rejects almost every block with one cached load; only the survivors search the group list.
constexpr int kRestBinShift = 10;
struct RestBins { const uint32_t *bits; const int32_t *off; };   // off[c] = first bin of chromosome c (n_ref + 1 entries)
__global__ void k_rest_mark(const Group *G, const DiscBlock *D, int32_t nG, int32_t read_len, const int32_t *ref_len, uint32_t *bits, const int32_t *off) {
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nG) return;
    const Group grp = G[g];
    int32_t a = D[grp.ds].pos - read_len, b = grp.right + read_len - 1;  // positions [a, b]
    if (a < 0) a = 0;
    const int32_t last = ref_len[grp.chr] > 0 ? ref_len[grp.chr] : 0;
    if (b > last) b = last;
    for (int32_t k = a >> kRestBinShift; k <= (b >> kRestBinShift); k++) { const int32_t bin = off[grp.chr] + k; atomicOr(&bits[bin >> 5], 1u << (bin & 31)); }
}
// group of a candidate block at (c, q): the last group whose (start - ReadLen) lies at or left of it, if the block starts left of
// that group's right end + ReadLen; -1 otherwise
__device__ __forceinline__ int32_t rest_group_of(const Group *G, const DiscBlock *D, int32_t nG, int32_t read_len, int32_t c, int32_t q) {
    int32_t lo = 0, hi = nG;
    while (lo < hi) {
        const int32_t m = (lo + hi) >> 1;
        const Group g = G[m];
        const int32_t s = D[g.ds].pos - read_len;
        if (g.chr < c || (g.chr == c && s <= q)) lo = m + 1; else hi = m;
    }
    const int32_t gi = lo - 1;
    if (gi < 0) return -1;
    const Group g = G[gi];
    return (g.chr != c || q >= g.right + read_len) ? -1 : gi;
}
__global__ void k_rest_collect(DevBatch b, const uint8_t *cls, const Group *G, const DiscBlock *D, int32_t nG, int32_t read_len, RestBins rb, const int32_t *ref_len,
                               RestBlock *out, uint32_t *out_key, int64_t cap, int64_t *counter) {
    const int64_t r0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;  // four records per thread: one 32-bit load of their class bytes
    uint32_t w = 0;
    if (r0 + 3 < b.n_rec) w = *reinterpret_cast<const uint32_t *>(cls + r0);
    else for (int k = 0; k < 4; k++) if (r0 + k < b.n_rec) w |= (uint32_t)cls[r0 + k] << (8 * k);
    const bool any = (w & (0x01010101u * CLS_REST)) != 0;
    if (!__any_sync(0xffffffffu, any)) return;
    // pass 1: which (record, block) pairs qualify -- a bit each (4 records x up to 15 non-first blocks); pass 2 writes them to slots
    // reserved with ONE atomic per warp (the single list counter serialises otherwise: tens of millions of candidates)
    uint64_t hit = 0;
    if (any)
        for (int j = 0; j < 4; j++) {
            if (!((w >> (8 * j)) & CLS_REST)) continue;  // CLS_CONC, a mate flag, >= 2 blocks
            const int64_t r = r0 + j;
            const uint32_t o = b.blk_off[r], e = b.blk_off[r + 1];
            const int32_t c = b.ref_id[r];
            const int32_t last = ref_len[c] > 0 ? ref_len[c] : 0;
            for (uint32_t k = o + 1; k < e && k - o <= 15; k++) {
                const int32_t q = b.blk_ref_pos[k];
                if (q < 0 || q > last) continue;  // (cannot lie in any group's range, which is clipped to the chromosome)
                const int32_t bin = rb.off[c] + (q >> kRestBinShift);
                if (!((rb.bits[bin >> 5] >> (bin & 31)) & 1u)) continue;
                if (rest_group_of(G, D, nG, read_len, c, q) >= 0) hit |= 1ull << (16 * j + (k - o));
            }
        }
    const int cnt = __popcll(hit);
    int inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc, d); if ((int)(threadIdx.x & 31) >= d) inc += u; }
    const int tot = __shfl_sync(0xffffffffu, inc, 31);
    if (tot == 0) return;
    long long base = 0;
    if ((threadIdx.x & 31) == 31) base = (long long)atomicAdd((unsigned long long *)counter, (unsigned long long)tot);
    base = __shfl_sync(0xffffffffu, base, 31);
    int64_t slot = base + inc - cnt;
    while (hit) {
        const int bit = __ffsll((long long)hit) - 1;
        hit &= hit - 1;
        const int j = bit >> 4, kk = bit & 15;
        const int64_t r = r0 + j;
        const uint32_t k = b.blk_off[r] + kk;
        const int32_t c = b.ref_id[r], q = b.blk_ref_pos[k];
        if (slot < cap) {
            out[slot] = RestBlock{c, q, q + b.blk_match_ref[k], (int32_t)r};
            out_key[slot] = (uint32_t)rest_group_of(G, D, nG, read_len, c, q);
        }
        slot++;
    }
}

// island cut flags: flag[g] = 1 when the seed machine may be restarted at group g
__global__ void k_island_cuts(SeedInputs in, uint8_t *flag) {
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= in.nG) return;
    SeedMachine sm;
    sm.in = in;
    flag[g] = (g == in.g_lo) ? 1 : ((g < in.g_lo || g >= in.g_hi) ? 0 : (sm.island_cut(g) ? 1 : 0));  // groups before g_lo belong to earlier shards
}
struct IsCutOp {
    const uint8_t *flag;
    __device__ bool operator()(int32_t g) const { return flag[g] != 0; }
};
// scratch each island needs: [2i] = op slots, [2i+1] = margin slots
constexpr int32_t kHeavySpanDev = 1 << 14;  // islands spanning more records than this get a whole block instead of a warp (measured: 1 << 12 moves the
                                            // tail from the warps to the blocks and lengthens the kernel, 5.5 -> 6.6 ms)
__global__ void k_island_caps(SeedInputs in, const int32_t *isl_start, int32_t n_isl, int32_t *cap_ops, int32_t *cap_mar, int32_t *span) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_isl) return;
    SeedMachine sm;
    sm.in = in;
    const int32_t ga = isl_start[i], gb = (i + 1 < n_isl) ? isl_start[i + 1] : in.g_hi;
    const int32_t thresh = kSeedThresh, RL = in.read_len;
    int32_t mmax = 0;
    int64_t rmax = 0;  // widest position range the margins of one group can span (all lie in [group start - ReadLen, group right + thresh])
    for (int32_t g = ga; g < gb; g++) {
        const Group grp = in.G[g];
        const int32_t s0 = in.D[grp.ds].pos;
        { const int64_t r = (int64_t)grp.right - s0 + RL + thresh + 2; if (r <= in.dense_max_r && r > rmax) rmax = r; }
        int32_t m = 2 * (grp.de - grp.ds);
        {   // PartAlignPos entries of the group (:392-393)
            int32_t lo = 0, hi = in.nP;
            while (lo < hi) { int32_t q = (lo + hi) >> 1; if (in.Pchr[q] < grp.chr || (in.Pchr[q] == grp.chr && in.Ppos[q] < s0 - RL)) lo = q + 1; else hi = q; }
            int32_t lo2 = lo, hi2 = in.nP;
            while (lo2 < hi2) { int32_t q = (lo2 + hi2) >> 1; if (in.Pchr[q] < grp.chr || (in.Pchr[q] == grp.chr && in.Ppos[q] < grp.right + RL)) lo2 = q + 1; else hi2 = q; }
            m += lo2 - lo;
        }
        {   // PartialAlignCluster entries whose block start can land in the margin range (:420-434)
            const int32_t lo = sm.lb_pc_pos(0, in.n_pc, grp.chr, s0 - thresh - in.lmax), hi = sm.lb_pc_pos(lo, in.n_pc, grp.chr, grp.right + thresh);
            m += hi - lo;
        }
        if (m > mmax) mmax = m;
    }
    const int64_t r0 = ga > 0 ? in.trigger[ga - 1] : in.first_kept;
    const int64_t r1 = in.trigger[gb - 1] < in.n_rec ? in.trigger[gb - 1] : in.n_rec;
    const int32_t ndp = sm.lb_list(in.dp_rec, in.n_dp, r1) - sm.lb_list(in.dp_rec, in.n_dp, r0);
    mmax += (ndp > 0 ? ndp : 0) + 16;
    cap_ops[i] = 4 * (in.G[gb - 1].de - in.G[ga].ds) + 2 * mmax + 64;
    int32_t pw = 1;
    while (pw < mmax + 2) pw <<= 1;  // sort_margins pads to a power of two; + the five per-break tables
    int64_t w0 = r0;  // the windows were emptied at the last 0-coverage record before the island's first group
    if (ga > 0) {
        int32_t cc, cr;
        const Group gp = in.G[ga - 1], gn = in.G[ga];
        const int32_t z = sm.last_is0(in.trigger[ga - 1], in.trigger[ga] < in.n_rec ? in.trigger[ga] : in.n_rec, gp.chr, gp.right, gn.chr, in.D[gn.ds].pos, &cc, &cr);
        if (z >= 0) w0 = in.gap_rec[z];
    }
    span[i] = (int32_t)((r1 - w0) > 0x7fffffff ? 0x7fffffff : (r1 - w0));  // records the island may have to walk
    // scratch: six regions of mcap ints (margin list + the five per-break tables) + 8 cells; islands that use position-indexed
    // tables need 5 (R + 2) + 2 min(nM, R) ints behind the list
    int64_t mc = pw;
    if (in.dense_max_r > 0) {
        const int64_t r = rmax < 16 * (int64_t)mmax + 4096 ? rmax : 16 * (int64_t)mmax + 4096;
        const int64_t need = (5 * (r + 2) + 2 * (r < mmax + 2 ? r : (int64_t)mmax + 2) + 2 + 4) / 5 + 1;
        if (need > mc) mc = need;
    }
    cap_mar[i] = (int32_t)(6 * mc + 8);
}
__global__ void k_gather_i32(const int32_t *src, const int32_t *idx, int32_t n, int32_t *out) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[idx[i]];
}
constexpr int kSeedBlock = 512;        // threads per block of the seed kernels
constexpr int kHeavySpan = kHeavySpanDev;
// Position-indexed break tables (sq_seed.cuh: tabulate_dense) on every island, for sub-clusters whose margins span at most this
// many positions; wider ones keep the sorted margin lists.
constexpr int32_t kSeedDenseRange = 1 << 16;
constexpr int32_t kSeedMarginSmem = 11264;  // ints of shared memory per block: the sorted margins / the window accumulators of the position-indexed tables (44 KB)
struct IsHeavyOp {
    const int32_t *span; const int32_t *n_prefix; bool want_heavy;
    __device__ bool operator()(int32_t i) const { return i >= *n_prefix && ((span[i] > kHeavySpan) == want_heavy); }
};
template <class W>
__device__ __forceinline__ void seed_one_island(const SeedInputs &in, int32_t i, bool inherited, const int32_t *isl_start, int32_t n_isl, const int64_t *off_ops,
                                                const int64_t *off_mar, SeedOp *ops, int32_t *margin, int32_t *n_out, int32_t *g_done, int32_t *err, int32_t *n_out_ret, int32_t *fast, int32_t fast_cap) {
    SeedMachineT<W> sm;
    sm.in = in;
    const int32_t ga = isl_start[i], gb = (i + 1 < n_isl) ? isl_start[i + 1] : in.g_hi;
    sm.out = ops + off_ops[i]; sm.out_cap = (int32_t)(off_ops[i + 1] - off_ops[i]);
    sm.margin = margin + off_mar[i]; sm.margin_cap = (int32_t)(off_mar[i + 1] - off_mar[i]);
    sm.msearch = fast; sm.msearch_cap = fast_cap;
    sm.use_dense = in.dense_max_r > 0;
    const int32_t gd = sm.run_island(ga, gb, inherited);
    if (W::lane() == 0) { g_done[i] = gd; n_out[i] = sm.st.n_out; if (sm.error) atomicMax(err, sm.error); }
    if (n_out_ret) *n_out_ret = sm.st.n_out;
}
// Sequential prefix (one block): islands from 0 until one has emitted a segment -- until then the machine truly has no
// last segment.  Writes *n_prefix = number of islands consumed.
__global__ void __launch_bounds__(kSeedBlock) k_seed_prefix(SeedInputs in, const int32_t *isl_start, int32_t n_isl, const int64_t *off_ops, const int64_t *off_mar,
                                                          SeedOp *ops, int32_t *margin, int32_t *n_out, int32_t *g_done, int32_t *err, int32_t *n_prefix) {
    int32_t i = 0;
    for (; i < n_isl; i++) {
        int32_t emitted = 0;
        seed_one_island<CoopBlock>(in, i, false, isl_start, n_isl, off_ops, off_mar, ops, margin, n_out, g_done, err, &emitted, nullptr, 0);
        if (emitted > 0) { i++; break; }
    }
    if (threadIdx.x == 0) *n_prefix = i;
}
// All other islands in parallel, each starting from an inherited (far-left) last segment: blocks [0, n_heavy) take one
// heavy island each (SeedMachineT<CoopBlock>), the remaining blocks take one light island per warp (SeedMachineT<CoopWarp>).
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, 1024 / BLOCK) k_seed_islands(SeedInputs in, const int32_t *isl_start, int32_t n_isl, const int64_t *off_ops, const int64_t *off_mar,
                                                           SeedOp *ops, int32_t *margin, int32_t *n_out, int32_t *g_done, int32_t *err,
                                                           const int32_t *heavy, int32_t n_heavy, const int32_t *light, int32_t n_light) {
    __shared__ int32_t s_margins[kSeedMarginSmem];  // sorted margins of the island being processed (whole block, or one slice per warp)
    if ((int32_t)blockIdx.x < n_heavy) {
        seed_one_island<CoopBlock>(in, heavy[blockIdx.x], true, isl_start, n_isl, off_ops, off_mar, ops, margin, n_out, g_done, err, nullptr, s_margins, kSeedMarginSmem);
        return;
    }
    const int32_t k = ((int32_t)blockIdx.x - n_heavy) * (BLOCK / 32) + (threadIdx.x >> 5);
    if (k >= n_light) return;
    constexpr int32_t per_warp = kSeedMarginSmem / (BLOCK / 32);
    seed_one_island<CoopWarp>(in, light[k], true, isl_start, n_isl, off_ops, off_mar, ops, margin, n_out, g_done, err, nullptr, s_margins + (threadIdx.x >> 5) * per_warp, per_warp);
}

// The op lists of the islands, concatenated in island order WITHOUT their unused capacity (the scratch of an island is sized for
// the worst case: two ops per margin).  One block: islands up to the first one that the stream ended in the middle of
// (g_done < start of the next island; nothing later is ever processed), an exclusive scan of their op counts, the copies.
// out_meta[0] = number of ops, out_meta[1] = first group that was not processed.
__global__ void __launch_bounds__(1024) k_ops_dense(const int32_t *isl_start, int32_t n_isl, int32_t g_hi, const int32_t *n_out, const int32_t *g_done, const int64_t *off_ops,
                                                    const SeedOp *ops, SeedOp *dense, int64_t *out_meta) {
    __shared__ int32_t s_first_bad, s_warp[32], s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_first_bad = n_isl; s_carry = 0; }
    __syncthreads();
    int32_t fb = n_isl;
    for (int32_t i = tid; i < n_isl; i += 1024) {
        const int32_t nxt = i + 1 < n_isl ? isl_start[i + 1] : g_hi;
        if (g_done[i] < nxt && i < fb) fb = i;
    }
    fb = __reduce_min_sync(0xffffffffu, fb);
    if (lane == 0 && fb < n_isl) atomicMin(&s_first_bad, fb);
    __syncthreads();
    const int32_t first_bad = s_first_bad;
    const int32_t n_use = first_bad < n_isl ? first_bad + 1 : n_isl;  // the island that stopped early still contributes its ops
    for (int32_t base = 0; base < n_use; base += 1024) {
        const int32_t i = base + tid;
        const int32_t c = i < n_use ? n_out[i] : 0;
        int32_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        int32_t wbase = 0;
        for (int w = 0; w < warp; w++) wbase += s_warp[w];
        const int32_t at = s_carry + wbase + inc - c;
        if (i < n_use) { const SeedOp *src = ops + off_ops[i]; for (int32_t k = 0; k < c; k++) dense[at + k] = src[k]; }
        __syncthreads();
        if (tid == 1023) s_carry = at + c;
        __syncthreads();
    }
    if (tid == 0) { out_meta[0] = s_carry; out_meta[1] = first_bad < n_isl ? g_done[first_bad] : g_hi; }
}

// ------------------------------------------------------------------------------------------------
// kernels: segment table index
// ------------------------------------------------------------------------------------------------
// bin_seg[bin_off[c] + k] = segment of chromosome c holding position k << bin_shift (the last segment of c when that
// position is the chromosome end itself)
__global__ void k_build_bins(NodeTable nt, int32_t *bin_seg, int32_t n_bins) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bins) return;
    int32_t lo = 0, hi = nt.n_ref;  // chromosome of bin i: last c with bin_off[c] <= i
    while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (nt.bin_off[m + 1] <= i) lo = m + 1; else hi = m; }
    bin_seg[i] = bin_seg_value(nt, lo, i - nt.bin_off[lo]);
}

// ------------------------------------------------------------------------------------------------
// kernels: depth
// ------------------------------------------------------------------------------------------------
__global__ void k_depth_disc(NodeTable nt, const DiscBlock *D, int32_t nD, int32_t *cnt, int32_t *sum) {
    const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nD) return;
    const DiscBlock d = D[k];
    if (d.chr < 0 || d.chr >= nt.n_ref) return;
    const int32_t c0 = nt.chr_first[d.chr], c1 = nt.chr_first[d.chr + 1];
    const int32_t j = seg_last_pos_le(nt, d.chr, c0, c1, d.pos);  // segment whose turn consumes this block (:774)
    if (j >= c0 && d.pos >= nt.pos[j] && d.pos + d.len <= nt.end[j]) { atomicAdd(&cnt[j], 1); atomicAdd(&sum[j], d.len); }
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
    if (n == "seed_window_records") return ctx->h_counters.p ? ctx->h_counters.p[29] : -1;  // concordant-cluster window sizes summed over the groups
    if (n == "n_rec") return ctx->have_batch ? ctx->batch.n_rec : -1;
    if (n == "n_blk") return ctx->have_batch ? ctx->batch.n_blk : -1;
    if (n == "slow_records") return ctx->h_counters.p ? (int64_t)*(int32_t *)(ctx->h_counters.p + 18) : -1;  // records handled by k_edges_generic
    if (n == "qualifying_records") return ctx->cov_nq;
    if (n == "short_other_blocks") return ctx->n_short_other;        // ReadsOther blocks of <= 3 bp in the last depth pass
    if (n == "unstable_depth_blocks") return ctx->n_unstable_other;  // ... whose segment depends on the tie order of sort(ReadsOther): resolved by replaying that sort
    if (n == "other_sort_status") return ctx->other_sort_status;
    if (n == "edges_single_path") return ctx->h_counters.p ? ctx->h_counters.p[16] : -1;
    if (n == "bam_members") return ctx->bam_members;                // BGZF members (with data) of the last sqg_load_concordant_bam
    if (n == "bam_windows") return ctx->bam_windows;
    if (n == "bam_repair_rounds") return ctx->bam_repair_rounds;    // rounds of segments walked again from their true entry, summed over the windows
    if (n == "edges_generic_path") return ctx->h_counters.p ? ctx->h_counters.p[17] : -1;
    return -1;
}

}  // extern "C"

// ctx->batch = the context's own arrays (o_*) holding n_rec records and n_blk blocks
static void point_batch_at_own_arrays(sqg_ctx *ctx, int64_t n_rec, int64_t n_blk) {
    DevBatch &b = ctx->batch;
    b.n_rec = n_rec; b.n_blk = n_blk;
    b.ref_id = ctx->o_ref_id.p; b.pos = ctx->o_pos.p; b.mate_ref_id = ctx->o_mate_ref_id.p; b.mate_pos = ctx->o_mate_pos.p; b.end_pos = ctx->o_end_pos.p;
    b.flag = ctx->o_flag.p; b.total_len = ctx->o_total_len.p; b.lowphred_run = ctx->o_lowphred_run.p; b.mapq = ctx->o_mapq.p; b.aux = ctx->o_aux.p;
    b.blk_off = ctx->o_blk_off.p; b.blk_ref_pos = ctx->o_blk_ref_pos.p; b.blk_match_ref = ctx->o_blk_match_ref.p;
    b.blk_read_pos = ctx->o_blk_read_pos.p; b.blk_match_read = ctx->o_blk_match_read.p;
}
// A new batch is resident: nothing computed on the previous one applies (the segment table, have_nodes, still does).  `wire`: its
// arrays come from the wire decode, whose consistency flag run_classify checks and whose classification may already be running
// (classify_prelaunched, set during that upload, stands); every other batch starts unclassified.
static void reset_batch_state(sqg_ctx *ctx, bool owned, int64_t first_record_index, bool wire) {
    ctx->have_batch = true; ctx->batch_owned = owned; ctx->batch_restricted = false; ctx->first_record_index = first_record_index;
    ctx->classified = false; ctx->cov_compacted = false; ctx->have_edge_table = false; ctx->wire_loaded = wire;
    if (!wire) ctx->classify_prelaunched = false;
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
#define UP(buf, src, cnt)                                                                                       \
    do {                                                                                                        \
        CK(ctx->buf.ensure((cnt) ? (cnt) : 1));                                                                 \
        if (cnt) CK(cudaMemcpyAsync(ctx->buf.p, hb->src, (cnt) * sizeof(*hb->src), cudaMemcpyHostToDevice, ctx->stream)); \
    } while (0)
    UP(o_ref_id, ref_id, n); UP(o_pos, pos, n); UP(o_mate_ref_id, mate_ref_id, n); UP(o_mate_pos, mate_pos, n); UP(o_end_pos, end_pos, n);
    UP(o_flag, flag, n); UP(o_total_len, total_len, n); UP(o_lowphred_run, lowphred_run, n); UP(o_mapq, mapq, n); UP(o_aux, aux, n);
    UP(o_blk_off, blk_off, n + 1);
    UP(o_blk_ref_pos, blk_ref_pos, nb); UP(o_blk_match_ref, blk_match_ref, nb); UP(o_blk_read_pos, blk_read_pos, nb); UP(o_blk_match_read, blk_match_read, nb);
#undef UP
    point_batch_at_own_arrays(ctx, hb->n_rec, hb->n_blk);
    PHASE_END("h2d");
    reset_batch_state(ctx, true, first_record_index, false);
    return SQG_OK;
}

static int classify_setup(sqg_ctx *ctx, int64_t cand_cap, P1Out &o);
static int classify_launch(sqg_ctx *ctx, const P1Out &o, int64_t tiles);
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
    CK(ctx->o_ref_id.ensure(n1)); CK(ctx->o_pos.ensure(n1)); CK(ctx->o_mate_ref_id.ensure(n1)); CK(ctx->o_mate_pos.ensure(n1)); CK(ctx->o_end_pos.ensure(n1));
    CK(ctx->o_flag.ensure(n1)); CK(ctx->o_total_len.ensure(n1)); CK(ctx->o_lowphred_run.ensure(n1)); CK(ctx->o_mapq.ensure(n1)); CK(ctx->o_aux.ensure(n1));
    CK(ctx->o_blk_off.ensure(n1 + 1));
    CK(ctx->o_blk_ref_pos.ensure(nb1)); CK(ctx->o_blk_match_ref.ensure(nb1)); CK(ctx->o_blk_read_pos.ensure(nb1)); CK(ctx->o_blk_match_read.ensure(nb1));
    CK(ctx->w_dpos.ensure(n1)); CK(ctx->w_span.ensure(n1)); CK(ctx->w_dmate.ensure(n1)); CK(ctx->w_lp.ensure(n1)); CK(ctx->w_an.ensure(n1));
    CK(ctx->w_bdref.ensure(nwb1)); CK(ctx->w_bmref.ensure(nwb1)); CK(ctx->w_brpos.ensure(nwb1)); CK(ctx->w_bmread.ensure(nwb1)); CK(ctx->w_tile_wblk.ensure(nt1));
    CK(ctx->w_tile_ref.ensure(nt1)); CK(ctx->w_tile_pos.ensure(nt1)); CK(ctx->w_tile_blk.ensure(nt1)); CK(ctx->w_tile_rexc.ensure(nt1)); CK(ctx->w_tile_bexc.ensure(nt1));
    CK(ctx->w_rec_exc.ensure(w->n_rec_exc ? (size_t)w->n_rec_exc : 1)); CK(ctx->w_blk_exc.ensure(w->n_blk_exc ? (size_t)w->n_blk_exc : 1));
    CK(ctx->d_counters.ensure(32)); CK(ctx->h_counters.ensure(32));
    cudaStream_t up = ctx->stream_up;
    // the copy stream starts after everything the main stream still has queued on the previous batch
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream)); CK(cudaStreamWaitEvent(up, ctx->ev_fork, 0));
    CK(cudaMemsetAsync(ctx->d_counters.p + 28, 0, sizeof(int64_t), ctx->stream));
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
    wo.bad = (int32_t *)(ctx->d_counters.p + 28);
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

// (test / diagnostic) the resident batch back into host arrays
extern "C" int sqg_download_concordant(sqg_ctx *ctx, sqg_batch *out) {
    if (!ctx || !out) return SQG_EINVAL;
    if (!ctx->have_batch) FAIL(SQG_ESTATE, "no concordant batch loaded");
    const DevBatch &b = ctx->batch;
    if (out->n_rec != b.n_rec || out->n_blk != b.n_blk) FAIL(SQG_EINVAL, "sqg_download_concordant: n_rec / n_blk do not match the resident batch");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)b.n_rec, nb = (size_t)b.n_blk;
#define DN(field, cnt) do { if ((cnt) > 0) CK(cudaMemcpyAsync((void *)out->field, b.field, (cnt) * sizeof(*b.field), cudaMemcpyDeviceToHost, ctx->stream)); } while (0)
    DN(ref_id, n); DN(pos, n); DN(mate_ref_id, n); DN(mate_pos, n); DN(end_pos, n); DN(flag, n); DN(total_len, n); DN(lowphred_run, n); DN(mapq, n); DN(aux, n);
    DN(blk_off, n + 1); DN(blk_ref_pos, nb); DN(blk_match_ref, nb); DN(blk_read_pos, nb); DN(blk_match_read, nb);
#undef DN
    if (ctx->wire_loaded) CK(cudaMemcpyAsync(ctx->h_counters.p + 28, ctx->d_counters.p + 28, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->wire_loaded && *(int32_t *)(ctx->h_counters.p + 28)) FAIL(SQG_EINVAL, "wire batch is inconsistent (escape without an exception entry, or block counts that contradict the tile table)");
    return SQG_OK;
}

extern "C" int sqg_attach_concordant_device(sqg_ctx *ctx, const sqg_batch *db, int64_t first_record_index) {
    if (!ctx || !db || db->n_rec < 0 || db->n_blk < 0) return SQG_EINVAL;
    if (db->n_rec >= 0x7fffff00ll) FAIL(SQG_EUNSUPPORTED, "more than 2^31 records per context: shard the stream");
    CK(cudaSetDevice(ctx->device));
    if (ctx->cov_pending) { CK(cudaStreamSynchronize(ctx->stream_cov)); ctx->cov_pending = false; }  // the previous batch's arrays belong to the caller again
    DevBatch &b = ctx->batch;
    b.n_rec = db->n_rec; b.n_blk = db->n_blk;
    b.ref_id = db->ref_id; b.pos = db->pos; b.mate_ref_id = db->mate_ref_id; b.mate_pos = db->mate_pos; b.end_pos = db->end_pos;
    b.flag = db->flag; b.total_len = db->total_len; b.lowphred_run = db->lowphred_run; b.mapq = db->mapq; b.aux = db->aux;
    b.blk_off = db->blk_off; b.blk_ref_pos = db->blk_ref_pos; b.blk_match_ref = db->blk_match_ref; b.blk_read_pos = db->blk_read_pos; b.blk_match_read = db->blk_match_read;
    reset_batch_state(ctx, false, first_record_index, false);
    return SQG_OK;
}

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
    PCK(ctx->d_pre_part.ensure(4 * nr + n_ref + 1)); PCK(ctx->d_pre_part2.ensure(4 * nr + n_ref + 1)); PCK(ctx->d_pre_cnt.ensure(8)); PCK(ctx->h_pre_cnt.ensure(8));
    auto temp = [&](size_t bytes) { return ctx->d_temp3.ensure(bytes + 256); };
    int64_t launches = 0;
    PCK(cudaMemsetAsync(ctx->d_pre_ndis.p + nr, 0, 4, st));
    k_pre_count<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_ndis.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p);
    size_t tb = 0, tb2 = 0;
    PCK(cub::DeviceScan::ExclusiveSum(nullptr, tb, ctx->d_pre_ndis.p, ctx->d_pre_off.p, (int)(nr + 1), st));
    PCK(cub::DeviceScan::ExclusiveScan(nullptr, tb2, ctx->d_pre_pusher.p, ctx->d_pre_pusher.p, MaxI32(), (int32_t)-1, (int)nr, st));
    PCK(temp(std::max(tb, tb2)));
    PCK(cub::DeviceScan::ExclusiveSum(ctx->d_temp3.p, tb, ctx->d_pre_ndis.p, ctx->d_pre_off.p, (int)(nr + 1), st));
    PCK(cub::DeviceScan::ExclusiveScan(ctx->d_temp3.p, tb2, ctx->d_pre_pusher.p, ctx->d_pre_pusher.p, MaxI32(), (int32_t)-1, (int)nr, st));
    PCK(cudaMemcpyAsync(ctx->h_pre_cnt.p, ctx->d_pre_off.p + nr, 8, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
    const int64_t nD = ctx->h_pre_cnt.p[0];
    if (nD >= 0x7fffff00ll) return (int)cudaErrorInvalidValue;
    PCK(ctx->d_gs_keys.ensure((size_t)nD + 1)); PCK(ctx->d_gs_idx.ensure((size_t)nD + 1)); PCK(ctx->d_gs_scratch.ensure(gsort::bytes_needed((size_t)nD)));
    PCK(ctx->d_disc.ensure((size_t)nD + 1)); PCK(ctx->d_pre_endkey.ensure((size_t)nD + 1)); PCK(ctx->d_pre_excl.ensure((size_t)nD + 1)); PCK(ctx->d_pre_incl.ensure((size_t)nD + 1));
    PCK(ctx->d_pre_opens.ensure((size_t)nD + 1)); PCK(ctx->d_pre_open.ensure((size_t)nD + 1));
    // PartAlignPos is resize()d to n_ref entries (0, 0) and then appended to (:203-204)
    PCK(cudaMemsetAsync(ctx->d_pre_part.p, 0, (size_t)n_ref * 8, st));
    const unsigned long long np0 = (unsigned long long)n_ref;
    PCK(cudaMemcpyAsync(ctx->d_pre_cnt.p, &np0, 8, cudaMemcpyHostToDevice, st));
    k_pre_write<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_off.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p, ctx->d_gs_keys.p, ctx->d_gs_idx.p, ctx->d_pre_part.p,
                                                                 (unsigned long long *)ctx->d_pre_cnt.p);
    PCK(cudaMemcpyAsync(ctx->h_pre_cnt.p + 1, ctx->d_pre_cnt.p, 8, cudaMemcpyDeviceToHost, st));
    launches += 6;
    // std::sort's permutation of bamdiscordant (:264): tie order is observable (SURVEY.md App. A-11)
    int rc = gsort::sort_like_std_device(ctx->d_gs_keys.p, ctx->d_gs_idx.p, (size_t)nD, ctx->d_gs_scratch.p, st, &launches);
    ctx->gs_last_status = rc;
    if (rc < 0) return -rc;
    if (rc != 0) {  // std::sort would have left the quicksort path (never seen on alignment data): the CPU twin, from a fresh copy of the keys
        const unsigned long long np1 = (unsigned long long)n_ref;
        PCK(cudaMemcpyAsync(ctx->d_pre_cnt.p, &np1, 8, cudaMemcpyHostToDevice, st));
        k_pre_write<<<blocks_for((int64_t)nr), kThreads, 0, st>>>(c, ctx->d_pre_off.p, ctx->d_pre_pusher.p, ctx->d_pre_lastk.p, ctx->d_gs_keys.p, ctx->d_gs_idx.p, ctx->d_pre_part.p,
                                                                     (unsigned long long *)ctx->d_pre_cnt.p);
        std::vector<uint64_t> hk((size_t)nD); std::vector<uint32_t> hi((size_t)nD);
        PCK(cudaMemcpyAsync(hk.data(), ctx->d_gs_keys.p, (size_t)nD * 8, cudaMemcpyDeviceToHost, st));
        PCK(cudaMemcpyAsync(hi.data(), ctx->d_gs_idx.p, (size_t)nD * 4, cudaMemcpyDeviceToHost, st));
        PCK(cudaStreamSynchronize(st));
        std::vector<sqh::SortKey> a((size_t)nD);
        for (int64_t i = 0; i < nD; i++) a[(size_t)i] = sqh::SortKey{hk[(size_t)i], hi[(size_t)i]};
        sqh::sort_keys_like_std(a.data(), a.data() + a.size(), 8);
        for (int64_t i = 0; i < nD; i++) hi[(size_t)i] = a[(size_t)i].k;
        PCK(cudaMemcpyAsync(ctx->d_gs_idx.p, hi.data(), (size_t)nD * 4, cudaMemcpyHostToDevice, st));
        PCK(cudaStreamSynchronize(st));
    }
    PCK(cudaStreamSynchronize(st));
    const int64_t nP = ctx->h_pre_cnt.p[1];
    PCK(ctx->d_pchr.ensure((size_t)nP + 1)); PCK(ctx->d_ppos.ensure((size_t)nP + 1));
    {   // sort(PartAlignPos) by (chr, pos) (:262): a total order on the values, any stable or unstable sort agrees
        int key_bits = 33;
        while (key_bits < 64 && (1ll << (key_bits - 32)) < (long long)n_ref) key_bits++;
        PCK(cub::DeviceRadixSort::SortKeys(nullptr, tb, ctx->d_pre_part.p, ctx->d_pre_part2.p, (int)nP, 0, key_bits, st));
        PCK(temp(tb));
        PCK(cub::DeviceRadixSort::SortKeys(ctx->d_temp3.p, tb, ctx->d_pre_part.p, ctx->d_pre_part2.p, (int)nP, 0, key_bits, st));
        k_pre_split_part<<<blocks_for(nP), kThreads, 0, st>>>(ctx->d_pre_part2.p, nP, ctx->d_pchr.p, ctx->d_ppos.p);
        launches += 4;
    }
    k_pre_gather<<<blocks_for(nD + 1), kThreads, 0, st>>>(c, ctx->d_gs_idx.p, nD, ctx->d_disc.p, ctx->d_pre_endkey.p);
    int32_t nG = 0;
    if (nD > 0) {
        PCK(cub::DeviceScan::ExclusiveScan(nullptr, tb, ctx->d_pre_endkey.p, ctx->d_pre_excl.p, MaxU64(), (uint64_t)0, (int)nD, st));
        PCK(cub::DeviceScan::InclusiveScan(nullptr, tb2, ctx->d_pre_endkey.p, ctx->d_pre_incl.p, MaxU64(), (int)nD, st));
        PCK(temp(std::max(tb, tb2)));
        PCK(cub::DeviceScan::ExclusiveScan(ctx->d_temp3.p, tb, ctx->d_pre_endkey.p, ctx->d_pre_excl.p, MaxU64(), (uint64_t)0, (int)nD, st));
        PCK(cub::DeviceScan::InclusiveScan(ctx->d_temp3.p, tb2, ctx->d_pre_endkey.p, ctx->d_pre_incl.p, MaxU64(), (int)nD, st));
        k_pre_opens<<<blocks_for(nD), kThreads, 0, st>>>(ctx->d_disc.p, ctx->d_pre_excl.p, nD, ctx->params.read_len, ctx->d_pre_opens.p);
        cub::CountingInputIterator<int32_t> cnt(0);
        PreOpenOp op{ctx->d_pre_opens.p};
        int32_t *d_ng = (int32_t *)(ctx->d_pre_cnt.p + 2);
        PCK(cub::DeviceSelect::If(nullptr, tb, cnt, ctx->d_pre_open.p, d_ng, (int)nD, op, st));
        PCK(temp(tb));
        PCK(cub::DeviceSelect::If(ctx->d_temp3.p, tb, cnt, ctx->d_pre_open.p, d_ng, (int)nD, op, st));
        PCK(cudaMemcpyAsync(ctx->h_pre_cnt.p + 2, ctx->d_pre_cnt.p + 2, 8, cudaMemcpyDeviceToHost, st));
        PCK(cudaStreamSynchronize(st));
        nG = *(int32_t *)(ctx->h_pre_cnt.p + 2);
        PCK(ctx->d_groups.ensure((size_t)nG + 1));
        k_pre_groups<<<blocks_for(nG), kThreads, 0, st>>>(ctx->d_disc.p, ctx->d_pre_open.p, d_ng, ctx->d_pre_excl.p, ctx->d_pre_incl.p, nD, ctx->d_groups.p);
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
static int finish_prepass(sqg_ctx *ctx) {
    ctx->prepass_worker.wait();
    if (ctx->prepass_uploaded) return SQG_OK;
    if (ctx->pre_upload_err) { ctx->err = std::string("upload of the pre-pass products: ") + cudaGetErrorString((cudaError_t)ctx->pre_upload_err); return SQG_ECUDA; }
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_pre, 0));
    ctx->prepass_uploaded = true;
    return SQG_OK;
}
static int ensure_temp(sqg_ctx *ctx, size_t bytes) { CK(ctx->d_temp.ensure(bytes + 256)); return SQG_OK; }
#define ENSURE_TEMP(bytes) do { int rc_ = ensure_temp(ctx, bytes); if (rc_) return rc_; } while (0)

static bool batch_bulk_ok(const DevBatch &b) {  // TMA bulk copies need 16-byte aligned sources
    const void *ptrs[] = {b.ref_id, b.pos, b.mate_ref_id, b.mate_pos, b.end_pos, b.flag, b.total_len, b.lowphred_run, b.mapq, b.aux, b.blk_off,
                          b.blk_ref_pos, b.blk_match_ref, b.blk_read_pos, b.blk_match_read};
    for (const void *q : ptrs) if (((uintptr_t)q) & 15u) return false;
    return true;
}
static constexpr size_t kTileSmemBytes = sizeof(TileStage) + 128;

// classify stage (phase 1): class bytes, gap / partial / displaced lists, first kept record, lmax; validates the batch
// Classification, part 1: buffers, counters and the kernel's argument block for a batch of n records (cand_cap candidates).
static int classify_setup(sqg_ctx *ctx, int64_t cand_cap, P1Out &o) {
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec, n_tiles = (n + kTile - 1) / kTile;
    CK(ctx->d_cls.ensure(n + 4)); CK(ctx->d_flen.ensure(n + 4)); CK(ctx->d_scratch32.ensure(n + 1));
    CK(ctx->d_counters.ensure(32)); CK(ctx->h_counters.ensure(32));
    CK(ctx->d_qstage_key.ensure((size_t)n + 1)); CK(ctx->d_qstage_end.ensure((size_t)n + 1));
    CK(ctx->d_tileagg.ensure(n_tiles + 1)); CK(ctx->d_chain64.ensure(n_tiles + 8)); CK(ctx->d_ccmax.ensure(n_tiles + 1)); CK(ctx->d_cov_nq.ensure(n_tiles + 2)); CK(ctx->d_cov_qmax.ensure(n_tiles + 2));
    CK(ctx->d_cand_key.ensure(cand_cap));
    o.cls = ctx->d_cls.p; o.first_len = ctx->d_flen.p; o.agg = ctx->d_tileagg.p; o.ccmax = ctx->d_ccmax.p; o.cov_nq = ctx->d_cov_nq.p; o.cov_qmax = ctx->d_cov_qmax.p; o.qstage_key = ctx->d_qstage_key.p; o.qstage_end = ctx->d_qstage_end.p; o.gate_word = ctx->d_chain64.p; o.n_tiles = (int32_t)n_tiles;
    o.cand_rec = ctx->d_scratch32.p; o.cand_key = ctx->d_cand_key.p; o.cand_cap = (int32_t)cand_cap;
    // counters: [0..1] totals n_gap, n_pc, n_dp (int32) | [2] first_kept | [3] lmax | [4] n_cand, ticket (int32) | [20] validation flags
    CK(cudaMemsetAsync(ctx->d_counters.p, 0, 5 * sizeof(int64_t), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_counters.p + 20, 0, sizeof(int64_t), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_chain64.p, 0, n_tiles * sizeof(uint64_t), ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_counters.p + 2, &n, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    o.first_kept = (long long *)(ctx->d_counters.p + 2); o.lmax = (int32_t *)(ctx->d_counters.p + 3);
    o.n_cand = (int32_t *)(ctx->d_counters.p + 4); o.ticket = o.n_cand + 1;
    o.bad_flags = (int32_t *)(ctx->d_counters.p + 20);
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
static int classify_launch(sqg_ctx *ctx, const P1Out &o, int64_t tiles) {
    if (tiles <= 0) return SQG_OK;
    const DevBatch &b = ctx->batch;
    k_classify_tiles<<<(unsigned)tiles, kTileThreads, kTileSmemBytes, ctx->stream>>>(b, ctx->params, o, batch_bulk_ok(b) ? 1 : 0);
    ctx->launches++;
    CK(cudaGetLastError());
    return SQG_OK;
}

static int run_classify(sqg_ctx *ctx) {
    if (ctx->classified) return SQG_OK;
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    PHASE_BEGIN("classify");
    CK(ctx->d_counters.ensure(32)); CK(ctx->h_counters.ensure(32));
    ctx->n_gap = 0; ctx->n_pc = 0; ctx->n_dp = 0; ctx->lmax = 0; ctx->first_kept = n; ctx->end_other = 0; ctx->classify_attempts = 0;
    if (n > 0) {
        const int64_t n_tiles = (n + kTile - 1) / kTile;
        int64_t cand_cap = std::max<int64_t>({(int64_t)ctx->d_cand_key.cap, n / 16, (int64_t)1 << 20});
        int32_t n_cand = 0;
        for (int attempt = 0; attempt < 2; attempt++) {
            cand_cap = std::min<int64_t>(cand_cap, n + 1);
            int32_t *totals = (int32_t *)ctx->d_counters.p;
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
            LAUNCH(k_tile_scan, 1, 1024, ctx->d_tileagg.p, (int32_t)n_tiles, totals, (uint64_t *)(ctx->d_counters.p + 21));
            CK(cudaMemcpyAsync(ctx->h_counters.p, ctx->d_counters.p, 5 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaMemcpyAsync(ctx->h_counters.p + 20, ctx->d_counters.p + 20, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            if (ctx->wire_loaded) CK(cudaMemcpyAsync(ctx->h_counters.p + 28, ctx->d_counters.p + 28, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            if (ctx->wire_loaded && *(int32_t *)(ctx->h_counters.p + 28)) FAIL(SQG_EINVAL, "wire batch is inconsistent (escape without an exception entry, or block counts that contradict the tile table)");
            const int32_t flags = *(int32_t *)(ctx->h_counters.p + 20);
            if (flags & 1) FAIL(SQG_EINVAL, "record with ref_id outside [-1, n_ref)");
            if (flags & 2) FAIL(SQG_EUNSUPPORTED, "mapped record with ref_id -1");
            if (flags & 4) FAIL(SQG_EUNSUPPORTED, "record with more than 16 aligned blocks or a decreasing blk_off");
            if (flags & 8) FAIL(SQG_EINVAL, "batch is not sorted by (ref_id, pos)");
            n_cand = *(int32_t *)(ctx->h_counters.p + 4);
            ctx->classify_attempts = attempt + 1;
            if (!(flags & 16)) break;
            if (attempt == 1) FAIL(SQG_ENOMEM, "coverage-gap candidate buffer overflow");
            cand_cap = n + 1;  // every record can be a candidate at worst
        }
        const int32_t *sel = (const int32_t *)ctx->h_counters.p;
        ctx->n_pc = sel[1]; ctx->n_dp = sel[2]; ctx->first_kept = ctx->h_counters.p[2];
        ctx->lmax = *(const int32_t *)(ctx->h_counters.p + 3);
        ctx->end_other = (uint64_t)ctx->h_counters.p[21];
        CK(ctx->d_gap.ensure((size_t)n_cand + 1)); CK(ctx->d_other.ensure((size_t)n_cand + 1));
        CK(ctx->d_pc.ensure((size_t)ctx->n_pc + 1)); CK(ctx->d_dp.ensure((size_t)ctx->n_dp + 1));
        if (n_cand > 0) {
            LAUNCH(k_finish_gaps, blocks_for(n_cand), kThreads, b, ctx->d_tileagg.p, ctx->d_scratch32.p, ctx->d_cand_key.p, n_cand, ctx->params.read_len, (int32_t *)ctx->d_counters.p);
            size_t tb = 0;
            CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_scratch32.p, ctx->d_gap.p, ctx->d_cand_key.p, ctx->d_other.p, n_cand, 0, 32, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceRadixSort::SortPairs(ctx->d_temp.p, tb, ctx->d_scratch32.p, ctx->d_gap.p, ctx->d_cand_key.p, ctx->d_other.p, n_cand, 0, 32, ctx->stream));
            ctx->launches += 3;
        }
        if (ctx->n_pc + ctx->n_dp > 0) LAUNCH(k_compact_lists, (unsigned)n_tiles, kTileThreads, ctx->d_cls.p, n, ctx->d_tileagg.p, ctx->d_pc.p, ctx->d_dp.p);
        CK(cudaMemcpyAsync(ctx->h_counters.p, ctx->d_counters.p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        PHASE_END("classify");
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->n_gap = sel[0];
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

static int install_nodes(sqg_ctx *ctx) {  // from h_nchr/h_npos/h_nend
    const int32_t N = (int32_t)ctx->h_nchr.size(), n_ref = ctx->params.n_ref;
    ctx->h_chr_first.assign(n_ref + 1, N);
    for (int32_t i = N - 1; i >= 0; i--) {
        const int32_t c = ctx->h_nchr[i];
        if (c < 0 || c >= n_ref) FAIL(SQG_EINVAL, "segment with chromosome outside [0, n_ref)");
        ctx->h_chr_first[c] = i;
    }
    for (int32_t c = n_ref - 1; c >= 0; c--) if (ctx->h_chr_first[c] == N) ctx->h_chr_first[c] = ctx->h_chr_first[c + 1];
    for (int32_t i = 0; i + 1 < N; i++) {
        const bool same = ctx->h_nchr[i] == ctx->h_nchr[i + 1];
        if (ctx->h_nchr[i] > ctx->h_nchr[i + 1] || (same && ctx->h_nend[i] != ctx->h_npos[i + 1])) FAIL(SQG_EINVAL, "segments must be sorted and tile each chromosome");
    }
    CK(ctx->d_nchr.ensure(N + 1)); CK(ctx->d_npos.ensure(N + 1)); CK(ctx->d_nend.ensure(N + 1)); CK(ctx->d_chr_first.ensure(n_ref + 2));
    if (N) {
        CK(cudaMemcpyAsync(ctx->d_nchr.p, ctx->h_nchr.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_npos.p, ctx->h_npos.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_nend.p, ctx->h_nend.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMemcpyAsync(ctx->d_chr_first.p, ctx->h_chr_first.data(), (n_ref + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->nt.n = N; ctx->nt.n_ref = n_ref; ctx->nt.chr = ctx->d_nchr.p; ctx->nt.pos = ctx->d_npos.p; ctx->nt.end = ctx->d_nend.p; ctx->nt.chr_first = ctx->d_chr_first.p;
    {   // coarse position index over the tiling (sq_common.cuh: seg_at)
        int64_t total = 0;
        for (int32_t c = 0; c < n_ref; c++) total += ctx->ref_len[c] > 0 ? ctx->ref_len[c] : 0;
        int32_t sh = 9;  // 512-bp bins: reads pile up exactly where segments are dense (fusion genes), so the bins must be fine
        while ((total >> sh) > (16ll << 20)) sh++;  // at most ~16M bins (64 MB, L2-resident where it is hot)
        ctx->h_bin_off.assign(n_ref + 1, 0);
        for (int32_t c = 0; c < n_ref; c++) ctx->h_bin_off[c + 1] = ctx->h_bin_off[c] + ((ctx->ref_len[c] > 0 ? ctx->ref_len[c] : 0) >> sh) + 1;
        const int32_t n_bins = ctx->h_bin_off[n_ref];
        CK(ctx->d_bin_off.ensure(n_ref + 2)); CK(ctx->d_bin_seg.ensure(n_bins + 1));
        CK(cudaMemcpyAsync(ctx->d_bin_off.p, ctx->h_bin_off.data(), (n_ref + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        ctx->nt.bin_off = ctx->d_bin_off.p; ctx->nt.bin_shift = sh; ctx->nt.bin_seg = nullptr;
        LAUNCH(k_build_bins, blocks_for(n_bins), kThreads, ctx->nt, ctx->d_bin_seg.p, n_bins);
        ctx->nt.bin_seg = ctx->d_bin_seg.p;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_nodes = true; ctx->have_edge_table = false;
    return SQG_OK;
}

extern "C" int sqg_set_nodes(sqg_ctx *ctx, const int32_t *chr, const int32_t *pos, const int32_t *len, int64_t n_nodes) {
    if (!ctx || !chr || !pos || !len || n_nodes <= 0 || n_nodes > 0x7ffffff0ll) return SQG_EINVAL;
    // the table must tile every chromosome from 0 to its length with segments of positive length: the position index (seg_at)
    // and the closed-form LocateRead index a chromosome's segments as [chr_first[c], chr_first[c+1]) and take a position below
    // the last segment's end to lie inside the chromosome's bins.  (Sortedness and contiguity are checked in install_nodes.)
    {
        const int32_t n_ref = ctx->params.n_ref;
        int32_t prev = -1;
        for (int64_t i = 0; i < n_nodes; i++) {
            const int32_t c = chr[i];
            if (c < 0 || c >= n_ref) FAIL(SQG_EINVAL, "set_nodes: segment " + std::to_string(i) + " has a chromosome outside [0, n_ref)");
            if (len[i] <= 0) FAIL(SQG_EINVAL, "set_nodes: segment " + std::to_string(i) + " has length <= 0");
            if (c != prev) {
                if (c < prev) FAIL(SQG_EINVAL, "set_nodes: segments must be sorted by chromosome");
                if (c > prev + 1) FAIL(SQG_EINVAL, "set_nodes: chromosome " + std::to_string(prev + 1) + " has no segment");
                if (pos[i] != 0) FAIL(SQG_EINVAL, "set_nodes: the first segment of chromosome " + std::to_string(c) + " does not start at 0");
                prev = c;
            }
            if (i + 1 == n_nodes || chr[i + 1] != c) {
                if ((int64_t)pos[i] + len[i] != (int64_t)ctx->ref_len[c])
                    FAIL(SQG_EINVAL, "set_nodes: the last segment of chromosome " + std::to_string(c) + " does not end at its length " + std::to_string(ctx->ref_len[c]));
            }
        }
        if (prev != n_ref - 1) FAIL(SQG_EINVAL, "set_nodes: chromosome " + std::to_string(prev + 1) + " has no segment");
    }
    CK(cudaSetDevice(ctx->device));
    ctx->h_nchr.assign(chr, chr + n_nodes); ctx->h_npos.assign(pos, pos + n_nodes); ctx->h_nend.resize(n_nodes);
    for (int64_t i = 0; i < n_nodes; i++) ctx->h_nend[i] = pos[i] + len[i];
    return install_nodes(ctx);
}

// seeds (device) -> normalised, genome-tiling segment table (SegmentGraph.cpp:19-38, 706-761)
static int tile_genome(sqg_ctx *ctx, std::vector<SeedNode> &seedv) {
    const int32_t n_seeds = (int32_t)seedv.size();
    SeedNode *s = seedv.data();
    std::sort(s, s + n_seeds, [](const SeedNode &a, const SeedNode &c) { return a.chr != c.chr ? a.chr < c.chr : (a.pos != c.pos ? a.pos < c.pos : a.len < c.len); });
    std::vector<SeedNode> norm;
    norm.reserve(n_seeds);
    for (int32_t i = 0; i < n_seeds; i++) {
        if (norm.empty() || norm.back().chr != s[i].chr || norm.back().pos + norm.back().len <= s[i].pos) norm.push_back(s[i]);
        else norm.back().len = std::max(norm.back().pos + norm.back().len, s[i].pos + s[i].len) - norm.back().pos;
    }
    ctx->h_nchr.clear(); ctx->h_npos.clear(); ctx->h_nend.clear();
    size_t k = 0;
    for (int32_t c = 0; c < ctx->params.n_ref; c++) {
        int32_t cur = 0;
        bool any = false;
        for (; k < norm.size() && norm[k].chr == c; k++) {
            int32_t st = norm[k].pos;
            const int32_t en = norm[k].pos + norm[k].len;
            if (norm[k].len <= 0 || en > ctx->ref_len[c]) FAIL(SQG_EUNSUPPORTED, "seed segment outside its chromosome (the reference asserts here, SegmentGraph.cpp:709)");
            if (st - cur > 100) { ctx->h_nchr.push_back(c); ctx->h_npos.push_back(cur); ctx->h_nend.push_back(st); }
            else st = cur;
            ctx->h_nchr.push_back(c); ctx->h_npos.push_back(st); ctx->h_nend.push_back(en);
            cur = en; any = true;
        }
        if (!any || cur != ctx->ref_len[c]) { ctx->h_nchr.push_back(c); ctx->h_npos.push_back(cur); ctx->h_nend.push_back(ctx->ref_len[c]); }
    }
    return install_nodes(ctx);
}

// Phase 3, first pass (sq_phase3.cuh: k_cov_compact): enqueued as soon as the class bytes exist -- it does not depend on the
// segment table, so sqg_build_nodes runs it while the host still waits for the chimeric pre-pass.  The count lands in
// h_counters[15] once the stream has been synchronised.
static int run_cov_compact(sqg_ctx *ctx) {
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
        size_t tb1 = 0, tb2 = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tb1, ctx->d_cov_nq.p, ctx->d_cov_rank0.p, (int)(n_ct + 1), st));
        CK(cub::DeviceScan::InclusiveScan(nullptr, tb2, ctx->d_cov_qmax.p, ctx->d_cov_incmax.p, MaxU64(), (int)n_ct, st));
        CK(ctx->d_temp_cov.ensure(std::max(tb1, tb2) + 256));
        CK(cudaMemsetAsync(ctx->d_cov_nq.p + n_ct, 0, 4, st));
        CK(cub::DeviceScan::ExclusiveSum(ctx->d_temp_cov.p, tb1, ctx->d_cov_nq.p, ctx->d_cov_rank0.p, (int)(n_ct + 1), st));
        CK(cub::DeviceScan::InclusiveScan(ctx->d_temp_cov.p, tb2, ctx->d_cov_qmax.p, ctx->d_cov_incmax.p, MaxU64(), (int)n_ct, st));
        ctx->launches += 4;
        int rc = phase_begin(ctx, "k_cov_compact", st);
        if (rc) return rc;
        k_cov_gather<<<(unsigned)n_tiles, kCovThreads, 0, st>>>(ctx->d_qstage_key.p, ctx->d_qstage_end.p, ctx->d_cov_nq.p, ctx->d_cov_rank0.p, ctx->d_cov_incmax.p, (int32_t)n_ct, (int32_t)n_tiles,
                                                                ctx->d_qkey.p, ctx->d_qend.p, ctx->d_covtile.p);
        ctx->launches++;
        CK(cudaGetLastError());
        rc = phase_end(ctx, "k_cov_compact", st);
        if (rc) return rc;
        CK(cudaMemcpyAsync(ctx->d_counters.p + 15, ctx->d_cov_rank0.p + n_ct, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(ctx->h_counters.p + 15, ctx->d_counters.p + 15, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(ctx->ev_cov_done, st));
        ctx->cov_pending = true;
    } else { CK(ctx->d_qkey.ensure(1)); CK(ctx->d_qend.ensure(1)); CK(ctx->d_covtile.ensure(1)); }
    ctx->cov_compacted = true;
    return SQG_OK;
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
    size_t tb = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, it, ctx->d_other_off.p, (int)(n + 1), ctx->stream));
    ENSURE_TEMP(tb);
    CK(cub::DeviceScan::ExclusiveSum(ctx->d_temp.p, tb, it, ctx->d_other_off.p, (int)(n + 1), ctx->stream));
    ctx->launches += 2;
    int32_t m32 = 0;
    CK(cudaMemcpyAsync(&m32, ctx->d_other_off.p + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int64_t M = m32;
    if (M <= 0) return SQG_OK;
    CK(ctx->d_other_key.ensure((size_t)M + 1)); CK(ctx->d_other_idx.ensure((size_t)M + 1)); CK(ctx->d_other_len.ensure((size_t)M + 1)); CK(ctx->d_other_own.ensure((size_t)M + 1));
    LAUNCH(k_other_fill, blocks_for(n), kThreads, b, ctx->d_cls.p, ctx->r_break, ctx->d_other_off.p, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p);
    CK(ctx->d_gs_scratch.ensure(gsort::bytes_needed((size_t)M)));
    int rc = gsort::sort_like_std_device(ctx->d_other_key.p, ctx->d_other_idx.p, (size_t)M, ctx->d_gs_scratch.p, ctx->stream, &ctx->launches);
    if (rc < 0) { ctx->err = std::string("ReadsOther sort: ") + cudaGetErrorString((cudaError_t)(-rc)); return SQG_ECUDA; }
    ctx->other_sort_status = rc;
    if (rc != 0) {  // std::sort would have left the quicksort path: the CPU twin, from a fresh copy of the keys
        LAUNCH(k_other_fill, blocks_for(n), kThreads, b, ctx->d_cls.p, ctx->r_break, ctx->d_other_off.p, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p);
        std::vector<uint64_t> hk((size_t)M);
        CK(cudaMemcpyAsync(hk.data(), ctx->d_other_key.p, (size_t)M * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        std::vector<sqh::SortKey> a((size_t)M);
        for (int64_t i = 0; i < M; i++) a[(size_t)i] = sqh::SortKey{hk[(size_t)i], (uint32_t)i};
        sqh::sort_keys_like_std(a.data(), a.data() + a.size(), 16);
        std::vector<uint32_t> hi((size_t)M);
        for (int64_t i = 0; i < M; i++) { hk[(size_t)i] = a[(size_t)i].key; hi[(size_t)i] = a[(size_t)i].k; }
        CK(cudaMemcpyAsync(ctx->d_other_key.p, hk.data(), (size_t)M * 8, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_other_idx.p, hi.data(), (size_t)M * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    LAUNCH(k_other_own, blocks_for(M), kThreads, ctx->nt, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p, M, ctx->d_other_own.p);
    CK(cub::DeviceScan::InclusiveScan(nullptr, tb, ctx->d_other_own.p, ctx->d_other_own.p, MaxI32(), (int)M, ctx->stream));
    ENSURE_TEMP(tb);
    CK(cub::DeviceScan::InclusiveScan(ctx->d_temp.p, tb, ctx->d_other_own.p, ctx->d_other_own.p, MaxI32(), (int)M, ctx->stream));
    ctx->launches += 2;
    LAUNCH(k_other_apply, blocks_for(M), kThreads, ctx->nt, ctx->d_other_key.p, ctx->d_other_idx.p, ctx->d_other_len.p, ctx->d_other_own.p, M, cnt_other, sum_other);
    return SQG_OK;
}

// Phase 2 (sq_phase2.cuh): one pass over the batch for the depth numerators (do_depth) and the raw edges of the chimeric
// reads + the concordant stream (do_edges); then the hint fix-up chains and the sort + reduce of the (key, count) pairs.
static int run_assign(sqg_ctx *ctx, bool do_depth, bool do_edges) {
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
        // counters: [9] raw pairs | [10] sensitive concordant reads, sensitive chimeric reads (int32 each)
        CK(cudaMemsetAsync(ctx->d_counters.p + 9, 0, 2 * sizeof(int64_t), ctx->stream));
        unsigned long long *d_cnt = (unsigned long long *)(ctx->d_counters.p + 9);
        int32_t *d_nsens = (int32_t *)(ctx->d_counters.p + 10);
        PairSink sink{ctx->d_ekeys.p, ctx->d_ew.p, cap, d_cnt};
        if (do_depth) {
            CK(cudaMemsetAsync(ctx->d_cnt3.p, 0, (3 * (size_t)N + 4) * 4, ctx->stream));
            CK(cudaMemsetAsync(ctx->d_sum3.p, 0, (3 * (size_t)N + 4) * 4, ctx->stream));
            if (nD > 0 && ctx->shard_index == 0) LAUNCH(k_depth_disc, blocks_for(nD), kThreads, ctx->nt, ctx->d_disc.p, nD, ctx->d_cnt3.p, ctx->d_sum3.p);
        }
        CK(cudaMemsetAsync(ctx->d_counters.p + 22, 0, 2 * sizeof(int64_t), ctx->stream));  // [22] used_init flag | [23] out hint
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
            a.path_counts = (unsigned long long *)(ctx->d_counters.p + 16);
            CK(cudaMemsetAsync(ctx->d_counters.p + 16, 0, 3 * sizeof(int64_t), ctx->stream));
            CK(ctx->d_slow.ensure(slow_cap));
            a.slow_list = ctx->d_slow.p; a.n_slow = (int32_t *)(ctx->d_counters.p + 18); a.slow_cap = (int32_t)std::min<int64_t>(ctx->d_slow.cap, 0x7fffffff);
            // ReadsOther blocks of <= 3 bp: counters [27] = #short blocks, #order-dependent ones (int32 each)
            CK(ctx->d_omask.ensure((size_t)N + 2)); CK(ctx->d_shorts.ensure((size_t)short_cap));
            a.omask = ctx->d_omask.p; a.shorts = ctx->d_shorts.p; a.n_short = (int32_t *)(ctx->d_counters.p + 27); a.short_cap = (int32_t)std::min<int64_t>(short_cap, 0x7fffffff);
            CK(cudaMemsetAsync(ctx->d_counters.p + 27, 0, sizeof(int64_t), ctx->stream));
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
                LAUNCH(k_fix_heads, 256, 128, ctx->d_scratch32.p, ctx->d_sens.p, d_nsens, conc_sens_cap, ctx->d_head.p, ctx->shard_init_hint, (int32_t *)(ctx->d_counters.p + 22));
                LAUNCH(k_fix_chains<false>, 256, 128, b, cd, ctx->params, ctx->nt, ctx->d_scratch32.p, n, ctx->d_sens.p, d_nsens, conc_sens_cap, ctx->d_head.p, sink);
                if (ctx->shard_count > 1) LAUNCH(k_last_located, 1, 1, ctx->d_scratch32.p, n, (int32_t *)(ctx->d_counters.p + 23));
            }
            PHASE_END("k_assign");
        }
        CK(cudaMemcpyAsync(ctx->h_counters.p + 9, ctx->d_counters.p + 9, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_counters.p + 16, ctx->d_counters.p + 16, 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_counters.p + 22, ctx->d_counters.p + 22, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_counters.p + 27, ctx->d_counters.p + 27, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        n_short = do_depth && n > 0 ? ((int32_t *)(ctx->h_counters.p + 27))[0] : 0;
        n_unstable = do_depth && n > 0 ? ((int32_t *)(ctx->h_counters.p + 27))[1] : 0;
        ctx->shard_lead_sensitive = *(int32_t *)(ctx->h_counters.p + 22) != 0;
        ctx->shard_out_hint = (ctx->shard_count > 1 && do_edges && n > 0) ? *(int32_t *)(ctx->h_counters.p + 23) : -1;
        n_raw = ctx->h_counters.p[9];
        const int32_t ns_conc = ((int32_t *)(ctx->h_counters.p + 10))[0], ns_chim = ((int32_t *)(ctx->h_counters.p + 10))[1];
        ctx->n_sensitive = (int64_t)ns_conc + ns_chim;
        const int64_t n_slow = *(int32_t *)(ctx->h_counters.p + 18);
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

// BuildNode_STAR up to the seed segments: classification, the chimeric pre-pass, the island-parallel state machine.
// Leaves this batch's seed ops (island order) in ctx->shard_ops; a range shard owns the groups from shard_g_lo on.
static int seed_stage(sqg_ctx *ctx, HostLap &lap) {
    const DevBatch &b = ctx->batch;
    const int64_t n = b.n_rec;
    ctx->shard_seeded = false;
    int rc = run_classify(ctx);
    if (rc) return rc;
    lap("classify");
    rc = finish_prepass(ctx);
    if (rc) return rc;
    lap("wait for pre-pass + upload");
    const int32_t nD = ctx->pre_nD, nG = ctx->pre_nG, nP = ctx->pre_nP;
    if (nD <= 0) FAIL(SQG_EUNSUPPORTED, "no discordant block in the chimeric reads: BuildNode_STAR is undefined there (SegmentGraph.cpp:757 on an empty vector)");

    PHASE_BEGIN("seed");
    CK(ctx->d_trigger.ensure(nG + 1));
    LAUNCH(k_triggers, blocks_for(nG), kThreads, b, ctx->d_cls.p, ctx->d_groups.p, nG, ctx->d_trigger.p);
    // ConcordRest candidates, sorted by (chr,pos)
    RestBins rbins;
    {   // bitmap of the 1024-bp bins that some group's extended range touches
        const int32_t n_ref = ctx->params.n_ref;
        std::vector<int32_t> off((size_t)n_ref + 1, 0);
        for (int32_t c = 0; c < n_ref; c++) off[c + 1] = off[c] + ((ctx->ref_len[c] > 0 ? ctx->ref_len[c] : 0) >> kRestBinShift) + 1;
        const size_t words = ((size_t)off[n_ref] + 31) / 32 + 1;
        CK(ctx->d_restbits.ensure(words)); CK(ctx->d_restoff.ensure((size_t)n_ref + 1)); CK(ctx->d_reflen.ensure((size_t)n_ref + 1));
        CK(cudaMemsetAsync(ctx->d_restbits.p, 0, words * 4, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_restoff.p, off.data(), ((size_t)n_ref + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));  // (pageable source: staged before the call returns)
        CK(cudaMemcpyAsync(ctx->d_reflen.p, ctx->ref_len.data(), (size_t)n_ref * 4, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(k_rest_mark, blocks_for(nG), kThreads, ctx->d_groups.p, ctx->d_disc.p, nG, ctx->params.read_len, ctx->d_reflen.p, ctx->d_restbits.p, ctx->d_restoff.p);
        rbins.bits = ctx->d_restbits.p; rbins.off = ctx->d_restoff.p;
    }
    int64_t rest_cap = std::max<int64_t>(1024, ctx->d_rest.cap);
    int64_t n_rest = 0;
    for (int attempt = 0; attempt < 2; attempt++) {
        CK(ctx->d_rest.ensure(rest_cap)); CK(ctx->d_rest2.ensure(rest_cap)); CK(ctx->d_restkey.ensure(rest_cap)); CK(ctx->d_restkey2.ensure(rest_cap));
        CK(cudaMemsetAsync(ctx->d_counters.p + 4, 0, sizeof(int64_t), ctx->stream));
        if (n > 0) LAUNCH(k_rest_collect, blocks_for((n + 3) / 4), kThreads, b, ctx->d_cls.p, ctx->d_groups.p, ctx->d_disc.p, nG, ctx->params.read_len, rbins, ctx->d_reflen.p,
                          ctx->d_rest.p, ctx->d_restkey.p, rest_cap, ctx->d_counters.p + 4);
        CK(cudaMemcpyAsync(ctx->h_counters.p + 4, ctx->d_counters.p + 4, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        n_rest = ctx->h_counters.p[4];
        lap("  seed: triggers + rest collect");
        if (n_rest <= rest_cap) break;
        rest_cap = n_rest + 1024;
    }
    if (n_rest > 0) {
        size_t tb = 0;
        int key_bits = 1;  // the owning group: the table is binned by group, not ordered inside a group
        while (key_bits < 32 && (1ll << key_bits) < (long long)nG) key_bits++;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_restkey.p, ctx->d_restkey2.p, ctx->d_rest.p, ctx->d_rest2.p, (int)n_rest, 0, key_bits, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceRadixSort::SortPairs(ctx->d_temp.p, tb, ctx->d_restkey.p, ctx->d_restkey2.p, ctx->d_rest.p, ctx->d_rest2.p, (int)n_rest, 0, key_bits, ctx->stream));
        ctx->launches += 4;
    }
    // the state machine, island-parallel
    SeedInputs in;
    in.b = b; in.cls = ctx->d_cls.p; in.first_len = ctx->d_flen.p; in.gap_other = ctx->d_other.p;
    in.gap_rec = ctx->d_gap.p; in.n_gap = ctx->n_gap; in.pc_rec = ctx->d_pc.p; in.n_pc = ctx->n_pc;
    in.dp_rec = ctx->d_dp.p; in.n_dp = ctx->n_dp; in.lmax = ctx->lmax; in.n_rec = n;
    in.ccmax = n > 0 ? ctx->d_ccmax.p : nullptr; in.cc_tile = kTile;
    in.D = ctx->d_disc.p; in.nD = nD; in.G = ctx->d_groups.p; in.nG = nG; in.trigger = ctx->d_trigger.p;
    in.Pchr = ctx->d_pchr.p; in.Ppos = ctx->d_ppos.p; in.nP = nP;
    in.rest = ctx->d_rest2.p; in.rest_g = ctx->d_restkey2.p; in.n_rest = (int32_t)n_rest; in.read_len = ctx->params.read_len; in.first_kept = ctx->first_kept;
    // range shard (sqg_set_shard): the groups whose right end lies left of this batch's first kept record were triggered in
    // an earlier shard; when another shard follows, the pending segment of the last island is closed at the batch end
    int32_t g_lo = 0;
    if (ctx->shard_index > 0) {
        g_lo = nG;
        if (ctx->first_kept < n) {
            int32_t rp[2];
            CK(cudaMemcpyAsync(&rp[0], b.ref_id + ctx->first_kept, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaMemcpyAsync(&rp[1], b.pos + ctx->first_kept, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            g_lo = 0;
            while (g_lo < nG) {
                const Group &gg = ctx->h_groups[g_lo];
                if (rp[0] < 0 || gg.chr < rp[0] || (gg.chr == rp[0] && gg.right < rp[1])) g_lo++; else break;
            }
        }
    }
    ctx->shard_g_lo = g_lo;
    // groups whose trigger lies behind the batch (trigger == n; triggers are non-decreasing along the groups) are never
    // processed here: keep them out of the islands (they would all pile onto the last one)
    int32_t g_hi = nG;
    {
        std::vector<int64_t> h_trig((size_t)nG);
        CK(cudaMemcpyAsync(h_trig.data(), ctx->d_trigger.p, (size_t)nG * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        g_hi = (int32_t)(std::lower_bound(h_trig.begin(), h_trig.end(), n) - h_trig.begin());
        lap("  seed: rest sort + triggers back");
    }
    if (g_hi < g_lo) g_hi = g_lo;
    in.g_hi = g_hi;
    in.g_lo = g_lo; in.has_next = ctx->shard_index + 1 < ctx->shard_count; in.end_other = ctx->end_other;
    in.dense_max_r = kSeedDenseRange;
    CK(ctx->d_cutflag.ensure(nG + 1)); CK(ctx->d_isl.ensure(nG + 2));
    LAUNCH(k_island_cuts, blocks_for(nG, 64), 64, in, ctx->d_cutflag.p);
    CK(cudaMemsetAsync(ctx->d_counters.p + 5, 0, sizeof(int64_t), ctx->stream));
    if (g_hi - g_lo > 0) {
        cub::CountingInputIterator<int32_t> cnt(g_lo);
        IsCutOp op{ctx->d_cutflag.p};
        size_t tb = 0;
        CK(cub::DeviceSelect::If(nullptr, tb, cnt, ctx->d_isl.p, (int32_t *)(ctx->d_counters.p + 5), g_hi - g_lo, op, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceSelect::If(ctx->d_temp.p, tb, cnt, ctx->d_isl.p, (int32_t *)(ctx->d_counters.p + 5), g_hi - g_lo, op, ctx->stream));
        ctx->launches += 2;
    }
    CK(cudaMemcpyAsync(ctx->h_counters.p + 5, ctx->d_counters.p + 5, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t n_isl = *(int32_t *)(ctx->h_counters.p + 5);
    lap("  seed: island cuts");
    CK(ctx->d_cap_ops.ensure(2 * (size_t)n_isl + 4)); CK(ctx->d_cap_mar.ensure(n_isl + 2)); CK(ctx->d_off_ops.ensure(n_isl + 2)); CK(ctx->d_off_mar.ensure(n_isl + 2));
    CK(ctx->d_isl_nout.ensure(n_isl + 1)); CK(ctx->d_isl_gdone.ensure(n_isl + 1));
    CK(cudaMemsetAsync(ctx->d_cap_ops.p, 0, (n_isl + 2) * 4, ctx->stream)); CK(cudaMemsetAsync(ctx->d_cap_mar.p, 0, (n_isl + 2) * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_isl_nout.p, 0, (n_isl + 1) * 4, ctx->stream));
    CK(ctx->d_span.ensure(n_isl + 2)); CK(ctx->d_heavy.ensure(n_isl + 2)); CK(ctx->d_light.ensure(n_isl + 2));
    LAUNCH(k_island_caps, blocks_for(n_isl, 64), 64, in, ctx->d_isl.p, n_isl, ctx->d_cap_ops.p, ctx->d_cap_mar.p, ctx->d_span.p);
    {
        size_t tb = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, ctx->d_cap_ops.p, ctx->d_off_ops.p, n_isl + 1, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceScan::ExclusiveSum(ctx->d_temp.p, tb, ctx->d_cap_ops.p, ctx->d_off_ops.p, n_isl + 1, ctx->stream));
        CK(cub::DeviceScan::ExclusiveSum(ctx->d_temp.p, tb, ctx->d_cap_mar.p, ctx->d_off_mar.p, n_isl + 1, ctx->stream));
        ctx->launches += 4;
    }
    int64_t tot[2];
    CK(cudaMemcpyAsync(&tot[0], ctx->d_off_ops.p + n_isl, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&tot[1], ctx->d_off_mar.p + n_isl, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    lap("  seed: island caps + offsets");
    CK(ctx->d_ops.ensure(tot[0] + 1)); CK(ctx->d_margin.ensure(tot[1] + 1));
    int32_t *d_err = (int32_t *)(ctx->d_counters.p + 7), *d_nprefix = (int32_t *)(ctx->d_counters.p + 6);
    CK(cudaMemsetAsync(ctx->d_counters.p + 6, 0, 2 * sizeof(int64_t), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_counters.p + 29, 0, sizeof(int64_t), ctx->stream));
    in.win_count = (unsigned long long *)(ctx->d_counters.p + 29);
    // (a shard that follows one with an emitted segment starts with an inherited last segment: no sequential prefix)
    if (!(ctx->shard_index > 0 && ctx->shard_prior_emission) && n_isl > 0)
        LAUNCH(k_seed_prefix, 1, kSeedBlock, in, ctx->d_isl.p, n_isl, ctx->d_off_ops.p, ctx->d_off_mar.p, ctx->d_ops.p, ctx->d_margin.p,
               ctx->d_isl_nout.p, ctx->d_isl_gdone.p, d_err, d_nprefix);
    CK(cudaMemsetAsync(ctx->d_counters.p + 13, 0, sizeof(int64_t), ctx->stream));
    if (n_isl > 0) {
        cub::CountingInputIterator<int32_t> cnt(0);
        size_t tb = 0;
        IsHeavyOp oh{ctx->d_span.p, d_nprefix, true}, ol{ctx->d_span.p, d_nprefix, false};
        int32_t *d_nh = (int32_t *)(ctx->d_counters.p + 13);
        CK(cub::DeviceSelect::If(nullptr, tb, cnt, ctx->d_heavy.p, d_nh, n_isl, oh, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceSelect::If(ctx->d_temp.p, tb, cnt, ctx->d_heavy.p, d_nh, n_isl, oh, ctx->stream));
        CK(cub::DeviceSelect::If(ctx->d_temp.p, tb, cnt, ctx->d_light.p, d_nh + 1, n_isl, ol, ctx->stream));
        ctx->launches += 3;
    }
    CK(cudaMemcpyAsync(ctx->h_counters.p + 13, ctx->d_counters.p + 13, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t n_heavy = ((int32_t *)(ctx->h_counters.p + 13))[0], n_light = ((int32_t *)(ctx->h_counters.p + 13))[1];
    ctx->n_heavy = n_heavy;
    lap("  seed: prefix + heavy/light split");
    if (n_heavy > 1) {  // longest islands first: the kernel's critical path is its largest island
        // d_cap_ops is free again after the offset scans: sort scratch [keys | keys2]
        int32_t *k1 = ctx->d_cap_ops.p, *k2 = ctx->d_cap_ops.p + n_heavy;
        LAUNCH(k_gather_i32, blocks_for(n_heavy), kThreads, ctx->d_span.p, ctx->d_heavy.p, n_heavy, k1);
        size_t tb = 0;
        CK(cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, k1, k2, ctx->d_heavy.p, ctx->d_light.p + n_light, n_heavy, 0, 32, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceRadixSort::SortPairsDescending(ctx->d_temp.p, tb, k1, k2, ctx->d_heavy.p, ctx->d_light.p + n_light, n_heavy, 0, 32, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_heavy.p, ctx->d_light.p + n_light, n_heavy * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        ctx->launches += 2;
    }
    // Phase 3's compaction pass only needs the class bytes.  It is forked HERE, behind the short kernels of this stage and beside the
    // island machine: enqueued right after the classification, its 10^5 blocks sat in front of the ConcordRest collection, which is
    // on the critical path (5.7 ms instead of 1.4 ms).  (The two share the SMs without gaining from it: alone the island kernel
    // takes 5.4 ms and the compaction 2.3, together 7.6; forking the compaction beside the depth tile kernel instead moves the
    // same 2 ms there.  The step is bound by the sum of the work, not by a critical path.)
    rc = run_cov_compact(ctx);
    if (rc) return rc;
    if (n_heavy + n_light > 0) {
        PHASE_BEGIN("k_seed_islands");
        // (block size measured at 100 M pairs: 256 threads 9.6 ms, 512 threads 7.5 ms, 1024 threads 8.9 ms -- the kernel needs both
        // many islands in flight and many lanes on the few long ones)
        k_seed_islands<kSeedBlock><<<(unsigned)(n_heavy + (n_light + kSeedBlock / 32 - 1) / (kSeedBlock / 32)), kSeedBlock, 0, ctx->stream>>>(in, ctx->d_isl.p, n_isl, ctx->d_off_ops.p, ctx->d_off_mar.p,
               ctx->d_ops.p, ctx->d_margin.p, ctx->d_isl_nout.p, ctx->d_isl_gdone.p, d_err, ctx->d_heavy.p, n_heavy, ctx->d_light.p, n_light);
        ctx->launches++;
        CK(cudaGetLastError());
        PHASE_END("k_seed_islands");
    }
    PHASE_END("seed");
    lap("seed: enqueue");
    // this batch's op lists in island order: compacted on the device (the islands' scratch is sized for the worst case, two ops
    // per margin -- copying that capacity cost more than the whole tiling stage), then one small copy
    CK(ctx->d_ops_dense.ensure((size_t)(tot[0] > 0 ? tot[0] : 1)));
    LAUNCH(k_ops_dense, 1, 1024, ctx->d_isl.p, n_isl, g_hi, ctx->d_isl_nout.p, ctx->d_isl_gdone.p, ctx->d_off_ops.p, ctx->d_ops.p, ctx->d_ops_dense.p, ctx->d_counters.p + 24);
    CK(cudaMemcpyAsync(ctx->h_counters.p + 24, ctx->d_counters.p + 24, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_counters.p + 6, ctx->d_counters.p + 6, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_counters.p + 29, ctx->d_counters.p + 29, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<int64_t> trig_last(1, n);
    if (nG > 0) CK(cudaMemcpyAsync(trig_last.data(), ctx->d_trigger.p + (nG - 1), sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t serr = *(int32_t *)(ctx->h_counters.p + 7);
    if (serr) FAIL(SQG_ENOMEM, serr == 1 ? "seed machine: margin scratch overflow" : "seed machine: output overflow");
    const int64_t n_ops_dense = ctx->h_counters.p[24];
    const int32_t g_done = (int32_t)ctx->h_counters.p[25];  // (== nG exactly when every group was triggered by this batch)
    CK(ctx->h_ops.ensure((size_t)n_ops_dense + 1));
    if (n_ops_dense > 0) {
        CK(cudaMemcpyAsync(ctx->h_ops.p, ctx->d_ops_dense.p, (size_t)n_ops_dense * sizeof(SeedOp), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->shard_ops.assign(ctx->h_ops.p, ctx->h_ops.p + n_ops_dense);
    ctx->shard_g_done = g_done;
    ctx->shard_trig_last = trig_last[0];
    ctx->n_islands = n_isl;
    ctx->shard_seeded = true;
    lap("seed: wait + ops");
    return SQG_OK;
}

// The rest of BuildNode_STAR from the stitched seed segments: tiling, depth numerators, and (eagerly) the edge table.
static int finish_stage(sqg_ctx *ctx, std::vector<SeedNode> &seeds, HostLap &lap, int32_t **chr, int32_t **pos, int32_t **len, int64_t *n_nodes,
                        int32_t **count3, int32_t **sumlen3, int32_t *reads_other_nonempty) {
    const int64_t n = ctx->batch.n_rec;
    const int32_t nG = ctx->pre_nG;
    if (seeds.empty()) FAIL(SQG_EUNSUPPORTED, "no seed segment was produced: BuildNode_STAR is undefined there (SegmentGraph.cpp:757 on an empty vector)");
    PHASE_BEGIN("tile");
    int rc = tile_genome(ctx, seeds);
    if (rc) return rc;
    PHASE_END("tile");

    // break index of the depth streams (:338-339): the first kept record after the last group's trigger is still pushed.
    // Range shards: the shard planner keeps two kept records of the owning shard behind every group, so the break falls
    // into the shard that owns the last group; later shards contribute nothing to the depth streams.
    ctx->r_break = n;
    if (ctx->shard_index > 0 && ctx->shard_g_lo == nG) ctx->r_break = 0;
    else if (ctx->shard_g_done == nG) {
        // find it on the device-side class bytes via a tiny host loop over a copied window
        int64_t r = ctx->shard_trig_last + 1;
        std::vector<uint8_t> win(4096);
        bool found = false;
        while (r < n && !found) {
            const int64_t m = std::min<int64_t>(4096, n - r);
            CK(cudaMemcpyAsync(win.data(), ctx->d_cls.p + r, m, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            for (int64_t k = 0; k < m; k++) if (win[k] & CLS_KEEP) { ctx->r_break = r + k + 1; found = true; break; }
            r += m;
        }
    }
    lap("tile + r_break");
    // phase 2 in one pass: per-segment depth and, eagerly, the assignment + raw edges sqg_build_edges will ask for
    const int32_t N = ctx->nt.n;
    rc = run_assign(ctx, true, true);
    if (rc) return rc;
    lap("assign + edge reduce");
    CK(ctx->h_chr.ensure(N)); CK(ctx->h_pos.ensure(N)); CK(ctx->h_len.ensure(N)); CK(ctx->h_cnt3.ensure(3 * (size_t)N + 4)); CK(ctx->h_sum3.ensure(3 * (size_t)N + 4));
    CK(cudaMemcpyAsync(ctx->h_cnt3.p, ctx->d_cnt3.p, (3 * (size_t)N + 4) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_sum3.p, ctx->d_sum3.p, 3 * (size_t)N * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int32_t i = 0; i < N; i++) { ctx->h_chr.p[i] = ctx->h_nchr[i]; ctx->h_pos.p[i] = ctx->h_npos[i]; ctx->h_len.p[i] = ctx->h_nend[i] - ctx->h_npos[i]; }
    *chr = ctx->h_chr.p; *pos = ctx->h_pos.p; *len = ctx->h_len.p; *n_nodes = N;
    *count3 = ctx->h_cnt3.p; *sumlen3 = ctx->h_sum3.p;
    *reads_other_nonempty = ctx->h_cnt3.p[3 * (size_t)N] != 0;
    lap("outputs");
    return SQG_OK;
}

extern "C" int sqg_build_nodes(sqg_ctx *ctx, int32_t **chr, int32_t **pos, int32_t **len, int64_t *n_nodes,
                               int32_t **count3, int32_t **sumlen3, int32_t *reads_other_nonempty) {
    if (!ctx || !chr || !pos || !len || !n_nodes || !count3 || !sumlen3 || !reads_other_nonempty) return SQG_EINVAL;
    if (!ctx->have_batch || !ctx->have_chim) FAIL(SQG_ESTATE, "load the concordant batch and the chimeric reads first");
    if (ctx->shard_count > 1) FAIL(SQG_ESTATE, "this context is a range shard: use sqg_shard_seeds / sqg_shard_build");
    CK(cudaSetDevice(ctx->device));
    HostLap lap;
    int rc = seed_stage(ctx, lap);
    if (rc) return rc;
    std::vector<SeedNode> seeds;
    stitch_ops(ctx->shard_ops.data(), (int32_t)ctx->shard_ops.size(), seeds);
    return finish_stage(ctx, seeds, lap, chr, pos, len, n_nodes, count3, sumlen3, reads_other_nonempty);
}

// ---- range shards of one genome (SURVEY.md 8e) --------------------------------------------------------------------
extern "C" int sqg_set_shard(sqg_ctx *ctx, int32_t index, int32_t count) {
    if (!ctx || count < 1 || index < 0 || index >= count) return SQG_EINVAL;
    ctx->shard_index = index; ctx->shard_count = count; ctx->shard_prior_emission = index > 0; ctx->shard_init_hint = 0;
    ctx->shard_seeded = false; ctx->have_edge_table = false;
    return SQG_OK;
}
extern "C" int sqg_shard_seeds(sqg_ctx *ctx, int32_t prior_emission, const int32_t **ops, int64_t *n_ops) {
    if (!ctx || !ops || !n_ops) return SQG_EINVAL;
    if (!ctx->have_batch || !ctx->have_chim) FAIL(SQG_ESTATE, "load the concordant batch and the chimeric reads first");
    CK(cudaSetDevice(ctx->device));
    ctx->shard_prior_emission = ctx->shard_index > 0 && prior_emission != 0;
    HostLap lap;
    int rc = seed_stage(ctx, lap);
    if (rc) return rc;
    static_assert(sizeof(SeedOp) == 16, "SeedOp crosses the C ABI as 4 x int32");
    *ops = (const int32_t *)ctx->shard_ops.data(); *n_ops = (int64_t)ctx->shard_ops.size();
    return SQG_OK;
}
extern "C" int sqg_shard_build(sqg_ctx *ctx, const int32_t *ops_all, int64_t n_ops_all, int32_t **chr, int32_t **pos, int32_t **len, int64_t *n_nodes,
                               int32_t **count3, int32_t **sumlen3, int32_t *reads_other_nonempty) {
    if (!ctx || (n_ops_all > 0 && !ops_all) || n_ops_all < 0 || n_ops_all > 0x7fffffff || !chr || !pos || !len || !n_nodes || !count3 || !sumlen3 || !reads_other_nonempty) return SQG_EINVAL;
    if (!ctx->shard_seeded) FAIL(SQG_ESTATE, "sqg_shard_seeds must run first");
    CK(cudaSetDevice(ctx->device));
    HostLap lap;
    std::vector<SeedNode> seeds;
    stitch_ops((const SeedOp *)ops_all, (int32_t)n_ops_all, seeds);
    ctx->shard_init_hint = 0;
    return finish_stage(ctx, seeds, lap, chr, pos, len, n_nodes, count3, sumlen3, reads_other_nonempty);
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
        size_t tb1 = 0, tb2 = 0, tb3 = 0;
        int32_t *d_nsel = (int32_t *)(ctx->d_counters.p + 5);
        CK(cub::DeviceScan::ExclusiveScan(nullptr, tb1, ctx->d_plan_reach.p, ctx->d_plan_reach.p, MaxU64(), (uint64_t)0, (int)n, ctx->stream));
        CK(cub::DeviceScan::ExclusiveScan(nullptr, tb2, ctx->d_plan_keep.p, ctx->d_plan_keep.p, MaxI32(), (int32_t)-1, (int)n, ctx->stream));
        CK(cub::DeviceSelect::If(nullptr, tb3, ctx->d_plan_cand.p, ctx->d_plan_sel.p, d_nsel, (int)n, PlanIsCand(), ctx->stream));
        ENSURE_TEMP(std::max({tb1, tb2, tb3}));
        CK(cub::DeviceScan::ExclusiveScan(ctx->d_temp.p, tb1, ctx->d_plan_reach.p, ctx->d_plan_reach.p, MaxU64(), (uint64_t)0, (int)n, ctx->stream));
        CK(cub::DeviceScan::ExclusiveScan(ctx->d_temp.p, tb2, ctx->d_plan_keep.p, ctx->d_plan_keep.p, MaxI32(), (int32_t)-1, (int)n, ctx->stream));
        CK(cub::DeviceScan::ExclusiveScan(ctx->d_temp.p, tb2, ctx->d_plan_upd.p, ctx->d_plan_upd.p, MaxI32(), (int32_t)-1, (int)n, ctx->stream));
        LAUNCH(k_plan_cands, blocks_for(n), kThreads, b, ctx->params, ctx->d_cls.p, ctx->d_plan_reach.p, ctx->d_plan_keep.p, ctx->d_plan_upd.p,
               ctx->d_groups.p, ctx->d_disc.p, ctx->pre_nG, ctx->d_plan_cand.p);
        CK(cub::DeviceSelect::If(ctx->d_temp.p, tb3, ctx->d_plan_cand.p, ctx->d_plan_sel.p, d_nsel, (int)n, PlanIsCand(), ctx->stream));
        ctx->launches += 4;
        CK(cudaMemcpyAsync(ctx->h_counters.p + 5, ctx->d_counters.p + 5, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        n_cand = *(const int32_t *)(ctx->h_counters.p + 5);
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
    CK(ctx->d_counters.ensure(32)); CK(ctx->h_counters.ensure(32));
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
    move(ctx->o_ref_id.p, 4, lo, nr); move(ctx->o_pos.p, 4, lo, nr); move(ctx->o_mate_ref_id.p, 4, lo, nr); move(ctx->o_mate_pos.p, 4, lo, nr);
    move(ctx->o_end_pos.p, 4, lo, nr); move(ctx->o_flag.p, 2, lo, nr); move(ctx->o_total_len.p, 2, lo, nr); move(ctx->o_lowphred_run.p, 2, lo, nr);
    move(ctx->o_mapq.p, 1, lo, nr); move(ctx->o_aux.p, 1, lo, nr);
    move(ctx->o_blk_ref_pos.p, 4, b0, nb); move(ctx->o_blk_match_ref.p, 4, b0, nb); move(ctx->o_blk_read_pos.p, 2, b0, nb); move(ctx->o_blk_match_read.p, 2, b0, nb);
    CK(e);
    CK(cudaMemcpyAsync(tmp.p, ctx->o_blk_off.p + lo, (size_t)(nr + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    LAUNCH(k_keep_offsets, blocks_for(nr + 1), kThreads, ctx->o_blk_off.p, (const uint32_t *)tmp.p, nr + 1, (uint32_t)b0);
    CK(cudaStreamSynchronize(st));
    ctx->batch.n_rec = nr; ctx->batch.n_blk = nb;
    reset_batch_state(ctx, true, ctx->first_record_index + lo, ctx->wire_loaded);
    ctx->batch_restricted = true; ctx->classify_prelaunched = false;  // (a classification launched on the whole batch does not apply)
    return SQG_OK;
}

// sort raw keys, run-length reduce, unpack
static int reduce_edges(sqg_ctx *ctx, int64_t n_raw, const int32_t *d_weights_in) {
    ctx->n_unique_edges = 0;
    CK(ctx->d_ekeys2.ensure(n_raw + 1)); CK(ctx->d_ukeys.ensure(n_raw + 1)); CK(ctx->d_ecount.ensure(n_raw + 1));
    if (n_raw > 0) {
        size_t tb = 0;
        if (!d_weights_in) {
            CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, (int)n_raw, 0, 64, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceRadixSort::SortKeys(ctx->d_temp.p, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, (int)n_raw, 0, 64, ctx->stream));
            CK(cub::DeviceRunLengthEncode::Encode(nullptr, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_ecount.p, (int32_t *)(ctx->d_counters.p + 8), (int)n_raw, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceRunLengthEncode::Encode(ctx->d_temp.p, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_ecount.p, (int32_t *)(ctx->d_counters.p + 8), (int)n_raw, ctx->stream));
        } else {
            CK(ctx->d_sens.ensure(n_raw + 1));
            CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, d_weights_in, ctx->d_sens.p, (int)n_raw, 0, 64, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceRadixSort::SortPairs(ctx->d_temp.p, tb, ctx->d_ekeys.p, ctx->d_ekeys2.p, d_weights_in, ctx->d_sens.p, (int)n_raw, 0, 64, ctx->stream));
            CK(cub::DeviceReduce::ReduceByKey(nullptr, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_sens.p, ctx->d_ecount.p, (int32_t *)(ctx->d_counters.p + 8), cub::Sum(), (int)n_raw, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceReduce::ReduceByKey(ctx->d_temp.p, tb, ctx->d_ekeys2.p, ctx->d_ukeys.p, ctx->d_sens.p, ctx->d_ecount.p, (int32_t *)(ctx->d_counters.p + 8), cub::Sum(), (int)n_raw, ctx->stream));
        }
        ctx->launches += 5;
        CK(cudaMemcpyAsync(ctx->h_counters.p + 8, ctx->d_counters.p + 8, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->n_unique_edges = *(int32_t *)(ctx->h_counters.p + 8);
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
            CK(cudaMemsetAsync(ctx->d_counters.p + 26, 0, sizeof(int64_t), ctx->stream));
            LAUNCH(k_chim_diff, blocks_for(nb), kThreads, ctx->dc0_ref_pos.p, ctx->dc0_read_pos.p, ctx->dc0_match_ref.p, ctx->dc0_match_read.p,
                   ctx->dc_ref_pos.p, ctx->dc_read_pos.p, ctx->dc_match_ref.p, ctx->dc_match_read.p, nb, ctx->d_chimdiff.p, (int32_t)std::min<int64_t>(cap, 0x7fffffff), (int32_t *)(ctx->d_counters.p + 26));
            CK(cudaMemcpyAsync(ctx->h_counters.p + 26, ctx->d_counters.p + 26, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            const int64_t nd = *(int32_t *)(ctx->h_counters.p + 26);
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
    ctx->cov_nq = n > 0 ? ctx->h_counters.p[15] : 0;
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
        size_t tb = 0;
        CK(cub::DeviceScan::InclusiveScan(nullptr, tb, t, t, MaxI64(), (int)K, ctx->stream));
        ENSURE_TEMP(tb);
        CK(cub::DeviceScan::InclusiveScan(ctx->d_temp.p, tb, t, t, MaxI64(), (int)K, ctx->stream));
        ctx->launches += 2;
        CK(cudaMemsetAsync(ctx->d_counters.p + 12, 0, sizeof(int64_t), ctx->stream));
        LAUNCH(k_cov_verify, blocks_for(K), kThreads, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, (int32_t *)(ctx->d_counters.p + 12));
        CK(cudaMemcpyAsync(ctx->h_counters.p + 12, ctx->d_counters.p + 12, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->cov_chain_fallback = *(int32_t *)(ctx->h_counters.p + 12) != 0;
        if (ctx->cov_chain_fallback) {
            // literal chain, chunked at large jumps of r0 (one warp per chunk), validated; whole-list replay as a last resort
            cub::CountingInputIterator<int32_t> cnt(0);
            IsChainCutOp cop{r0, t};
            CK(ctx->d_chunks.ensure(K + 1));
            int32_t *chunks = ctx->d_chunks.p;
            CK(cub::DeviceSelect::If(nullptr, tb, cnt, chunks, (int32_t *)(ctx->d_counters.p + 14), (int)K, cop, ctx->stream));
            ENSURE_TEMP(tb);
            CK(cub::DeviceSelect::If(ctx->d_temp.p, tb, cnt, chunks, (int32_t *)(ctx->d_counters.p + 14), (int)K, cop, ctx->stream));
            CK(cudaMemcpyAsync(ctx->h_counters.p + 14, ctx->d_counters.p + 14, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            const int32_t n_chunks = *(int32_t *)(ctx->h_counters.p + 14);
            ctx->launches += 2;
            CK(ctx->d_chain_used.ensure(2 * (size_t)n_chunks + 2));
            int64_t *used = ctx->d_chain_used.p, *need = ctx->d_chain_used.p + n_chunks + 1;
            LAUNCH(k_cov_chain, blocks_for((int64_t)n_chunks * 32, 128), 128, ctx->d_qkey.p, nq, bpchr, bppos, K, ctx->params.concord_dist_pos, r0, t, chunks, n_chunks,
                   used, (const int64_t *)nullptr);
            // chunks whose predecessor's chain runs into them are replayed from its t; a few rounds settle runs of such chunks
            ctx->cov_chain_chunks = n_chunks;
            bool settled = false;
            for (int round = 0; round < 16 && !settled; round++) {
                CK(cudaMemsetAsync(ctx->d_counters.p + 12, 0, sizeof(int64_t), ctx->stream));
                LAUNCH(k_cov_chain_check, blocks_for(n_chunks), kThreads, chunks, n_chunks, r0, t, used, need, (int32_t *)(ctx->d_counters.p + 12));
                CK(cudaMemcpyAsync(ctx->h_counters.p + 12, ctx->d_counters.p + 12, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
                if (*(int32_t *)(ctx->h_counters.p + 12) == 0) { settled = true; break; }
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

// ------------------------------------------------------------------------------------------------
// Concordant BAM decoded on the device (sq_inflate.cuh, sq_bam.cuh): the host maps the file, indexes the BGZF members and
// streams the compressed bytes through pinned staging; per window of whole members the device inflates (one member per warp),
// finds the record boundaries (speculative segment starts proven in parallel, repaired in rounds) and decodes the records into
// the resident batch.  Only the header is read on the host.
// ------------------------------------------------------------------------------------------------
constexpr int kInflWarps = 8;
constexpr size_t kBamStage = 32u << 20;  // bytes per pinned staging buffer
enum { BS_CHANGED = 0, BS_BAD, BS_AUXBAD, BS_ERRKEY, BS_SEQ, BS_INFL, BS_N };

__global__ void __launch_bounds__(kInflWarps * 32) k_bam_inflate(const BamMember *mem, int64_t n, const uint8_t *comp, uint8_t *win, int64_t *small) {
    __shared__ InflateTables tabs[kInflWarps];
    __shared__ uint32_t crc_tab[256], x2n[32];
    crc_tab[threadIdx.x] = crc32_entry(threadIdx.x);
    if (threadIdx.x == 0) crc32_x2n(x2n);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * kInflWarps + warp;
    if (k >= n) return;
    const BamMember m = mem[k];
    uint8_t *out = win + m.out;
    InflateState s;
    int rc = 0;
    if (lane == 0) inflate_init(s, comp + m.cdata, m.clen, out, m.isize);
    for (;;) {  // lane 0 decodes; a long match comes back to the warp, which copies it
        uint32_t dst = 0, len = 0, dist = 1;
        if (lane == 0) rc = inflate_step(s, tabs[warp], kInflWarpCopyMin, &dst, &len, &dist);
        __syncwarp();
        rc = __shfl_sync(0xFFFFFFFFu, rc, 0);
        if (rc != 1) break;
        dst = __shfl_sync(0xFFFFFFFFu, dst, 0); len = __shfl_sync(0xFFFFFFFFu, len, 0); dist = __shfl_sync(0xFFFFFFFFu, dist, 0);
        for (uint32_t i = lane; i < len; i += 32) out[dst + i] = out[dst - dist + i % dist];  // sources all lie before dst
        __syncwarp();
    }
    if (rc < 0) { if (lane == 0) atomicOr((unsigned long long *)&small[BS_INFL], 1ull); return; }
    __syncwarp();
    const uint32_t a = (uint32_t)((uint64_t)m.isize * lane / 32), b = (uint32_t)((uint64_t)m.isize * (lane + 1) / 32);
    uint32_t crc = crc32_update(crc_tab, 0, out + a, b - a), len = b - a;
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t c2 = __shfl_down_sync(0xFFFFFFFFu, crc, off), l2 = __shfl_down_sync(0xFFFFFFFFu, len, off);
        if ((lane & (2 * off - 1)) == 0) { crc = crc32_combine(x2n, crc, c2, l2); len += l2; }
    }
    if (lane == 0 && crc != m.crc) atomicOr((unsigned long long *)&small[BS_INFL], 2ull);
}

struct BamWin { const uint8_t *b; int64_t L, Lstream; int32_t n_ref; int64_t S; const int64_t *seg; };
SQ_HD int64_t bam_seg_end(const BamWin &w, int64_t k) { return k + 1 < w.S ? w.seg[k + 1] : w.L; }

__global__ void k_bam_spec(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    const int64_t e = bam_seg_end(w, k);
    const int64_t a = k == 0 ? w.seg[0] : bam_spec_start(w.b, w.seg[k], e, w.L, w.Lstream, w.n_ref);
    const SegWalk r = bam_walk(w.b, a, e, w.L, w.Lstream, nullptr);
    start[k] = a; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
}
__global__ void k_bam_mark(BamWin w, const int64_t *start, const int64_t *exit, int64_t *newstart, uint8_t *redo, int64_t *small) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    const bool r = k > 0 && exit[k - 1] != start[k];
    redo[k] = r;
    if (r) { newstart[k] = exit[k - 1]; atomicAdd((unsigned long long *)&small[BS_CHANGED], 1ull); }
}
__global__ void k_bam_rewalk(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad, const int64_t *newstart, const uint8_t *redo) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S || !redo[k]) return;
    const SegWalk r = bam_walk(w.b, newstart[k], bam_seg_end(w, k), w.L, w.Lstream, nullptr);
    start[k] = newstart[k]; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
}
__global__ void k_bam_sequential(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad) {
    int64_t a = w.seg[0];
    for (int64_t k = 0; k < w.S; k++) {
        const SegWalk r = bam_walk(w.b, a, bam_seg_end(w, k), w.L, w.Lstream, nullptr);
        start[k] = a; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
        a = r.exit;
    }
}
__global__ void k_bam_offsets(BamWin w, const int64_t *start, const uint8_t *bad, const uint32_t *base, int64_t *rec_off, int64_t *small) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    if (bad[k]) { atomicOr((unsigned long long *)&small[BS_BAD], 1ull); return; }
    bam_walk(w.b, start[k], bam_seg_end(w, k), w.L, w.Lstream, rec_off + base[k]);
}

struct BamOut {
    int32_t *ref_id, *pos, *mate_ref_id, *mate_pos, *end_pos;
    uint16_t *flag, *total_len, *lowphred_run;
    uint8_t *mapq, *aux;
    uint32_t *blk_off;
    int32_t *blk_ref_pos, *blk_match_ref;
    uint16_t *blk_read_pos, *blk_match_read;
    uint16_t *lseq;  // non-null only under the synthesised-quality rule
};
__global__ void k_bam_decode(const uint8_t *b, const int64_t *rec_off, int64_t n, int64_t r0, BamDecodeParams prm, NameSet ns, BamOut o, uint32_t *nblk, int64_t *small) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    BamRec x;
    bam_decode(b + rec_off[i], prm, ns, x);
    const int64_t r = r0 + i;
    o.ref_id[r] = x.ref_id; o.pos[r] = x.pos; o.mate_ref_id[r] = x.mate_ref_id; o.mate_pos[r] = x.mate_pos; o.end_pos[r] = x.end_pos;
    o.flag[r] = x.flag; o.mapq[r] = x.mapq; o.aux[r] = x.aux;
    o.total_len[r] = (uint16_t)x.total_len;
    o.lowphred_run[r] = (uint16_t)(x.lowphred < 65535 ? x.lowphred : 65535);
    if (o.lseq) o.lseq[r] = (uint16_t)((uint32_t)x.lseq_cigar < 65535u ? (uint32_t)x.lseq_cigar : 65535u);
    nblk[i] = x.n_blk;
    if (x.aux_bad) atomicOr((unsigned long long *)&small[BS_AUXBAD], 1ull);
    if (x.l_seq) small[BS_SEQ] = 1;
    // pack_concordant's refusals, the first record in file order wins: key = record << 33 | (limit - 1) << 32 | TotalLen
    if (const int lim = packer_limit(x.n_blk, x.total_len))
        atomicMin((unsigned long long *)&small[BS_ERRKEY], ((unsigned long long)r << 33) | ((unsigned long long)(lim - 1) << 32) | (uint32_t)x.total_len);
}
__global__ void k_bam_blocks(const uint8_t *b, const int64_t *rec_off, int64_t n, int64_t r0, uint64_t b0, const uint64_t *incl, const uint32_t *nblk, BamOut o) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t first = b0 + incl[i] - nblk[i];
    o.blk_off[r0 + i + 1] = (uint32_t)(b0 + incl[i]);
    bam_blocks(b + rec_off[i], [&](uint32_t k, int32_t ref_pos, int32_t match_ref, int32_t read_pos, int32_t match_read) {
        o.blk_ref_pos[first + k] = ref_pos; o.blk_match_ref[first + k] = match_ref;
        o.blk_read_pos[first + k] = (uint16_t)read_pos; o.blk_match_read[first + k] = (uint16_t)match_read;
    });
}
__global__ void k_bam_null_qual(uint16_t *lowphred_run, const uint16_t *lseq, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) lowphred_run[i] = lseq[i];
}

namespace {
struct MappedFile {
    const uint8_t *p = nullptr; size_t n = 0;
    ~MappedFile() { if (p) munmap((void *)p, n); }
};
}  // namespace

static int bam_load(sqg_ctx *ctx, const char *path, const sqg_bam_decode *opt, int64_t first_record_index) {
    HostLap lap;
    MappedFile mf;
    {  // the host front end's wording for a missing / empty file
        int fd = ::open(path, O_RDONLY);
        if (fd < 0) FAIL(SQG_EINVAL, std::string("cannot open ") + path);
        struct stat st;
        if (fstat(fd, &st) != 0 || st.st_size < 4) { ::close(fd); FAIL(SQG_EINVAL, std::string(path) + " is empty"); }
        void *m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        ::close(fd);
        if (m == MAP_FAILED) FAIL(SQG_EINVAL, std::string("cannot map ") + path);
        mf.p = (const uint8_t *)m; mf.n = (size_t)st.st_size;
    }
    const uint8_t *f = mf.p;
    const bool raw = memcmp(f, "BAM\1", 4) == 0;
    std::vector<sqh::BgzfMember> mem;
    std::string e;
    if (!sqh::bam_loader_members(f, mf.n, raw, mem, e)) FAIL(SQG_EINVAL, e);
    std::vector<std::string> ref_names;
    std::vector<int32_t> ref_lens;
    size_t hdr_end = 0;
    std::string hdr_err;
    const bool hdr_ok = sqh::bam_read_header(f, mf.n, raw ? nullptr : &mem, ref_names, ref_lens, hdr_end, hdr_err);
    if (raw && !hdr_ok) FAIL(SQG_EINVAL, hdr_err);
    lap("bam: index + header");
    const int64_t T = mem.empty() ? 0 : (int64_t)(mem.back().off + mem.back().isize);
    // windows of whole members, about SQG_BAM_WINDOW_MB of inflated bytes
    const int64_t win_bytes = (int64_t)std::max(1, getenv("SQG_BAM_WINDOW_MB") ? atoi(getenv("SQG_BAM_WINDOW_MB")) : 1024) << 20;
    const std::vector<size_t> wcut = sqh::bam_window_cuts(mem, win_bytes, hdr_end);
    const size_t W = wcut.size() - 1;
    if (W == 0) FAIL(SQG_EINVAL, hdr_err);  // no data at all
    ctx->bam_members = (int64_t)mem.size(); ctx->bam_windows = (int64_t)W; ctx->bam_repair_rounds = 0;
    const int64_t nn = opt->n_names;
    const sqh::NameTable nt = sqh::bam_name_table(opt->names, opt->name_off, nn);
    const size_t cap = nt.hash.size();
    const int64_t blob_len = nn > 0 ? opt->name_off[nn] : 0;
    cudaStream_t st = ctx->stream;
    if (!ctx->stream_up) CK(cudaStreamCreateWithFlags(&ctx->stream_up, cudaStreamNonBlocking));
    cudaStream_t up = ctx->stream_up;
    while (ctx->bam_ev.size() < 3) { cudaEvent_t ev; CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)); ctx->bam_ev.push_back(ev); }
    CK(ctx->bam_nhash.ensure(cap)); CK(ctx->bam_nlen.ensure(cap)); CK(ctx->bam_noff.ensure(cap)); CK(ctx->bam_nblob.ensure((size_t)blob_len + 1));
    CK(cudaMemcpyAsync(ctx->bam_nhash.p, nt.hash.data(), cap * 8, cudaMemcpyHostToDevice, st)); CK(cudaMemcpyAsync(ctx->bam_nlen.p, nt.len.data(), cap * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->bam_noff.p, nt.off.data(), cap * 8, cudaMemcpyHostToDevice, st));
    if (blob_len) CK(cudaMemcpyAsync(ctx->bam_nblob.p, opt->names, (size_t)blob_len, cudaMemcpyHostToDevice, st));
    NameSet ns{ctx->bam_nhash.p, ctx->bam_nlen.p, ctx->bam_noff.p, ctx->bam_nblob.p, cap - 1, nn > 0};
    const int thr = phred_threshold(opt->phred33, opt->min_phred);
    const BamDecodeParams prm{thr};
    // with no qualities anywhere in the file the host decoder synthesises them ('I' everywhere, decode_alignment), which only
    // matters when the threshold lies above 'I': then the run is the read length of the CIGAR
    const bool keep_lseq = thr > 'I';
    CK(ctx->bam_small.ensure(BS_N)); CK(ctx->bam_hsmall.ensure(BS_N));
    CK(ctx->d_counters.ensure(32)); CK(ctx->h_counters.ensure(32));  // sqg_download_concordant reads the wire-consistency slot
    CK(cudaMemsetAsync(ctx->d_counters.p + 28, 0, sizeof(int64_t), st));
    for (int i = 0; i < 2; i++) CK(ctx->bam_stage[i].ensure(kBamStage));
    for (const char *nm : {"bam_h2d", "bam_inflate", "bam_records", "bam_decode"}) { ctx->acc_ms[nm] = 0.f; PhaseTimer &t = ctx->timers[nm]; if (!t.a) { CK(cudaEventCreate(&t.a)); CK(cudaEventCreate(&t.b)); } t.done = false; }
    const int64_t zero_small[BS_N] = {0, 0, 0, -1, 0, 0};  // BS_ERRKEY: ~0 as unsigned, the neutral element of atomicMin
    CK(cudaMemcpyAsync(ctx->bam_small.p, zero_small, sizeof(zero_small), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    int64_t R = 0;        // records so far
    uint64_t B = 0;       // blocks so far
    int64_t carry = 0;    // unconsumed tail of the previous window, at the front of this one's buffer
    int cur = 0;
    int fatal = 0;        // walk / header / capacity refusal: later windows are only inflated (an inflate error outranks it, as on the host)
    std::string fatal_msg;
    bool aux_bad = false;
    int64_t infl_bits = 0;
    auto elapsed = [&](const char *nm) { PhaseTimer &t = ctx->timers[nm]; float ms = 0.f; if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) ctx->acc_ms[nm] += ms; };
    for (size_t w = 0; w < W; w++) {
        const sqh::BgzfMember &m0 = mem[wcut[w]], &m1 = mem[wcut[w + 1] - 1];
        const int64_t wstream = (int64_t)m0.off, wisize = (int64_t)(m1.off + m1.isize) - wstream;
        const int64_t L = carry + wisize, Lstream = carry + (T - wstream);
        // -- upload: the file range of the window's members, through two pinned staging buffers; raw streams go straight to the window
        const size_t f0 = m0.cdata, f1 = m1.cdata + m1.clen;
        CK(ctx->bam_win[cur].grow((size_t)L + 8, 0, st));
        uint8_t *dwin = ctx->bam_win[cur].p;
        if (carry) CK(cudaMemcpyAsync(dwin, ctx->bam_win[cur ^ 1].p + (ctx->bam_win_len - carry), (size_t)carry, cudaMemcpyDeviceToDevice, st));
        uint8_t *dst = raw ? dwin + carry : nullptr;
        if (!raw) { CK(ctx->bam_comp.ensure(f1 - f0)); dst = ctx->bam_comp.p; }
        CK(cudaEventRecord(ctx->bam_ev[2], st)); CK(cudaStreamWaitEvent(up, ctx->bam_ev[2], 0));  // buffers free of the previous window
        CK(cudaEventRecord(ctx->timers["bam_h2d"].a, up));
        for (size_t o = f0, c = 0; o < f1; o += kBamStage, c++) {
            const size_t len = std::min(kBamStage, f1 - o), sb = c & 1;
            if (c >= 2) CK(cudaEventSynchronize(ctx->bam_ev[sb]));
            memcpy(ctx->bam_stage[sb].p, f + o, len);
            CK(cudaMemcpyAsync(dst + (o - f0), ctx->bam_stage[sb].p, len, cudaMemcpyHostToDevice, up));
            CK(cudaEventRecord(ctx->bam_ev[sb], up));
        }
        CK(cudaEventRecord(ctx->timers["bam_h2d"].b, up));
        CK(cudaStreamWaitEvent(st, ctx->timers["bam_h2d"].b, 0));
        // -- inflate
        CK(cudaEventRecord(ctx->timers["bam_inflate"].a, st));
        if (!raw) {
            const int64_t nm = (int64_t)(wcut[w + 1] - wcut[w]);
            std::vector<BamMember> hm((size_t)nm);
            for (int64_t i = 0; i < nm; i++) {
                const sqh::BgzfMember &m = mem[wcut[w] + (size_t)i];
                hm[(size_t)i] = BamMember{m.cdata - f0, (uint64_t)(carry + ((int64_t)m.off - wstream)), (uint32_t)m.clen, m.isize, m.crc, 0};
            }
            CK(ctx->bam_mem.ensure((size_t)nm));
            CK(cudaMemcpyAsync(ctx->bam_mem.p, hm.data(), hm.size() * sizeof(BamMember), cudaMemcpyHostToDevice, st));
            LAUNCH_ON(st, k_bam_inflate, (unsigned)((nm + kInflWarps - 1) / kInflWarps), kInflWarps * 32, ctx->bam_mem.p, nm, ctx->bam_comp.p, dwin, ctx->bam_small.p);
            CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));  // (pageable member table: the copy above must finish before hm goes)
            infl_bits |= ctx->bam_hsmall.p[BS_INFL];
        }
        CK(cudaEventRecord(ctx->timers["bam_inflate"].b, st));
        if (w == 0 && !hdr_ok && !fatal) { fatal = SQG_EINVAL; fatal_msg = hdr_err; }
        if (infl_bits || fatal) { CK(cudaStreamSynchronize(st)); elapsed("bam_h2d"); elapsed("bam_inflate"); carry = 0; continue; }
        // -- record boundaries
        CK(cudaEventRecord(ctx->timers["bam_records"].a, st));
        const std::vector<int64_t> seg = sqh::bam_window_segments(mem, wcut, w, carry, hdr_end);
        const int64_t S = (int64_t)seg.size();
        CK(ctx->bam_seg.ensure((size_t)S)); CK(ctx->bam_start.ensure((size_t)S)); CK(ctx->bam_exit.ensure((size_t)S)); CK(ctx->bam_newstart.ensure((size_t)S));
        CK(ctx->bam_cnt.ensure((size_t)S + 1)); CK(ctx->bam_base.ensure((size_t)S + 1)); CK(ctx->bam_bad.ensure((size_t)S)); CK(ctx->bam_redo.ensure((size_t)S));
        CK(cudaMemcpyAsync(ctx->bam_seg.p, seg.data(), (size_t)S * 8, cudaMemcpyHostToDevice, st));
        const BamWin bw{dwin, L, Lstream, (int32_t)ref_lens.size(), S, ctx->bam_seg.p};
        LAUNCH_ON(st, k_bam_spec, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p);
        for (int round = 0;; round++) {
            CK(cudaMemsetAsync(ctx->bam_small.p + BS_CHANGED, 0, 8, st));
            LAUNCH_ON(st, k_bam_mark, blocks_for(S), kThreads, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_newstart.p, ctx->bam_redo.p, ctx->bam_small.p);
            CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (ctx->bam_hsmall.p[BS_CHANGED] == 0) break;
            ctx->bam_repair_rounds++;
            if (round == kBamMaxRounds) {
                LAUNCH_ON(st, k_bam_sequential, 1, 1, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p);
                break;
            }
            LAUNCH_ON(st, k_bam_rewalk, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p, ctx->bam_newstart.p, ctx->bam_redo.p);
        }
        CK(cudaMemsetAsync(ctx->bam_cnt.p + S, 0, 4, st));
        size_t tb = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, ctx->bam_cnt.p, ctx->bam_base.p, (int)(S + 1), st));
        { const int rc_ = ensure_temp(ctx, tb); if (rc_) return rc_; }
        CK(cub::DeviceScan::ExclusiveSum(ctx->d_temp.p, tb, ctx->bam_cnt.p, ctx->bam_base.p, (int)(S + 1), st));
        int64_t nrec_w = 0, tail = 0;
        uint32_t nrec32 = 0;
        CK(cudaMemcpyAsync(&nrec32, ctx->bam_base.p + S, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&tail, ctx->bam_exit.p + (S - 1), 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nrec_w = nrec32;
        CK(ctx->bam_recoff.ensure((size_t)nrec_w + 1));
        LAUNCH_ON(st, k_bam_offsets, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_bad.p, ctx->bam_base.p, ctx->bam_recoff.p, ctx->bam_small.p);
        CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventRecord(ctx->timers["bam_records"].b, st));
        if (ctx->bam_hsmall.p[BS_BAD] || (w + 1 == W && tail != L)) { fatal = SQG_EINVAL; fatal_msg = "truncated or malformed BAM alignment record"; }
        else if (R + nrec_w >= 0x7fffff00ll) { fatal = SQG_EUNSUPPORTED; fatal_msg = "more than 2^31 records per context: shard the stream"; }
        if (fatal) { CK(cudaStreamSynchronize(st)); elapsed("bam_h2d"); elapsed("bam_inflate"); elapsed("bam_records"); carry = 0; continue; }
        // -- decode into the resident batch (capacity grows geometrically and keeps what earlier windows wrote)
        CK(cudaEventRecord(ctx->timers["bam_decode"].a, st));
        const size_t need = (size_t)(R + nrec_w) + 1, used = (size_t)R;
        CK(ctx->o_ref_id.grow(need, used, st)); CK(ctx->o_pos.grow(need, used, st)); CK(ctx->o_mate_ref_id.grow(need, used, st)); CK(ctx->o_mate_pos.grow(need, used, st));
        CK(ctx->o_end_pos.grow(need, used, st)); CK(ctx->o_flag.grow(need, used, st)); CK(ctx->o_total_len.grow(need, used, st)); CK(ctx->o_lowphred_run.grow(need, used, st));
        CK(ctx->o_mapq.grow(need, used, st)); CK(ctx->o_aux.grow(need, used, st)); CK(ctx->o_blk_off.grow(need + 1, used + 1, st));
        if (keep_lseq) CK(ctx->bam_lseq.grow(need, used, st));
        if (R == 0) CK(cudaMemsetAsync(ctx->o_blk_off.p, 0, 4, st));
        CK(ctx->bam_nblk.ensure((size_t)nrec_w + 1)); CK(ctx->bam_incl.ensure((size_t)nrec_w + 1));
        BamOut bo{ctx->o_ref_id.p, ctx->o_pos.p, ctx->o_mate_ref_id.p, ctx->o_mate_pos.p, ctx->o_end_pos.p, ctx->o_flag.p, ctx->o_total_len.p, ctx->o_lowphred_run.p,
                  ctx->o_mapq.p, ctx->o_aux.p, ctx->o_blk_off.p, nullptr, nullptr, nullptr, nullptr, keep_lseq ? ctx->bam_lseq.p : nullptr};
        uint64_t nblk_w = 0;
        if (nrec_w > 0) {
            LAUNCH_ON(st, k_bam_decode, blocks_for(nrec_w), kThreads, dwin, ctx->bam_recoff.p, nrec_w, R, prm, ns, bo, ctx->bam_nblk.p, ctx->bam_small.p);
            tb = 0;
            CK(cub::DeviceScan::InclusiveSum(nullptr, tb, ctx->bam_nblk.p, ctx->bam_incl.p, (int)nrec_w, st));
            { const int rc_ = ensure_temp(ctx, tb); if (rc_) return rc_; }
            CK(cub::DeviceScan::InclusiveSum(ctx->d_temp.p, tb, ctx->bam_nblk.p, ctx->bam_incl.p, (int)nrec_w, st));
            CK(cudaMemcpyAsync(&nblk_w, ctx->bam_incl.p + (nrec_w - 1), 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        if (B + nblk_w > 0xFFFFFFFFull) { fatal = SQG_EUNSUPPORTED; fatal_msg = "more than 2^32 - 1 aligned blocks in one batch: shard the stream"; }
        else if (nrec_w > 0) {
            const size_t bneed = (size_t)(B + nblk_w) + 1;
            CK(ctx->o_blk_ref_pos.grow(bneed, (size_t)B, st)); CK(ctx->o_blk_match_ref.grow(bneed, (size_t)B, st));
            CK(ctx->o_blk_read_pos.grow(bneed, (size_t)B, st)); CK(ctx->o_blk_match_read.grow(bneed, (size_t)B, st));
            bo.blk_ref_pos = ctx->o_blk_ref_pos.p; bo.blk_match_ref = ctx->o_blk_match_ref.p; bo.blk_read_pos = ctx->o_blk_read_pos.p; bo.blk_match_read = ctx->o_blk_match_read.p;
            LAUNCH_ON(st, k_bam_blocks, blocks_for(nrec_w), kThreads, dwin, ctx->bam_recoff.p, nrec_w, R, B, ctx->bam_incl.p, ctx->bam_nblk.p, bo);
        }
        CK(cudaEventRecord(ctx->timers["bam_decode"].b, st));
        CK(cudaStreamSynchronize(st));
        elapsed("bam_h2d"); elapsed("bam_inflate"); elapsed("bam_records"); elapsed("bam_decode");
        R += nrec_w; B += nblk_w;
        carry = L - tail;
        ctx->bam_win_len = L;
        cur ^= 1;
    }
    CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    aux_bad = ctx->bam_hsmall.p[BS_AUXBAD] != 0;
    for (const char *nm : {"bam_h2d", "bam_inflate", "bam_records", "bam_decode"}) ctx->timers[nm].done = false;
    lap("bam: windows");
    // the host front end's order: inflate, header, record boundaries, aux fields, then the packer's own refusals
    if (infl_bits) FAIL(SQG_EINVAL, (infl_bits & 1) ? "corrupt deflate stream in a BGZF block" : "BGZF block fails its CRC32");
    if (fatal == SQG_EINVAL) FAIL(fatal, fatal_msg);
    if (aux_bad) FAIL(SQG_EINVAL, "malformed BAM alignment record");
    const uint64_t key = (uint64_t)ctx->bam_hsmall.p[BS_ERRKEY];
    if (key != ~0ull) {
        FAIL(SQG_EUNSUPPORTED, sqh::packer_refusal(key >> 33, (int)(key >> 32 & 1) + 1, (uint32_t)key));
    }
    if (fatal) FAIL(fatal, fatal_msg);
    if (R == 0) {  // an empty batch still has its blk_off[0]
        CK(ctx->o_blk_off.grow(1, 0, st));
        CK(cudaMemsetAsync(ctx->o_blk_off.p, 0, 4, st));
    }
    if (keep_lseq && R > 0 && ctx->bam_hsmall.p[BS_SEQ] == 0) LAUNCH_ON(st, k_bam_null_qual, blocks_for(R), kThreads, ctx->o_lowphred_run.p, ctx->bam_lseq.p, R);
    for (auto *b : {&ctx->o_ref_id, &ctx->o_pos, &ctx->o_mate_ref_id, &ctx->o_mate_pos, &ctx->o_end_pos, &ctx->o_blk_ref_pos, &ctx->o_blk_match_ref}) CK(b->grow(1, 0, st));
    for (auto *b : {&ctx->o_flag, &ctx->o_total_len, &ctx->o_lowphred_run, &ctx->o_blk_read_pos, &ctx->o_blk_match_read}) CK(b->grow(1, 0, st));
    CK(ctx->o_mapq.grow(1, 0, st)); CK(ctx->o_aux.grow(1, 0, st));
    point_batch_at_own_arrays(ctx, R, (int64_t)B);
    reset_batch_state(ctx, true, first_record_index, false);
    return SQG_OK;
}

extern "C" int sqg_load_concordant_bam(sqg_ctx *ctx, const char *path, const sqg_bam_decode *opt, int64_t first_record_index) {
    if (!ctx || !path || !opt || opt->n_names < 0 || (opt->n_names > 0 && (!opt->names || !opt->name_off))) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    ctx->have_batch = false;  // the resident arrays are rewritten from here on: a refused load leaves no batch
    ctx->acc_ms.clear();
    const int rc = bam_load(ctx, path, opt, first_record_index);
    if (rc == SQG_ECUDA) cudaGetLastError();
    return rc;
}
