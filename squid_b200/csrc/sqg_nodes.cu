// BuildNode_STAR: the seed machine over the discordant groups, the genome tiling into the segment table and its position index,
// and the range-shard entry points of that stage.
#include <cub/cub.cuh>

#include <algorithm>
#include <vector>

#include "sq_seed.cuh"
#include "sqg_ctx.cuh"

using namespace sq;

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
// entry i of the position index (sq_common.cuh: seg_at); bin_off: n_ref + 1
__global__ void k_build_bins(NodeTable nt, const int32_t *bin_off, BinEnt *bins, int32_t n_bins) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bins) return;
    int32_t lo = 0, hi = nt.n_ref;  // chromosome of bin i: last c with bin_off[c] <= i
    while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (bin_off[m + 1] <= i) lo = m + 1; else hi = m; }
    bins[i] = bin_ent_value(nt, lo, i - bin_off[lo], bin_off[lo + 1] - bin_off[lo]);
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
    CK(ctx->d_nchr.ensure(N + 1)); CK(ctx->d_npos.ensure(N + 1)); CK(ctx->d_nend.ensure(N + 1)); CK(ctx->d_chr_head.ensure(n_ref + 1));
    if (N) {
        CK(cudaMemcpyAsync(ctx->d_nchr.p, ctx->h_nchr.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_npos.p, ctx->h_npos.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_nend.p, ctx->h_nend.data(), N * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    ctx->nt.n = N; ctx->nt.n_ref = n_ref; ctx->nt.chr = ctx->d_nchr.p; ctx->nt.pos = ctx->d_npos.p; ctx->nt.end = ctx->d_nend.p;
    {   // position index over the tiling (sq_common.cuh: seg_at): per-chromosome headers and 16-byte bin entries
        int64_t total = 0;
        for (int32_t c = 0; c < n_ref; c++) total += ctx->ref_len[c] > 0 ? ctx->ref_len[c] : 0;
        int32_t sh = 9;  // 512-bp bins: reads pile up exactly where segments are dense (fusion genes), so the bins must be fine
        while ((total >> sh) > (16ll << 20)) sh++;  // at most ~16M bins (256 MB; only the bins the reads touch are hot in L2)
        ctx->h_bin_off.assign(n_ref + 1, 0);
        for (int32_t c = 0; c < n_ref; c++) ctx->h_bin_off[c + 1] = ctx->h_bin_off[c] + ((ctx->ref_len[c] > 0 ? ctx->ref_len[c] : 0) >> sh) + 1;
        const int32_t n_bins = ctx->h_bin_off[n_ref];
        ctx->h_head.resize(n_ref);
        for (int32_t c = 0; c < n_ref; c++) ctx->h_head[c] = chr_head_value(ctx->h_chr_first.data(), ctx->h_nend.data(), ctx->h_bin_off.data(), c);
        CK(ctx->d_bin_off.ensure(n_ref + 2)); CK(ctx->d_bins.ensure(n_bins + 1));
        CK(cudaMemcpyAsync(ctx->d_bin_off.p, ctx->h_bin_off.data(), (n_ref + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (n_ref) CK(cudaMemcpyAsync(ctx->d_chr_head.p, ctx->h_head.data(), n_ref * sizeof(ChrHead), cudaMemcpyHostToDevice, ctx->stream));
        ctx->nt.head = ctx->d_chr_head.p; ctx->nt.bin_shift = sh; ctx->nt.bins = nullptr;
        LAUNCH(k_build_bins, blocks_for(n_bins), kThreads, ctx->nt, ctx->d_bin_off.p, ctx->d_bins.p, n_bins);
        ctx->nt.bins = ctx->d_bins.p;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_nodes = true; ctx->have_edge_table = false;
    return SQG_OK;
}

extern "C" int sqg_set_nodes(sqg_ctx *ctx, const int32_t *chr, const int32_t *pos, const int32_t *len, int64_t n_nodes) {
    if (!ctx || !chr || !pos || !len || n_nodes <= 0 || n_nodes > 0x7ffffff0ll) return SQG_EINVAL;
    // the table must tile every chromosome from 0 to its length with segments of positive length: the position index (seg_at)
    // and the closed-form LocateRead index a chromosome's segments as [head[c].c0, head[c].c1) and take a position below
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
    Counters *dc = ctx->cnt.d.p;
    const Counters &hc = *ctx->cnt.h.p;
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
        CK(ctx->cnt.zero(ctx->stream, &dc->n_rest));
        if (n > 0) LAUNCH(k_rest_collect, blocks_for((n + 3) / 4), kThreads, b, ctx->d_cls.p, ctx->d_groups.p, ctx->d_disc.p, nG, ctx->params.read_len, rbins, ctx->d_reflen.p,
                          ctx->d_rest.p, ctx->d_restkey.p, rest_cap, &dc->n_rest);
        CK(ctx->cnt.to_host(ctx->stream, &dc->n_rest));
        CK(cudaStreamSynchronize(ctx->stream));
        n_rest = hc.n_rest;
        lap("  seed: triggers + rest collect");
        if (n_rest <= rest_cap) break;
        rest_cap = n_rest + 1024;
    }
    if (n_rest > 0) {
        int key_bits = 1;  // the owning group: the table is binned by group, not ordered inside a group
        while (key_bits < 32 && (1ll << key_bits) < (long long)nG) key_bits++;
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortPairs(t, tb, ctx->d_restkey.p, ctx->d_restkey2.p, ctx->d_rest.p, ctx->d_rest2.p, (int)n_rest, 0, key_bits, ctx->stream); }));
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
    CK(ctx->cnt.zero(ctx->stream, &dc->n_isl));
    if (g_hi - g_lo > 0) {
        cub::CountingInputIterator<int32_t> cnt(g_lo);
        IsCutOp op{ctx->d_cutflag.p};
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceSelect::If(t, tb, cnt, ctx->d_isl.p, &dc->n_isl, g_hi - g_lo, op, ctx->stream); }));
        ctx->launches += 2;
    }
    CK(ctx->cnt.to_host(ctx->stream, &dc->n_isl));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t n_isl = hc.n_isl;
    lap("  seed: island cuts");
    CK(ctx->d_cap_ops.ensure(2 * (size_t)n_isl + 4)); CK(ctx->d_cap_mar.ensure(n_isl + 2)); CK(ctx->d_off_ops.ensure(n_isl + 2)); CK(ctx->d_off_mar.ensure(n_isl + 2));
    CK(ctx->d_isl_nout.ensure(n_isl + 1)); CK(ctx->d_isl_gdone.ensure(n_isl + 1));
    CK(cudaMemsetAsync(ctx->d_cap_ops.p, 0, (n_isl + 2) * 4, ctx->stream)); CK(cudaMemsetAsync(ctx->d_cap_mar.p, 0, (n_isl + 2) * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_isl_nout.p, 0, (n_isl + 1) * 4, ctx->stream));
    CK(ctx->d_span.ensure(n_isl + 2)); CK(ctx->d_heavy.ensure(n_isl + 2)); CK(ctx->d_light.ensure(n_isl + 2));
    LAUNCH(k_island_caps, blocks_for(n_isl, 64), 64, in, ctx->d_isl.p, n_isl, ctx->d_cap_ops.p, ctx->d_cap_mar.p, ctx->d_span.p);
    CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, ctx->d_cap_ops.p, ctx->d_off_ops.p, n_isl + 1, ctx->stream); }));
    CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, ctx->d_cap_mar.p, ctx->d_off_mar.p, n_isl + 1, ctx->stream); }));
    ctx->launches += 4;
    int64_t tot[2];
    CK(cudaMemcpyAsync(&tot[0], ctx->d_off_ops.p + n_isl, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&tot[1], ctx->d_off_mar.p + n_isl, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    lap("  seed: island caps + offsets");
    CK(ctx->d_ops.ensure(tot[0] + 1)); CK(ctx->d_margin.ensure(tot[1] + 1));
    int32_t *d_err = &dc->seed_err, *d_nprefix = &dc->n_prefix;
    CK(ctx->cnt.zero(ctx->stream, &dc->n_prefix, &dc->win_count));
    in.win_count = &dc->win_count;
    // (a shard that follows one with an emitted segment starts with an inherited last segment: no sequential prefix)
    if (!(ctx->shard_index > 0 && ctx->shard_prior_emission) && n_isl > 0)
        LAUNCH(k_seed_prefix, 1, kSeedBlock, in, ctx->d_isl.p, n_isl, ctx->d_off_ops.p, ctx->d_off_mar.p, ctx->d_ops.p, ctx->d_margin.p,
               ctx->d_isl_nout.p, ctx->d_isl_gdone.p, d_err, d_nprefix);
    CK(ctx->cnt.zero(ctx->stream, &dc->n_heavy_light));
    if (n_isl > 0) {
        cub::CountingInputIterator<int32_t> cnt(0);
        IsHeavyOp oh{ctx->d_span.p, d_nprefix, true}, ol{ctx->d_span.p, d_nprefix, false};
        int32_t *d_nh = dc->n_heavy_light;
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceSelect::If(t, tb, cnt, ctx->d_heavy.p, d_nh, n_isl, oh, ctx->stream); }));
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceSelect::If(t, tb, cnt, ctx->d_light.p, d_nh + 1, n_isl, ol, ctx->stream); }));
        ctx->launches += 3;
    }
    CK(ctx->cnt.to_host(ctx->stream, &dc->n_heavy_light));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t n_heavy = hc.n_heavy_light[0], n_light = hc.n_heavy_light[1];
    ctx->n_heavy = n_heavy;
    lap("  seed: prefix + heavy/light split");
    if (n_heavy > 1) {  // longest islands first: the kernel's critical path is its largest island
        // d_cap_ops is free again after the offset scans: sort scratch [keys | keys2]
        int32_t *k1 = ctx->d_cap_ops.p, *k2 = ctx->d_cap_ops.p + n_heavy;
        LAUNCH(k_gather_i32, blocks_for(n_heavy), kThreads, ctx->d_span.p, ctx->d_heavy.p, n_heavy, k1);
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceRadixSort::SortPairsDescending(t, tb, k1, k2, ctx->d_heavy.p, ctx->d_light.p + n_light, n_heavy, 0, 32, ctx->stream); }));
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
    LAUNCH(k_ops_dense, 1, 1024, ctx->d_isl.p, n_isl, g_hi, ctx->d_isl_nout.p, ctx->d_isl_gdone.p, ctx->d_off_ops.p, ctx->d_ops.p, ctx->d_ops_dense.p, dc->ops_dense);
    CK(ctx->cnt.to_host(ctx->stream, &dc->ops_dense, &dc->win_count));
    std::vector<int64_t> trig_last(1, n);
    if (nG > 0) CK(cudaMemcpyAsync(trig_last.data(), ctx->d_trigger.p + (nG - 1), sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int32_t serr = hc.seed_err;
    if (serr) FAIL(SQG_ENOMEM, serr == 1 ? "seed machine: margin scratch overflow" : "seed machine: output overflow");
    const int64_t n_ops_dense = hc.ops_dense[0];
    const int32_t g_done = (int32_t)hc.ops_dense[1];  // (== nG exactly when every group was triggered by this batch)
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
