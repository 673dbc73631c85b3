// Phase 2 of the path in ONE pass over the record batch, once the segment table exists: per-segment depth of the
// concordant stream (BuildNode_STAR part D, SegmentGraph.cpp:784-825) and read-to-segment assignment + raw edges of the
// stream (RawEdgesOther, :1557-1696).  Tiles are staged with TMA bulk copies (sq_stream.cuh) and are independent.
//   * Segment lookups go through the position index of the segment table (seg_at): one table read and a step or two.
//   * Records with at most one aligned block (nine in ten) take a register-only path (read_edges_single); the others
//     are collected per tile and run the generic read_edges densely packed, so a warp never drags 31 idle lanes through it.
//   * Edges are not written one by one: every tile counts them in a small shared-memory hash table (keys repeat massively
//     in sorted input) and flushes (key, count) pairs; the sort + reduce that follows sees ~1 % of the raw volume.
//   * Depth: ReadsOther blocks are counted directly; ReadsMain needs the forward-only segment cursor = running maximum
//     of the per-read target.  The tile counts with its LOCAL running maximum and records (first target, maximum);
//     k_depth_fix corrects the few tiles whose incoming cursor was ahead of their first target.
#ifndef SQ_PHASE2_CUH
#define SQ_PHASE2_CUH
#include "sq_depth_cover.cuh"
#include "sq_locate.cuh"
#include "sq_phase1.cuh"
#include "sq_stream.cuh"

namespace sq {

struct PairSink {  // raw (edge key, weight) pairs
    uint64_t *keys; int32_t *w; int64_t cap; unsigned long long *counter;
    __device__ __forceinline__ void add(uint64_t k, int32_t weight) {
        const unsigned long long slot = atomicAdd(counter, 1ull);
        if ((int64_t)slot < cap) { keys[slot] = k; w[slot] = weight; }
    }
    __device__ __forceinline__ void operator()(uint64_t k) { add(k, 1); }
};

constexpr int kEdgeSlots = 256;      // shared-memory edge table of a tile
constexpr int kDepthWin = 64;        // segments [base, base + 64) of a tile are counted in shared memory
constexpr uint64_t kEmptyKey = ~0ull;

struct TileEdgeTable {
    unsigned long long keys[kEdgeSlots];
    int32_t cnt[kEdgeSlots];
    PairSink spill;
    __device__ __forceinline__ void operator()(uint64_t k) {
        uint32_t h = (uint32_t)((k * 0x9E3779B97F4A7C15ull) >> 56);
#pragma unroll 1
        for (int probe = 0; probe < 8; probe++, h = (h + 1) & (kEdgeSlots - 1)) {
            const unsigned long long old = atomicCAS(&keys[h], (unsigned long long)kEmptyKey, (unsigned long long)k);
            if (old == kEmptyKey || old == k) { atomicAdd(&cnt[h], 1); return; }
        }
        spill.add(k, 1);
    }
};

struct DepthTile {  // per tile, for k_depth_fix
    int32_t first_target;  // target of the first counted read of the tile (INT32_MAX if none)
    int32_t max_target;    // maximum target of the tile (-1 if none); after k_depth_scan: the cursor before the tile
};
struct P2Args {
    const uint8_t *cls;
    NodeTable nt;
    Params p;
    int64_t r_break;
    int32_t do_depth, do_edges;
    int32_t *cnt_main, *sum_main, *cnt_other, *sum_other, *other_nonempty;
    DepthTile *dtile;
    int32_t *res0;
    PairSink sink;
    int32_t *sens; int32_t *n_sens; int32_t sens_cap;
    const BatchDesc *desc; const NodeTable *nt_dev;  // device copies for the out-of-line generic path
    unsigned long long *path_counts;  // [0] records through read_edges_single, [1] through the generic read_edges (statistics)
    int32_t *slow_list; int32_t *n_slow; int32_t slow_cap;  // records left to k_edges_generic
    // ReadsOther blocks of <= 3 bp (sq_depth_cover.cuh): per-segment start masks, the deferred short blocks (chr, start, len, node)
    uint32_t *omask; int4 *shorts; int32_t *n_short; int32_t short_cap;
};

constexpr uint32_t kP2Fields = F_REF | F_MREF | F_MPOS | F_FLAG | F_TLEN | F_LOWQ | F_CLS | F_BLOCKS;

// one shared-memory counter pair per segment of the window, else global; leaders of equal-key groups add for the group
__device__ __forceinline__ void depth_add(int32_t seg, int32_t len, bool on, int32_t base, int32_t *s_cnt, int32_t *s_sum, int32_t *g_cnt, int32_t *g_sum) {
    const unsigned act = __ballot_sync(0xffffffffu, on);
    if (!on) return;
    const unsigned m = __match_any_sync(act, seg);
    const int32_t tot = __reduce_add_sync(m, len);
    if ((int)(threadIdx.x & 31) == __ffs(m) - 1) {
        const uint32_t w = (uint32_t)(seg - base);
        if (w < (uint32_t)kDepthWin) { atomicAdd(&s_cnt[w], __popc(m)); atomicAdd(&s_sum[w], tot); }
        else { atomicAdd(&g_cnt[seg], __popc(m)); atomicAdd(&g_sum[seg], tot); }
    }
}

// RawEdgesOther for a record with several aligned blocks: the generic rules, read straight from HBM (the tile's bytes are
// still in L2) and kept out of line so that the hot single-block path stays small.  Returns the res0 code.
// (the block lists live in local memory, sized by the record's own block count -- three in all but a handful of records -- so
// they stay in L1 instead of striding through a 1 KB frame per thread.  A register-only variant -- both lists in one array of
// compile-time size, every loop unrolled and guarded by the list lengths -- was written, verified and measured: 96 registers per
// thread, 20 instead of 28 resident warps per SM, 10.7 ms against 6.8 ms at 100 M pairs.  This kernel lives on occupancy.)
template <int MAXB>
__device__ __forceinline__ int32_t conc_edges_sized(const DevBatch &b, const Params &p, const NodeTable &nt, int64_t r, TileEdgeTable *edges) {
    Blk F[MAXB + 1], S[MAXB + 1];
    int32_t node[2 * MAXB + 2];
    ReadView rv; rv.F = F; rv.S = S;
    bool is_first;
    conc_load_read(b, r, rv, is_first);
    if (rv.nF + rv.nS == 0) return -2;
    return read_edges(nt, p, rv, MODE_OTHER, is_first, false, 0, node, *edges) ? node[0] : -3;
}
__device__ __noinline__ int32_t conc_edges_generic(const BatchDesc *desc, const NodeTable *ntp, int64_t r, TileEdgeTable *edges) {
    const DevBatch &b = desc->b;
    const Params &p = desc->p;
    const NodeTable nt = *ntp;
    if (!conc_builds_edges(b, p, r)) return -2;
    const uint32_t nb = b.blk_off[r + 1] - b.blk_off[r];
    if (nb <= 3) return conc_edges_sized<3>(b, p, nt, r, edges);
    return conc_edges_sized<kMaxBlocks>(b, p, nt, r, edges);
}

// ReadsOther, the two rare cases (sq_depth_cover.cuh): an entry that starts d <= 2 bp right of the start of its segment m2 goes
// into that segment's start mask; a block of <= 3 bp is not counted here but deferred to the second pass.  Out of line.
__device__ __noinline__ bool depth_other_rare(uint32_t *omask, int4 *shorts, int32_t *n_short, int32_t short_cap, int32_t rid, int32_t st, int32_t l, int32_t m2, int32_t d, bool on) {
    if (l > kSeedThresh) {
        // (every read spliced into an exon that opens a segment lands here with the same bit: look before the atomic)
        if (m2 != kNoNode && !(__ldcg(&omask[m2]) & (1u << d))) atomicOr(&omask[m2], 1u << d);
        return on;
    }
    if (m2 != kNoNode && (uint32_t)d <= 2u) { const uint32_t bit = 1u << (3 + 3 * d + ((l < 1 ? 1 : l) - 1)); if (!(__ldcg(&omask[m2]) & bit)) atomicOr(&omask[m2], bit); }
    const int32_t q = atomicAdd(n_short, 1);
    if (q < short_cap) shorts[q] = make_int4(rid, st, l, kNoNode);
    return false;
}

template <bool DO_DEPTH, bool DO_EDGES>
__global__ void __launch_bounds__(kTileThreads, 7) k_assign_tiles(DevBatch b, P2Args a, int bulk_ok) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    TileStage &s = *reinterpret_cast<TileStage *>(smem_raw);
    __shared__ TileEdgeTable s_edges;
    __shared__ int32_t s_dcnt[2][kDepthWin], s_dsum[2][kDepthWin];
    __shared__ uint16_t s_slow[kTile], s_mid[kTile];
    __shared__ int32_t s_cmax[kTileChunks];
    __shared__ int32_t s_nslow, s_nmid, s_base, s_other, s_first, s_seg[4];
    int32_t *s_m = s.end_pos;   // per record: depth target of its first block (-1: not counted)
    uint8_t *s_cont = s.mapq;   // per record: first block contained in that target
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned full = 0xffffffffu;
    const int64_t tile = blockIdx.x;
    const StageTicket tk = stage_issue<kP2Fields>(s, b, a.cls, tile, bulk_ok != 0);
    const TileInfo ti = tk.ti;
    const int n = ti.n;
    const int64_t rec0 = ti.rec0;
    for (int i = tid; i < kEdgeSlots; i += kTileThreads) { s_edges.keys[i] = kEmptyKey; s_edges.cnt[i] = 0; }
    for (int i = tid; i < 2 * kDepthWin; i += kTileThreads) { (&s_dcnt[0][0])[i] = 0; (&s_dsum[0][0])[i] = 0; }
    if (tid == 0) { s_edges.spill = a.sink; s_nslow = 0; s_nmid = 0; s_other = 0; s_first = 0x7fffffff; s_base = -(1 << 30); }
    stage_wait<kP2Fields>(s, b, a.cls, tk);
    const bool staged = ti.nb >= 0;
    const TileBatch tb = tile_view(s, ti, b);
    if (tid == 0) {
        // The segment that holds the tile's first block: sorted input keeps most of the tile (usually all of it) inside this
        // one segment, so it is looked up once and every block of the tile is first tested against it.  The window of
        // segments counted in shared memory starts one segment to its left.
        s_seg[0] = -1; s_seg[1] = 0; s_seg[2] = 0; s_seg[3] = 0;
        for (int i = 0; i < n; i++) {
            const uint32_t o0 = s.blk_off[i];
            if (s.blk_off[i + 1] > o0 && s.ref_id[i] >= 0 && s.ref_id[i] < a.nt.n_ref) {
                const int32_t c = s.ref_id[i], c0 = a.nt.chr_first[c], c1 = a.nt.chr_first[c + 1];
                const int32_t st = staged ? tb.blk_ref_pos[o0] : b.blk_ref_pos[o0];
                if (c1 > c0) {
                    const int32_t sg = seg_at(a.nt, c, c0, c1, st);
                    s_base = sg - 1;
                    s_seg[0] = c; s_seg[1] = sg; s_seg[2] = a.nt.pos[sg]; s_seg[3] = a.nt.end[sg];
                }
                break;
            }
        }
    }
    __syncthreads();
    const int32_t base = s_base;
    const int32_t wc = s_seg[0], ws = s_seg[1], wq = s_seg[2], we = s_seg[3];  // wc == -1: no such segment
    const NodeTable &nt = a.nt;

    // ---- pass A: depth targets + ReadsOther; edges of the single-block records ------------------------------------
#pragma unroll 1
    for (int j = 0; j < kTileRPT; j++) {
        const int i = j * kTileThreads + tid;
        const int64_t r = rec0 + i;
        const bool in = i < n;
        const uint8_t c8 = in ? s.cls[i] : (uint8_t)0;
        const uint32_t o0 = in ? s.blk_off[i] : 0u, nb = in ? s.blk_off[i + 1] - o0 : 0u;
        const int32_t rid = in ? s.ref_id[i] : -1;
        // depth
        int32_t m = -1;
        if (DO_DEPTH) {
            const bool counted = in && r < a.r_break && (c8 & CLS_HASBLK);
            int32_t st0 = 0, l0 = 0;
            bool cont = false;
            if (counted) {
                st0 = staged ? tb.blk_ref_pos[o0] : b.blk_ref_pos[o0]; l0 = staged ? tb.blk_match_ref[o0] : b.blk_match_ref[o0];
                if (rid == wc && wq <= st0 && st0 < we && l0 > kSeedThresh) { m = ws; cont = st0 + l0 <= we + kSeedThresh; }  // depth_target / depth_contained in the tile's segment
                else { m = depth_target(nt, rid, st0, l0); cont = m != kNoNode && depth_contained(nt, m, rid, st0, l0); }
                if (nb > 1) s_other = 1;
            }
            const uint32_t nb_max = __reduce_max_sync(full, counted ? nb : 0u);
            for (uint32_t k = 1; k < nb_max; k++) {  // ReadsOther: every block is counted in its own target segment
                bool on = false;
                int32_t m2 = 0, l = 0;
                if (counted && k < nb) {
                    const int32_t st = staged ? tb.blk_ref_pos[o0 + k] : b.blk_ref_pos[o0 + k];
                    l = staged ? tb.blk_match_ref[o0 + k] : b.blk_match_ref[o0 + k];
                    int32_t pj;
                    if (rid == wc && wq <= st && st < we) { m2 = ws; pj = wq; on = st + l <= we + kSeedThresh; }  // the tile's segment
                    else {
                        m2 = depth_target(nt, rid, st, kSeedThresh + 1);  // first segment ending right of the start
                        pj = st - 100;
                        if (m2 != kNoNode) { pj = nt.pos[m2]; on = nt.chr[m2] == rid && st >= pj - kSeedThresh && st + l <= nt.end[m2] + kSeedThresh; }
                    }
                    // rare: a block of <= 3 bp (deferred), or one that starts within 2 bp of its segment's start (start mask)
                    if (l <= kSeedThresh || (uint32_t)(st - pj) <= 2u) on = depth_other_rare(a.omask, a.shorts, a.n_short, a.short_cap, rid, st, l, m2, st - pj, on);
                }
                depth_add(m2, l, on, base, s_dcnt[1], s_dsum[1], a.cnt_other, a.sum_other);
            }
            if (in) {
                s_m[i] = m;
                // is the block contained (+-3) in its own target?  (pass B only looks again when the cursor is elsewhere)
                s_cont[i] = cont ? 1 : 0;
            }
            const int32_t cm = __reduce_max_sync(full, m);
            const unsigned vm = __ballot_sync(full, m >= 0);
            if (lane == 0) {
                s_cmax[j * kWarpsPerTile + warp] = cm;
                if (vm) atomicMin(&s_first, (j * kWarpsPerTile + warp) * 32 + __ffs(vm) - 1);
            }
        }
        // edges
        if (DO_EDGES) {
            int32_t out = -2;
            if (in && (c8 & CLS_KEEP)) {
                if (nb <= 1 && staged) {
                    const uint16_t f = s.flag[i];
                    const bool has_mate = has_mate_block(f, s.mate_ref_id[i]);
                    bool builds = true;
                    Blk own;
                    own.ref_id = rid; own.rev = flag_rev(f); own.ref_pos = 0; own.match_ref = 0; own.read_pos = 0; own.match_read = 0;
                    if (nb == 1) {
                        own.ref_pos = tb.blk_ref_pos[o0]; own.match_ref = tb.blk_match_ref[o0]; own.read_pos = tb.blk_read_pos[o0]; own.match_read = tb.blk_match_read[o0];
                        if (has_mate) builds = own.read_pos <= 15 || (int32_t)s.lowphred_run[i] > a.p.max_lowphred_len;
                    }
                    // both blocks well inside the tile's segment: each locates there whatever the scan order, nothing to emit
                    const bool own_in = nb == 0 || (rid == wc && own.match_ref > kLocateTol && wq <= own.ref_pos && own.ref_pos + kLocateTol < we && own.ref_pos + own.match_ref - kLocateTol <= we);
                    const bool mate_in = !has_mate || (s.mate_ref_id[i] == wc && wq <= s.mate_pos[i] && s.mate_pos[i] + kLocateTol < we && s.mate_pos[i] + kMateBlockLen - kLocateTol <= we);
                    if (builds && (nb == 1 || has_mate) && own_in && mate_in) out = ws;
                    else if (builds && (nb == 1 || has_mate)) { out = -4; s_mid[atomicAdd(&s_nmid, 1)] = (uint16_t)i; }  // pass B1
                } else if (staged && rid == wc) {
                    // several blocks: if every one of them (and the mate block) lies well inside the tile's segment, each locates
                    // there -- the first by the closed form, the others because they fit the cursor -- and no rule emits anything
                    const uint16_t f = s.flag[i];
                    const bool has_mate = has_mate_block(f, s.mate_ref_id[i]);
                    bool all_in = !has_mate || (s.mate_ref_id[i] == wc && wq <= s.mate_pos[i] && s.mate_pos[i] + kLocateTol < we && s.mate_pos[i] + kMateBlockLen - kLocateTol <= we);
                    int32_t front_rp = 0x7fffffff;
                    for (uint32_t k = 0; k < nb; k++) {
                        const int32_t p0 = tb.blk_ref_pos[o0 + k], m0 = tb.blk_match_ref[o0 + k], rp = tb.blk_read_pos[o0 + k];
                        all_in = all_in && m0 > kLocateTol && wq <= p0 && p0 + kLocateTol < we && p0 + m0 - kLocateTol <= we;
                        if (rp < front_rp) front_rp = rp;
                    }
                    const bool builds = !has_mate || front_rp <= 15 || (int32_t)s.lowphred_run[i] > a.p.max_lowphred_len;  // :1601-1605
                    if (!builds) out = -2;
                    else if (all_in) out = ws;
                    else { out = -4; s_slow[atomicAdd(&s_nslow, 1)] = (uint16_t)i; }
                } else {
                    out = -4;  // generic path below
                    s_slow[atomicAdd(&s_nslow, 1)] = (uint16_t)i;
                }
            }
            if (in) {
                // (-4 = deferred to pass B1 / B2 / k_edges_generic, which overwrite it.  Written here all the same: when the deferred
                // list overflows, the records past its capacity are never processed in this attempt, and the hint fix-up, which
                // runs before the host notices and repeats the pass, must not find stale values of an earlier batch in their place)
                a.res0[r] = out;
                if (out == -3) { const int32_t q = atomicAdd(a.n_sens, 1); if (q < a.sens_cap) a.sens[q] = (int32_t)r; }
            }
        }
    }
    __syncthreads();
    // ---- pass B1: single-block records that left the tile's segment, densely packed ---------------------------------
    if (DO_EDGES) {
        const int nm = s_nmid;
#pragma unroll 1
        for (int q = tid; q < nm; q += kTileThreads) {
            const int i = s_mid[q];
            const int64_t r = rec0 + i;
            const uint16_t f = s.flag[i];
            const uint32_t o0 = s.blk_off[i], nb = s.blk_off[i + 1] - o0;
            Blk own;
            own.ref_id = s.ref_id[i]; own.rev = flag_rev(f); own.ref_pos = 0; own.match_ref = 0; own.read_pos = 0; own.match_read = 0;
            if (nb == 1) { own.ref_pos = tb.blk_ref_pos[o0]; own.match_ref = tb.blk_match_ref[o0]; own.read_pos = tb.blk_read_pos[o0]; own.match_read = tb.blk_match_read[o0]; }
            const int32_t out = read_edges_single(nt, a.p, nb == 1, own, has_mate_block(f, s.mate_ref_id[i]), mate_block_of(f, s.mate_ref_id[i], s.mate_pos[i]), flag_first(f),
                                                  (int32_t)s.total_len[i], s_edges);
            a.res0[r] = out;
            if (out == -3) { const int32_t k = atomicAdd(a.n_sens, 1); if (k < a.sens_cap) a.sens[k] = (int32_t)r; }
        }
    }
    // ---- the multi-block records that left the tile's segment ----------------------------------------------------------------
    // They go to k_edges_generic's list.  (Measured and dropped: processing them right here with the generic rules, from the
    // staged tile -- slower, see sqg_api.cu.  Also measured and dropped: a register-only rule set for the plain ones among them --
    // every block well inside one segment, nine in ten -- run here as a "pass B2": 43 M of the 53 M records of the benchmark leave
    // the list, k_edges_generic 5.4 -> 1.5 ms, this kernel 5.5 -> 9.3 ms: the same cost per record either way.)
    if (DO_EDGES) {
        __shared__ int32_t s_slow_base;
        const int ns = s_nslow;
        if (tid == 0 && ns > 0) s_slow_base = atomicAdd(a.n_slow, ns);
        __syncthreads();
        if (ns > 0) {
            const int32_t base_q = s_slow_base;
            for (int q = tid; q < ns; q += kTileThreads)
                if (base_q + q < a.slow_cap) a.slow_list[base_q + q] = (int32_t)(rec0 + s_slow[q]);
        }
    }
    // ---- ReadsMain with the tile-local cursor -----------------------------------------------------------------------
    if (DO_DEPTH) {
        if (warp == 0) {
            int32_t inc = lane < kTileChunks ? s_cmax[lane] : -1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, inc, d); if (lane >= d && u > inc) inc = u; }
            const int32_t tot = __shfl_sync(full, inc, 31);
            int32_t exc = __shfl_up_sync(full, inc, 1);
            if (lane == 0) exc = -1;
            if (lane < kTileChunks) s_cmax[lane] = exc;
            if (lane == 0) {
                DepthTile d; d.max_target = tot; d.first_target = s_first < kTile ? s_m[s_first] : 0x7fffffff;
                a.dtile[tile] = d;
                if (s_other) *a.other_nonempty = 1;
            }
        }
        __syncthreads();
#pragma unroll 1
        for (int j = 0; j < kTileRPT; j++) {
            const int i = j * kTileThreads + tid;
            const int32_t m = i < n ? s_m[i] : -1;
            int32_t v = m;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, v, d); if (lane >= d && u > v) v = u; }
            const int32_t e = s_cmax[j * kWarpsPerTile + warp];
            if (e > v) v = e;  // cursor at this read: running maximum of the targets so far in the tile
            bool on = false;
            int32_t l0 = 0;
            if (m >= 0 && v != kNoNode && v < nt.n) {
                const uint32_t o0 = s.blk_off[i];
                l0 = staged ? tb.blk_match_ref[o0] : b.blk_match_ref[o0];
                if (v == m) on = s_cont[i] != 0;
                else on = depth_contained(nt, v, s.ref_id[i], staged ? tb.blk_ref_pos[o0] : b.blk_ref_pos[o0], l0);
            }
            depth_add(v, l0, on, base, s_dcnt[0], s_dsum[0], a.cnt_main, a.sum_main);
        }
    }
    __syncthreads();
    // ---- flush the tile's tables --------------------------------------------------------------------------------------
    if (DO_DEPTH) {
        for (int w = tid; w < kDepthWin; w += kTileThreads) {
            const int32_t seg = base + w;
            if (s_dcnt[0][w]) { atomicAdd(&a.cnt_main[seg], s_dcnt[0][w]); atomicAdd(&a.sum_main[seg], s_dsum[0][w]); }
            if (s_dcnt[1][w]) { atomicAdd(&a.cnt_other[seg], s_dcnt[1][w]); atomicAdd(&a.sum_other[seg], s_dsum[1][w]); }
        }
    }
    if (DO_EDGES && tid == 0 && a.path_counts) { atomicAdd(a.path_counts, (unsigned long long)s_nmid); atomicAdd(a.path_counts + 1, (unsigned long long)s_nslow); }
    if (DO_EDGES) {  // one reservation in the raw pair list per tile
        int mine = 0;
        for (int h = tid; h < kEdgeSlots; h += kTileThreads) mine += s_edges.cnt[h] != 0;
        int inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(full, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) s_cmax[warp] = inc;
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < kWarpsPerTile; w++) { const int c = s_cmax[w]; s_cmax[w] = tot; tot += c; }
            s_nslow = tot;
            if (tot > 0) { const unsigned long long at = atomicAdd(a.sink.counter, (unsigned long long)tot); s_cmax[kWarpsPerTile] = (int32_t)(at & 0x7fffffffu); s_cmax[kWarpsPerTile + 1] = (int32_t)(at >> 31); }
        }
        __syncthreads();
        if (s_nslow > 0) {
            long long at = ((long long)s_cmax[kWarpsPerTile + 1] << 31) + s_cmax[kWarpsPerTile] + s_cmax[warp] + inc - mine;
            for (int h = tid; h < kEdgeSlots; h += kTileThreads)
                if (s_edges.cnt[h]) { if (at < a.sink.cap) { a.sink.keys[at] = (uint64_t)s_edges.keys[h]; a.sink.w[at] = s_edges.cnt[h]; } at++; }
        }
    }
}

// The records k_assign_tiles left over (several aligned blocks, not all inside one segment): the generic rules, one record
// per thread, every lane busy.  Edges are counted in a per-block table like in the tile kernel.
template <int MIN_BLOCKS>
__global__ void __launch_bounds__(128, MIN_BLOCKS) k_edges_generic(P2Args a) {
    __shared__ TileEdgeTable s_edges;
    __shared__ int32_t s_tot, s_woff[4];
    __shared__ unsigned long long s_at;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < kEdgeSlots; i += 128) { s_edges.keys[i] = kEmptyKey; s_edges.cnt[i] = 0; }
    if (tid == 0) s_edges.spill = a.sink;
    __syncthreads();
    const int32_t n = *a.n_slow < a.slow_cap ? *a.n_slow : a.slow_cap;
    // A block takes CONTIGUOUS runs of the list (tiles append their records in one piece, so a run is a stretch of the genome): the
    // run's edges repeat and are counted in the table, which is written out whenever it is more than half full -- never spilled
    // edge by edge through the one global counter.
    constexpr int32_t kRun = 128 * 4;
    for (int32_t base = blockIdx.x * kRun; base < n; base += gridDim.x * kRun) {
        const int32_t end = base + kRun < n ? base + kRun : n;
        for (int32_t q = base + tid; q < end; q += 128) {
            const int64_t r = a.slow_list[q];
            const int32_t out = conc_edges_generic(a.desc, a.nt_dev, r, &s_edges);
            a.res0[r] = out;
            if (out == -3) { const int32_t k = atomicAdd(a.n_sens, 1); if (k < a.sens_cap) a.sens[k] = (int32_t)r; }
        }
        __syncthreads();
        const bool last = base + (int64_t)gridDim.x * kRun >= n;
        int mine = 0;
        for (int h = tid; h < kEdgeSlots; h += 128) mine += s_edges.cnt[h] != 0;
        int inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
        if (lane == 31) s_woff[warp] = inc;
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < 4; w++) { const int c = s_woff[w]; s_woff[w] = tot; tot += c; }
            if (!last && tot <= kEdgeSlots / 2) tot = 0;  // room left: keep counting
            s_tot = tot;
            if (tot > 0) s_at = atomicAdd(a.sink.counter, (unsigned long long)tot);
        }
        __syncthreads();
        if (s_tot > 0) {
            long long at = (long long)s_at + s_woff[warp] + inc - mine;
            for (int h = tid; h < kEdgeSlots; h += 128)
                if (s_edges.cnt[h]) {
                    if (at < a.sink.cap) { a.sink.keys[at] = (uint64_t)s_edges.keys[h]; a.sink.w[at] = s_edges.cnt[h]; }
                    at++;
                    s_edges.keys[h] = kEmptyKey; s_edges.cnt[h] = 0;
                }
        }
        __syncthreads();
    }
}

// ReadsOther blocks of <= 3 bp, second pass: the segment each one is counted in (depth_short_node), and how many of them tie
// with an entry of the same (chr, start) that would move them (then the reference's answer is its unstable sort's tie order)
__global__ void k_depth_short_nodes(NodeTable nt, const uint32_t *omask, int4 *shorts, const int32_t *n_short, int32_t cap, int32_t *n_unstable) {
    const int32_t n = *n_short < cap ? *n_short : cap;
    for (int32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        int4 x = shorts[q];
        bool un = false;
        x.w = depth_short_node(nt, omask, x.x, x.y, x.z, &un);
        shorts[q] = x;
        if (un) atomicAdd(n_unstable, 1);
    }
}
__global__ void k_depth_short_apply(const int4 *shorts, int32_t n, int32_t *cnt_other, int32_t *sum_other) {
    for (int32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const int4 x = shorts[q];
        if (x.w != kNoNode) { atomicAdd(&cnt_other[x.w], 1); atomicAdd(&sum_other[x.w], x.z); }
    }
}
// ---- the tie order of sort(ReadsOther) (:781), only when some short block depends on it ----------------------------------
// ReadsOther in push order: the non-first blocks of the records that feed the depth streams, keyed by (chr, start).
struct OtherCountOp {
    const uint32_t *blk_off; const uint8_t *cls; int64_t r_break;
    __device__ int32_t operator()(int64_t r) const { if (r >= r_break || !(cls[r] & CLS_HASBLK)) return 0; const uint32_t nb = blk_off[r + 1] - blk_off[r]; return nb > 1 ? (int32_t)(nb - 1) : 0; }
};
__global__ void k_other_fill(DevBatch b, const uint8_t *cls, int64_t r_break, const int32_t *off, uint64_t *keys, uint32_t *idx, int32_t *len) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= b.n_rec || r >= r_break || !(cls[r] & CLS_HASBLK)) return;
    const uint32_t o = b.blk_off[r], e = b.blk_off[r + 1];
    int32_t at = off[r];
    const uint64_t c = (uint64_t)(uint32_t)b.ref_id[r] << 32;
    for (uint32_t k = o + 1; k < e; k++, at++) { keys[at] = c | (uint32_t)b.blk_ref_pos[k]; idx[at] = (uint32_t)at; len[at] = b.blk_match_ref[k]; }
}
// own segment of every entry, in sorted order (long: first segment ending right of the start; short: earliest containing one)
__global__ void k_other_own(NodeTable nt, const uint64_t *keys, const uint32_t *idx, const int32_t *len, int64_t m, int32_t *own) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p < m) own[p] = depth_target(nt, (int32_t)(keys[p] >> 32), (int32_t)(uint32_t)keys[p], len[idx[p]]);
}
// the merge loop's cursor at entry p = running maximum of the own segments up to and including p: short entries are counted there
__global__ void k_other_apply(NodeTable nt, const uint64_t *keys, const uint32_t *idx, const int32_t *len, const int32_t *cursor, int64_t m, int32_t *cnt_other, int32_t *sum_other) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= m) return;
    const int32_t l = len[idx[p]];
    if (l > kSeedThresh) return;
    const int32_t c = cursor[p];
    if (c != kNoNode && c < nt.n && depth_contained(nt, c, (int32_t)(keys[p] >> 32), (int32_t)(uint32_t)keys[p], l)) { atomicAdd(&cnt_other[c], 1); atomicAdd(&sum_other[c], l); }
}

// exclusive running maximum of the per-tile maximum targets (one block of 32 warps, each walking a contiguous run of tiles
// 32 at a time); tiles with no counted read pass the cursor on
__global__ void __launch_bounds__(1024) k_depth_scan(DepthTile *dt, int32_t n_tiles) {
    __shared__ int32_t s_mx[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned full = 0xffffffffu;
    const int per = ((n_tiles + 31) / 32 + 31) / 32 * 32;
    const int lo = warp * per < n_tiles ? warp * per : n_tiles, hi = (warp + 1) * per < n_tiles ? (warp + 1) * per : n_tiles;
    int32_t mx = -1;
    for (int t = lo + lane; t < hi; t += 32) { const int32_t v = dt[t].max_target; if (v > mx) mx = v; }
    mx = __reduce_max_sync(full, mx);
    if (lane == 0) s_mx[warp] = mx;
    __syncthreads();
    mx = -1;
    for (int w = 0; w < warp; w++) if (s_mx[w] > mx) mx = s_mx[w];
    for (int base = lo; base < hi; base += 32) {
        const int t = base + lane;
        const int32_t own = t < hi ? dt[t].max_target : -1;
        int32_t inc = own;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, inc, d); if (lane >= d && u > inc) inc = u; }
        int32_t exc = __shfl_up_sync(full, inc, 1);
        if (lane == 0) exc = -1;
        if (t < hi) dt[t].max_target = exc > mx ? exc : mx;
        const int32_t tot = __shfl_sync(full, inc, 31);
        if (tot > mx) mx = tot;
    }
}

// Tiles whose incoming cursor is ahead of their first target counted some reads against the wrong segment: redo those
// reads literally (one thread per such tile; sorted input makes them rare).
__global__ void k_depth_fix(DevBatch b, const uint8_t *cls, NodeTable nt, int64_t r_break, const DepthTile *dt, int32_t n_tiles, int32_t *cnt_main, int32_t *sum_main) {
    const int32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const int32_t carry = dt[t].max_target;
    if (carry < 0 || dt[t].first_target == 0x7fffffff || carry <= dt[t].first_target) return;
    int32_t loc = -1;
    const int64_t r0 = (int64_t)t * kTile, r1 = r0 + kTile < b.n_rec ? r0 + kTile : b.n_rec;
    for (int64_t r = r0; r < r1 && r < r_break; r++) {
        if (!(cls[r] & CLS_HASBLK)) continue;
        const uint32_t o = b.blk_off[r];
        const int32_t c = b.ref_id[r], st = b.blk_ref_pos[o], l = b.blk_match_ref[o];
        const int32_t m = depth_target(nt, c, st, l);
        if (m > loc) loc = m;
        if (loc >= carry) break;  // from here on the local cursor was the true one
        if (loc != kNoNode && loc >= 0 && loc < nt.n && depth_contained(nt, loc, c, st, l)) { atomicAdd(&cnt_main[loc], -1); atomicAdd(&sum_main[loc], -l); }
        if (carry != kNoNode && carry < nt.n && depth_contained(nt, carry, c, st, l)) { atomicAdd(&cnt_main[carry], 1); atomicAdd(&sum_main[carry], l); }
    }
}

}  // namespace sq
#endif
