// Phase 1 of the path in ONE pass over the record batch: batch validation, record gate, duplicate filter against the
// previous gate-passing record, concordance / partial-alignment class, and everything the seed machine needs from the
// stream: the running otherChr/otherrightmost maximum at coverage gaps and the sparse lists of coverage-gap, partially
// aligned and displaced records.
// Reference: SegmentGraph.cpp:297-318 (gate, Equal), :651-689 (classes, otherrightmost), :616-620 (0-coverage test).
//
// Tiles are independent (no tile waits for another on the common path):
//   k_classify_tiles : stages a tile with TMA bulk copies, classifies it, writes the class bytes, the tile's aggregate
//                      (maximum other key, #partial, #displaced) and the coverage-gap CANDIDATES of the tile -- records that
//                      look like a gap when only the tile's own running maximum is known (a superset of the true gaps:
//                      the true maximum is never smaller).
//   k_tile_scan      : exclusive scan of the per-tile aggregates (one block).
//   k_finish_gaps    : decides every candidate with the exclusive maximum of its tile.
//   k_compact_lists  : ordered compaction of the partial / displaced record lists from the class bytes (1 B/record).
// The previous gate-passing record of a tile's first gate-passing record is found by a 32-record look behind the tile; only
// if that fails (a run of > 32 filtered records) the tile walks the per-tile gate words (decoupled look-back).
#ifndef SQ_PHASE1_CUH
#define SQ_PHASE1_CUH
#include "sq_classify.cuh"
#include "sq_depth_cover.cuh"
#include "sq_stream.cuh"

namespace sq {

// TileAgg, P1Out and BatchDesc: sq_stream.cuh
constexpr uint32_t kP1Fields = F_REF | F_POS | F_MREF | F_MPOS | F_FLAG | F_TLEN | F_LOWQ | F_MAPQ | F_AUX | F_BLOCKS;

// classification straight from HBM: records whose predecessor lies before the tile, tiles too dense to stage
__device__ __noinline__ ClassifyOut classify_from_hbm(const BatchDesc *desc, int64_t r, int64_t prev) { return classify_record(desc->b, desc->p, r, prev); }

__device__ __forceinline__ void push_candidates(const P1Out &o, unsigned mask, int64_t rec, uint64_t key, int32_t *s_bad) {
    const int lane = threadIdx.x & 31;
    int32_t base = 0;
    if (lane == 0) base = atomicAdd(o.n_cand, __popc(mask));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (mask & (1u << lane)) {
        const int32_t k = base + __popc(mask & ((1u << lane) - 1u));
        if (k < o.cand_cap) { o.cand_rec[k] = (int32_t)rec; o.cand_key[k] = key; }
        else atomicOr(s_bad, 16);
    }
}

__global__ void __launch_bounds__(kTileThreads, 8) k_classify_tiles(DevBatch b, Params p, P1Out o, int bulk_ok) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    TileStage &s = *reinterpret_cast<TileStage *>(smem_raw);
    __shared__ int s_tile;
    __shared__ uint32_t s_gate[kTileChunks];
    __shared__ int32_t s_cmax[kTileChunks];   // per chunk: max key end, then the exclusive maximum before the chunk
    __shared__ int32_t s_pc[kWarpsPerTile], s_dp[kWarpsPerTile], s_qcnt[kTileChunks];
    __shared__ long long s_prev_carry;
    __shared__ int32_t s_bad, s_lmax, s_minkeep, s_ccmax, s_nq, s_qmax;
    int32_t *s_end = s.end_pos;               // per record: end of the first block if the record updates otherrightmost, else 0
    uint16_t *s_flen = s.total_len;           // per record: first_len (a record's total_len is only read by its own thread, before)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned full = 0xffffffffu;
    if (tid == 0) { s_tile = atomicAdd(o.ticket, 1); s_bad = 0; s_lmax = 0; s_minkeep = kTile; s_ccmax = kNoCcEnd; s_nq = 0; s_qmax = -1; }
    __syncthreads();
    const int tile = s_tile;
    const StageTicket tk = stage_issue<kP1Fields>(s, b, nullptr, tile, bulk_ok != 0);
    const TileInfo ti = tk.ti;
    const int n = ti.n;
    const int64_t rec0 = ti.rec0;
    // while the copies fly: the 32 records before the tile, is one of them gate-passing?  (warp 0)
    long long walk = -2;  // -2: none within 32 records (and the stream does not start there)
    if (warp == 0) {
        const int64_t q = rec0 - 1 - lane;
        const bool g = q >= 0 && record_gate(b.flag[q], b.mapq[q], b.aux[q], b.ref_id[q], p.min_mapq);
        const unsigned m = __ballot_sync(full, g);
        if (m) walk = rec0 - 1 - (__ffs(m) - 1);
        else if (rec0 <= 32) walk = -1;
    }
    stage_wait<kP1Fields>(s, b, nullptr, tk);
    const TileBatch tb = tile_view(s, ti, b);

    // ---- gate bits + batch validation ----------------------------------------------------------------------------
#pragma unroll 1
    for (int j = 0; j < kTileRPT; j++) {
        const int i = j * kTileThreads + tid;
        bool g = false;
        int bad = 0;
        if (i < n) {
            const int32_t rid = s.ref_id[i];
            const uint16_t f = s.flag[i];
            g = record_gate(f, s.mapq[i], s.aux[i], rid, p.min_mapq);
            if (rid >= p.n_ref || rid < -1) bad |= 1;
            if (rid < 0 && flag_mapped(f)) bad |= 2;
            const uint32_t o0 = s.blk_off[i], o1 = s.blk_off[i + 1];
            if (o1 < o0 || o1 - o0 > (uint32_t)kMaxBlocks) bad |= 4;
            const int64_t r = rec0 + i;
            if (r + 1 < b.n_rec) {
                const int32_t rid2 = i + 1 < n ? s.ref_id[i + 1] : b.ref_id[r + 1], pos2 = i + 1 < n ? s.pos[i + 1] : b.pos[r + 1];
                const uint64_t k1 = rid < 0 ? ~0ull : (((uint64_t)(uint32_t)rid << 32) | (uint32_t)s.pos[i]);
                const uint64_t k2 = rid2 < 0 ? ~0ull : (((uint64_t)(uint32_t)rid2 << 32) | (uint32_t)pos2);
                if (k2 < k1) bad |= 8;
            }
        }
        const unsigned gm = __ballot_sync(full, g);
        if (lane == 0) s_gate[j * kWarpsPerTile + warp] = gm;
        if (bad) atomicOr(&s_bad, bad);
    }
    __syncthreads();
    const bool usable = !(s_bad & 5);  // bad ref_id / blk_off in the tile: nothing of it is classified (the call fails anyway)
    const bool staged = ti.nb >= 0;
    if (warp == 0) {  // the tile's gate word; the carry into the tile
        const uint32_t w = lane < kTileChunks ? s_gate[lane] : 0u;
        const unsigned nz = __ballot_sync(full, w != 0u);
        uint64_t agg = 0;
        if (nz) {
            const int hw = 31 - __clz(nz);
            const uint32_t hv = __shfl_sync(full, w, hw);
            agg = (uint64_t)(rec0 + hw * 32 + (31 - __clz(hv))) + 1ull;
        }
        if (lane == 0) word_publish(o.gate_word, tile, nz ? 2u : 1u, agg);
        if (nz && walk == -2) walk = (long long)word_lookback_max(o.gate_word, tile) - 1;  // rare: > 32 filtered records in a row
        if (lane == 0) s_prev_carry = walk;
    }
    __syncthreads();

    // ---- classify ------------------------------------------------------------------------------------------------
    // single-chromosome tiles (all but a handful) compare 32-bit block ends; the others are finished by one thread below
    const int32_t chr_tile = s.ref_id[0];
    const bool single_chr = chr_tile >= 0 && s.ref_id[n - 1] == chr_tile;
    int32_t flen_max = 0, npc = 0, ndp = 0, cc_max = kNoCcEnd, nq = 0, q_max = -1;
#pragma unroll 1
    for (int j = 0; j < kTileRPT; j++) {
        const int i = j * kTileThreads + tid;
        uint8_t c = 0;
        int32_t key_end = 0, co_len = 0;
        if (i < n && usable && ((s_gate[i >> 5] >> (i & 31)) & 1u)) {
            int word = i >> 5;
            uint32_t m = s_gate[word] & ((1u << (i & 31)) - 1u);
            while (m == 0u && word > 0) { word--; m = s_gate[word]; }
            const int64_t prev = m ? rec0 + word * 32 + (31 - __clz(m)) : (int64_t)s_prev_carry;
            const int64_t r = rec0 + i;
            const ClassifyOut co = (staged && prev >= rec0) ? classify_record(tb, p, r, prev) : classify_from_hbm(o.desc, r, prev);
            c = co.cls; key_end = (int32_t)(uint32_t)co.other_key;  // (other_key >> 32) - 1 == ref_id of the record
            co_len = co.first_len;
            if (co.first_len > flen_max) flen_max = co.first_len;
            if (co.cc_end > cc_max) cc_max = co.cc_end;
        }
        // phase 3 (ExactBPConcordantSupport's pass) keeps the gate-passing right-hand mates: counted here, per tile, so that its
        // compaction kernel knows every tile's rank offset without a look-back chain
        int32_t qs = -1;
        if (i < n && (c & CLS_GATE)) {
            const uint16_t f = s.flag[i];
            const int32_t rid = s.ref_id[i], ps = s.pos[i], mr = s.mate_ref_id[i], mp = s.mate_pos[i];
            if (cover_qualifies(c, f, rid, ps, mr, mp)) { qs = cover_start(f, rid, ps, mr, mp); if (qs < 0) qs = 0; }
        }
        const int chunk = j * kWarpsPerTile + warp;
        { const int32_t cq = __popc(__ballot_sync(full, qs >= 0)); nq += cq; if (lane == 0) s_qcnt[chunk] = cq; }
        { const int32_t m = __reduce_max_sync(full, qs); if (m > q_max) q_max = m; }
        if (i < n) { s.cls[i] = c; s_end[i] = key_end; s_flen[i] = (uint16_t)(co_len < 65535 ? co_len : 65535); }
        npc += __popc(__ballot_sync(full, (c & CLS_PART) != 0));
        ndp += __popc(__ballot_sync(full, (c & (CLS_CONC | CLS_DISPL)) == (CLS_CONC | CLS_DISPL)));
        const unsigned km = __ballot_sync(full, (c & CLS_KEEP) != 0);
        const int32_t cm = __reduce_max_sync(full, key_end);
        if (lane == 0) { s_cmax[chunk] = cm; if (km) atomicMin(&s_minkeep, chunk * 32 + __ffs(km) - 1); }
    }
    flen_max = __reduce_max_sync(full, flen_max);
    cc_max = __reduce_max_sync(full, cc_max);
    if (lane == 0) { s_pc[warp] = npc; s_dp[warp] = ndp; if (flen_max > 0) atomicMax(&s_lmax, flen_max); if (cc_max > kNoCcEnd) atomicMax(&s_ccmax, cc_max);
                     if (nq) atomicAdd(&s_nq, nq); if (q_max >= 0) atomicMax(&s_qmax, q_max); }
    __syncthreads();
    if (warp == 0) {  // chunk maxima -> exclusive maximum before each chunk; the tile's aggregate
        int32_t inc = lane < kTileChunks ? s_cmax[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, inc, d); if (lane >= d && u > inc) inc = u; }
        const int32_t tot = __shfl_sync(full, inc, 31);
        int32_t exc = __shfl_up_sync(full, inc, 1);
        if (lane == 0) exc = 0;
        if (lane < kTileChunks) s_cmax[lane] = exc;
        if (lane == 0) {
            int32_t a = 0, c2 = 0;
#pragma unroll
            for (int k = 0; k < kWarpsPerTile; k++) { a += s_pc[k]; c2 += s_dp[k]; }
            TileAgg g; g.n_pc = (uint32_t)a; g.n_dp = (uint32_t)c2;
            g.okmax = (single_chr && tot > 0) ? (((uint64_t)(uint32_t)(chr_tile + 1) << 32) | (uint32_t)tot) : 0ull;
            if (single_chr) o.agg[tile] = g;
            else { s_pc[0] = a; s_dp[0] = c2; }
        }
    }
    __syncthreads();
    // ---- coverage-gap candidates (decided with the tile-local maximum; k_finish_gaps applies the true one) ----------
    if (single_chr) {
#pragma unroll 1
        for (int j = 0; j < kTileRPT; j++) {
            const int i = j * kTileThreads + tid, chunk = j * kWarpsPerTile + warp;
            const bool keep = i < n && (s.cls[i] & CLS_KEEP);
            const int32_t pos = i < n ? s.pos[i] : 0;
            const int32_t base = s_cmax[chunk];
            // no record of the chunk can be a gap unless it lies more than ReadLen right of the maximum before the chunk
            // (before any contributing record of the tile the local key is (chr 0, 0), :284-285)
            const bool maybe = keep && (base == 0 ? (chr_tile != 0 || pos > p.read_len) : pos > base + p.read_len);
            if (!__any_sync(full, maybe)) continue;
            int32_t v = i < n ? s_end[i] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, v, d); if (lane >= d && u > v) v = u; }
            int32_t e = __shfl_up_sync(full, v, 1);
            if (lane == 0 || e < base) e = base;
            const bool gap = keep && (e == 0 ? (chr_tile != 0 || pos > p.read_len) : pos > e + p.read_len);
            const unsigned gm = __ballot_sync(full, gap);
            if (gm) push_candidates(o, gm, rec0 + i, e == 0 ? 0ull : (((uint64_t)(uint32_t)(chr_tile + 1) << 32) | (uint32_t)e), &s_bad);
        }
    } else if (tid == 0) {  // a tile that crosses a chromosome boundary (or holds unmapped records): one thread, literally
        uint64_t run = 0;
        for (int i = 0; i < n; i++) {
            if (s.cls[i] & CLS_KEEP) {
                const uint64_t e = run < (1ull << 32) ? (1ull << 32) : run;
                const int32_t oc = (int32_t)(e >> 32) - 1, orr = (int32_t)(uint32_t)e;
                if (s.ref_id[i] != oc || s.pos[i] > orr + p.read_len) {
                    const int32_t k = atomicAdd(o.n_cand, 1);
                    if (k < o.cand_cap) { o.cand_rec[k] = (int32_t)(rec0 + i); o.cand_key[k] = run; }
                    else atomicOr(&s_bad, 16);
                }
            }
            if (s_end[i] != 0) {  // the record updates otherrightmost (classify_record gave it an other_key)
                const uint64_t k = ((uint64_t)(uint32_t)(s.ref_id[i] + 1) << 32) | (uint32_t)s_end[i];
                if (k > run) run = k;
            }
        }
        TileAgg g; g.okmax = run; g.n_pc = (uint32_t)s_pc[0]; g.n_dp = (uint32_t)s_dp[0];
        o.agg[tile] = g;
    }
    // class bytes and first-block lengths out, 4 records at a time (rec0 is a multiple of kTile)
    if (4 * tid + 3 < n) {
        *reinterpret_cast<uint32_t *>(o.cls + rec0 + 4 * tid) = *reinterpret_cast<const uint32_t *>(&s.cls[4 * tid]);
        *reinterpret_cast<uint2 *>(o.first_len + rec0 + 4 * tid) = *reinterpret_cast<const uint2 *>(&s_flen[4 * tid]);
    } else for (int i = 4 * tid; i < n; i++) { o.cls[rec0 + i] = s.cls[i]; o.first_len[rec0 + i] = s_flen[i]; }
    {   // phase 3's (fragment start key, fragment end) pairs of the tile, in record order, compacted inside the tile: the record
        // fields are still staged, so the separate compaction pass over the whole batch (23 B per record) is gone
        const int32_t cq = lane < kTileChunks ? s_qcnt[lane] : 0;
        int32_t inc = cq;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int32_t u = __shfl_up_sync(full, inc, d); if (lane >= d) inc += u; }
        const int32_t exc = inc - cq;  // qualifying records of the tile before chunk `lane`
#pragma unroll 1
        for (int j = 0; j < kTileRPT; j++) {
            const int i = j * kTileThreads + tid;
            bool q = false;
            uint64_t key = 0;
            if (i < n) {
                const uint8_t c = s.cls[i];
                const uint16_t f = s.flag[i];
                const int32_t rid = s.ref_id[i], ps = s.pos[i], mr = s.mate_ref_id[i], mp = s.mate_pos[i];
                q = cover_qualifies(c, f, rid, ps, mr, mp);
                if (q) key = chrpos_key(rid, cover_start(f, rid, ps, mr, mp));
            }
            const unsigned qm = __ballot_sync(full, q);
            const int32_t before = __shfl_sync(full, exc, j * kWarpsPerTile + warp);
            if (q) {
                const int64_t at = (int64_t)tile * kTile + before + __popc(qm & ((1u << lane) - 1u));
                o.qstage_key[at] = key; o.qstage_end[at] = b.end_pos[rec0 + i];
            }
        }
    }
    __syncthreads();
    if (tid == 0) {
        o.cov_nq[tile] = (uint32_t)s_nq;
        uint64_t qk = 0;
        if (single_chr) { if (s_qmax >= 0) qk = chrpos_key(chr_tile, s_qmax); }
        else for (int i = 0; i < n; i++)  // a tile that crosses a chromosome boundary: literally
            if ((s.cls[i] & CLS_GATE) && cover_qualifies(s.cls[i], s.flag[i], s.ref_id[i], s.pos[i], s.mate_ref_id[i], s.mate_pos[i])) {
                const uint64_t k = chrpos_key(s.ref_id[i], cover_start(s.flag[i], s.ref_id[i], s.pos[i], s.mate_ref_id[i], s.mate_pos[i]));
                if (k > qk) qk = k;
            }
        o.cov_qmax[tile] = qk;
        o.ccmax[tile] = single_chr ? s_ccmax : kCcWalkTile;
        if (s_lmax > 0) atomicMax(o.lmax, s_lmax);
        if (s_minkeep < kTile) atomicMin(o.first_kept, (long long)(rec0 + s_minkeep));
        if (s_bad) atomicOr(o.bad_flags, s_bad);
    }
}

// Exclusive scan of the tile aggregates, in place (one block of 32 warps): okmax -> maximum over earlier tiles, n_pc / n_dp ->
// offsets.  Every warp owns a contiguous run of tiles and walks it 32 tiles at a time (coalesced), first to reduce the run,
// then -- with the carry of the runs before it -- to scan it.  totals[1] = #partial, totals[2] = #displaced, *ok_total = the
// maximum over all tiles.
__global__ void __launch_bounds__(1024) k_tile_scan(TileAgg *agg, int32_t n_tiles, int32_t *totals, uint64_t *ok_total) {
    __shared__ uint64_t s_ok[32];
    __shared__ uint32_t s_pc[32], s_dp[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned full = 0xffffffffu;
    const int per = ((n_tiles + 31) / 32 + 31) / 32 * 32;  // tiles per warp, a multiple of 32
    const int lo = warp * per < n_tiles ? warp * per : n_tiles, hi = (warp + 1) * per < n_tiles ? (warp + 1) * per : n_tiles;
    uint64_t ok = 0; uint32_t pc = 0, dp = 0;
    for (int t = lo + lane; t < hi; t += 32) { const TileAgg g = agg[t]; if (g.okmax > ok) ok = g.okmax; pc += g.n_pc; dp += g.n_dp; }
    ok = warp_max_u64(ok); pc = __reduce_add_sync(full, pc); dp = __reduce_add_sync(full, dp);
    if (lane == 0) { s_ok[warp] = ok; s_pc[warp] = pc; s_dp[warp] = dp; }
    __syncthreads();
    ok = 0; pc = 0; dp = 0;  // carry into this warp's run
    for (int w = 0; w < warp; w++) { if (s_ok[w] > ok) ok = s_ok[w]; pc += s_pc[w]; dp += s_dp[w]; }
    if (threadIdx.x == 1023) { totals[1] = (int32_t)(pc + s_pc[31]); totals[2] = (int32_t)(dp + s_dp[31]); }
    for (int base = lo; base < hi; base += 32) {
        const int t = base + lane;
        TileAgg g; g.okmax = 0; g.n_pc = 0; g.n_dp = 0;
        if (t < hi) g = agg[t];
        uint64_t iok = g.okmax; uint32_t ipc = g.n_pc, idp = g.n_dp;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t a = __shfl_up_sync(full, iok, d);
            const uint32_t x = __shfl_up_sync(full, ipc, d), y = __shfl_up_sync(full, idp, d);
            if (lane >= d) { if (a > iok) iok = a; ipc += x; idp += y; }
        }
        uint64_t eok = __shfl_up_sync(full, iok, 1); uint32_t epc = __shfl_up_sync(full, ipc, 1), edp = __shfl_up_sync(full, idp, 1);
        if (lane == 0) { eok = 0; epc = 0; edp = 0; }
        if (t < hi) { TileAgg e; e.okmax = eok > ok ? eok : ok; e.n_pc = pc + epc; e.n_dp = dp + edp; agg[t] = e; }
        const uint64_t tok = __shfl_sync(full, iok, 31);
        if (tok > ok) ok = tok;
        pc += __shfl_sync(full, ipc, 31); dp += __shfl_sync(full, idp, 31);
    }
    if (threadIdx.x == 1023 && ok_total) *ok_total = ok;  // otherChr/otherrightmost after the last record (range shards: sq_seed.cuh end_other)
}

// Candidate -> gap decision with the true running maximum; non-gaps get the key INT32_MAX so that a sort by record index
// leaves the gaps, ascending, in front.  totals[0] += #gaps.
__global__ void k_finish_gaps(DevBatch b, const TileAgg *excl, int32_t *cand_rec, uint64_t *cand_key, int32_t n_cand, int32_t read_len, int32_t *totals) {
    const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    bool gap = false;
    if (k < n_cand) {
        const int32_t r = cand_rec[k];
        uint64_t e = cand_key[k];
        const uint64_t c = excl[r / kTile].okmax;
        if (c > e) e = c;
        if (e < (1ull << 32)) e = 1ull << 32;
        const int32_t oc = (int32_t)(e >> 32) - 1, orr = (int32_t)(uint32_t)e;
        gap = b.ref_id[r] != oc || b.pos[r] > orr + read_len;
        cand_key[k] = e;
        if (!gap) cand_rec[k] = 0x7fffffff;
    }
    const unsigned m = __ballot_sync(0xffffffffu, gap);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&totals[0], __popc(m));
}

// Ordered lists of partially aligned (CLS_PART) and displaced (CLS_CONC|CLS_DISPL) records from the class bytes.
__global__ void __launch_bounds__(kTileThreads) k_compact_lists(const uint8_t *cls, int64_t n_rec, const TileAgg *excl, int32_t *pc_rec, int32_t *dp_rec) {
    __shared__ int32_t s_pc[kWarpsPerTile], s_dp[kWarpsPerTile];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t tile = blockIdx.x, rec0 = tile * (int64_t)kTile;
    const int64_t r0 = rec0 + 4 * tid;  // this thread: 4 consecutive records
    uint32_t w = 0;
    if (r0 + 3 < n_rec) w = *reinterpret_cast<const uint32_t *>(cls + r0);
    else for (int k = 0; k < 4; k++) if (r0 + k < n_rec) w |= (uint32_t)cls[r0 + k] << (8 * k);
    int32_t mypc = 0, mydp = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t c = (w >> (8 * k)) & 0xffu;
        mypc += (c & CLS_PART) ? 1 : 0;
        mydp += ((c & (CLS_CONC | CLS_DISPL)) == (CLS_CONC | CLS_DISPL)) ? 1 : 0;
    }
    if (!__syncthreads_or(mypc | mydp)) return;
    int32_t ipc = mypc, idp = mydp;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t a = __shfl_up_sync(0xffffffffu, ipc, d), c = __shfl_up_sync(0xffffffffu, idp, d);
        if (lane >= d) { ipc += a; idp += c; }
    }
    if (lane == 31) { s_pc[warp] = ipc; s_dp[warp] = idp; }
    __syncthreads();
    int32_t bpc = (int32_t)excl[tile].n_pc, bdp = (int32_t)excl[tile].n_dp;
    for (int k = 0; k < warp; k++) { bpc += s_pc[k]; bdp += s_dp[k]; }
    bpc += ipc - mypc; bdp += idp - mydp;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t c = (w >> (8 * k)) & 0xffu;
        if (c & CLS_PART) pc_rec[bpc++] = (int32_t)(r0 + k);
        if ((c & (CLS_CONC | CLS_DISPL)) == (CLS_CONC | CLS_DISPL)) dp_rec[bdp++] = (int32_t)(r0 + k);
    }
}

}  // namespace sq
#endif
