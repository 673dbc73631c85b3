// Stream-pass machinery shared by the three record-stream kernels (classify, assignment + depth, coverage):
//   * a tile of kTile consecutive records and the contiguous run of aligned blocks they own is staged in shared memory
//     with TMA bulk copies (cp.async.bulk, completion on an mbarrier) -- one elected thread issues ~14 copies instead of
//     every thread issuing dependent blk_off -> block loads;
//   * cross-tile prefix state (running maxima, compaction offsets) comes from scans of per-tile aggregates; the one
//     dependency a tile may have to resolve while it runs (the previous gate-passing record of the classification pass)
//     is carried with a decoupled look-back over one word per tile;
//   * tiles are handed out through an atomic ticket, which makes "tile t-1 is resident or done" hold for every running
//     tile t (forward progress of the look-back).
// sm_100a only (device code); nothing here runs on the host.
#ifndef SQ_STREAM_CUH
#define SQ_STREAM_CUH
#include "sq_common.cuh"

namespace sq {

constexpr int kTile = 512;           // records per tile
constexpr int kTileThreads = 128;    // threads per tile (kTile / kTileThreads records each, striped); 8 tiles resident per SM
constexpr int kTileRPT = kTile / kTileThreads;
constexpr int kWarpsPerTile = kTileThreads / 32;
constexpr int kTileChunks = kTile / 32;  // 32-record chunks: chunk c = records [32c, 32c+32) of the tile
constexpr int kTileBlkCap = 1152;    // staged blocks per tile (K <= 2.2 with the 8-element alignment slack: all but ~0.1 % of the tiles at the App. C block mix, whose K varies from gene to gene); denser tiles read HBM directly

// ---- what the host hands the stream kernels: the batch descriptor and the classification pass's outputs (sq_phase1.cuh),
// which the wire upload sets up as well as the classification stage --------------------------------------------------------
// (`desc` = device copy of the batch descriptor: taking the address of the kernel parameter would force a per-thread copy)
struct BatchDesc { DevBatch b; Params p; };
struct TileAgg {   // per tile: aggregate, then (after k_tile_scan) exclusive prefix
    uint64_t okmax;
    uint32_t n_pc, n_dp;
};
struct P1Out {
    uint8_t *cls;
    uint16_t *first_len;      // per record: length of the first kept block of a CLS_CONC record (65535 = too long for 16 bits), else 0
    TileAgg *agg;             // n_tiles
    uint32_t *cov_nq; uint64_t *cov_qmax;  // n_tiles: records of the tile that qualify for phase 3 (sq_phase3.cuh), their maximum start key
    uint64_t *qstage_key; int32_t *qstage_end;  // n_rec: the (start key, fragment end) pairs of those records, compacted inside each tile:
                                                // tile t owns [t * kTile, t * kTile + cov_nq[t]) (k_cov_gather closes the gaps)
    int32_t *ccmax;           // n_tiles: maximum end of the ConcordantCluster entries of the tile (kNoCcEnd: none; kCcWalkTile: several chromosomes)
    uint64_t *gate_word;      // n_tiles, zeroed: one-word chain of "1 + index of the last gate-passing record"
    int32_t *cand_rec; uint64_t *cand_key; int32_t *n_cand; int32_t cand_cap;
    int32_t *lmax;
    long long *first_kept;    // initialised to n_rec
    int32_t *bad_flags;       // 1 ref_id range, 2 mapped with ref_id -1, 4 blk_off, 8 unsorted, 16 candidate overflow
    int32_t *ticket;
    int32_t n_tiles;
    const struct BatchDesc *desc;  // device copy of (batch, params) for the out-of-line HBM path
};

// ---- mbarrier + bulk copy ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- decoupled look-back ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xffffffffu, v, d); if (o > v) v = o; }
    return v;
}

// One-word chain: per tile a 64-bit word, status in the top two bits (0 nothing, 1 aggregate, 2 inclusive prefix), payload
// (combined with max) below.  A single 8-byte access carries status and value together.
constexpr uint64_t kWordMask = (1ull << 62) - 1ull;
__device__ __forceinline__ void word_publish(uint64_t *w, int tile, uint32_t status, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(w + tile), "l"(((uint64_t)status << 62) | (v & kWordMask)) : "memory");
}
// warp-collective: maximum of the payloads of tiles [0, tile), walking back until a tile with an inclusive prefix
__device__ __forceinline__ uint64_t word_lookback_max(const uint64_t *w, int tile) {
    const int lane = threadIdx.x & 31;
    uint64_t xa = 0;
    for (int base = tile - 1; base >= 0; base -= 32) {
        const int p = base - lane;
        uint64_t v = 2ull << 62;
        if (p >= 0) {
            do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(w + p) : "memory"); } while ((v >> 62) == 0ull);
        }
        const unsigned pm = __ballot_sync(0xffffffffu, (v >> 62) == 2ull);
        const int stop = pm ? __ffs(pm) - 1 : 31;
        const uint64_t r = warp_max_u64(lane > stop ? 0ull : (v & kWordMask));
        if (r > xa) xa = r;
        if (pm) break;
    }
    return xa;
}

// ---- tile staging -----------------------------------------------------------------------------------------------------
// Shared-memory image of one tile.  Record arrays hold records [rec0, rec0 + n); block arrays hold blocks
// [blk0, blk0 + nb) where blk0 = blk_off[rec0] rounded down to a multiple of 8 (16-byte alignment of the 2-byte arrays).
struct TileStage {
    int32_t ref_id[kTile], pos[kTile], mate_ref_id[kTile], mate_pos[kTile], end_pos[kTile];
    uint32_t blk_off[kTile + 8];
    int32_t b_ref_pos[kTileBlkCap], b_match_ref[kTileBlkCap];
    uint16_t flag[kTile], total_len[kTile], lowphred_run[kTile];
    uint16_t b_read_pos[kTileBlkCap], b_match_read[kTileBlkCap];
    uint8_t mapq[kTile], aux[kTile], cls[kTile];
    uint64_t bar[2];  // [0] record arrays, [1] block arrays
};
enum : uint32_t {  // which arrays a kernel needs
    F_REF = 1u << 0, F_POS = 1u << 1, F_MREF = 1u << 2, F_MPOS = 1u << 3, F_END = 1u << 4, F_FLAG = 1u << 5, F_TLEN = 1u << 6,
    F_LOWQ = 1u << 7, F_MAPQ = 1u << 8, F_AUX = 1u << 9, F_CLS = 1u << 10, F_BPOS = 1u << 11, F_BMREF = 1u << 12, F_BRPOS = 1u << 13, F_BMREAD = 1u << 14,
    F_BLOCKS = F_BPOS | F_BMREF | F_BRPOS | F_BMREAD,
};
struct TileInfo {
    int64_t rec0; int32_t n;     // records [rec0, rec0 + n)
    int64_t blk0; int32_t nb;    // staged blocks [blk0, blk0 + nb); nb < 0: the tile's blocks are not staged (read HBM)
};

// Staging is split in two so that a kernel can overlap its own independent loads with the bulk copies:
//   stage_issue : one elected thread arms the mbarriers and issues the bulk copies (all threads call; contains barriers)
//   stage_wait  : every thread waits for the data (the last, partial tile and unaligned batches use plain loads here)
// `cls` may be nullptr.  `bulk_ok`: every base pointer is 16-byte aligned (checked on the host).
struct StageTicket {
    TileInfo ti;
    bool full, plain_blocks;
};
template <uint32_t FIELDS>
__device__ __forceinline__ StageTicket stage_issue(TileStage &s, const DevBatch &b, const uint8_t *cls, int64_t tile, bool bulk_ok) {
    __shared__ TileInfo s_ti;
    const int tid = threadIdx.x;
    const int64_t rec0 = tile * (int64_t)kTile;
    const int32_t n = (int32_t)((b.n_rec - rec0) < kTile ? (b.n_rec - rec0) : kTile);
    const bool full = bulk_ok && n == kTile;  // the last, partial tile is copied with plain loads (no over-read)
    if (tid == 0) { mbar_init(&s.bar[0], 1); mbar_init(&s.bar[1], 1); mbar_init_fence(); }
    __syncthreads();
    if (tid == 0) {
        TileInfo ti;
        ti.rec0 = rec0; ti.n = n;
        if (full) {
            uint32_t bytes = kTile * 4;  // blk_off
            if (FIELDS & F_REF) bytes += kTile * 4; if (FIELDS & F_POS) bytes += kTile * 4; if (FIELDS & F_MREF) bytes += kTile * 4;
            if (FIELDS & F_MPOS) bytes += kTile * 4; if (FIELDS & F_END) bytes += kTile * 4; if (FIELDS & F_FLAG) bytes += kTile * 2;
            if (FIELDS & F_TLEN) bytes += kTile * 2; if (FIELDS & F_LOWQ) bytes += kTile * 2; if (FIELDS & F_MAPQ) bytes += kTile;
            if (FIELDS & F_AUX) bytes += kTile; if (FIELDS & F_CLS) bytes += kTile;
            mbar_expect_tx(&s.bar[0], bytes);
            bulk_g2s(s.blk_off, b.blk_off + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_REF) bulk_g2s(s.ref_id, b.ref_id + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_POS) bulk_g2s(s.pos, b.pos + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_MREF) bulk_g2s(s.mate_ref_id, b.mate_ref_id + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_MPOS) bulk_g2s(s.mate_pos, b.mate_pos + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_END) bulk_g2s(s.end_pos, b.end_pos + rec0, kTile * 4, &s.bar[0]);
            if (FIELDS & F_FLAG) bulk_g2s(s.flag, b.flag + rec0, kTile * 2, &s.bar[0]);
            if (FIELDS & F_TLEN) bulk_g2s(s.total_len, b.total_len + rec0, kTile * 2, &s.bar[0]);
            if (FIELDS & F_LOWQ) bulk_g2s(s.lowphred_run, b.lowphred_run + rec0, kTile * 2, &s.bar[0]);
            if (FIELDS & F_MAPQ) bulk_g2s(s.mapq, b.mapq + rec0, kTile, &s.bar[0]);
            if (FIELDS & F_AUX) bulk_g2s(s.aux, b.aux + rec0, kTile, &s.bar[0]);
            if (FIELDS & F_CLS) bulk_g2s(s.cls, cls + rec0, kTile, &s.bar[0]);
        }
        // the tile's blocks are one contiguous run of the block arrays
        const uint32_t o0 = b.blk_off[rec0], o1 = b.blk_off[rec0 + n];
        const int64_t a0 = (int64_t)(o0 & ~7u), a1 = ((int64_t)o1 + 7) & ~(int64_t)7;
        ti.blk0 = a0;
        ti.nb = (o1 >= o0 && (int64_t)o1 <= b.n_blk && a1 - a0 <= kTileBlkCap) ? (int32_t)(a1 - a0) : -1;
        if (ti.nb >= 0 && a1 > b.n_blk) {  // rounding up would read past the arrays: stage exactly, with plain loads
            ti.nb = (int32_t)((int64_t)o1 - a0);
            ti.nb |= 0x40000000;  // marker: plain copy
        }
        if ((FIELDS & F_BLOCKS) && full && ti.nb > 0 && !(ti.nb & 0x40000000)) {
            const uint32_t nb = (uint32_t)ti.nb;
            uint32_t bytes = 0;
            if (FIELDS & F_BPOS) bytes += nb * 4; if (FIELDS & F_BMREF) bytes += nb * 4; if (FIELDS & F_BRPOS) bytes += nb * 2; if (FIELDS & F_BMREAD) bytes += nb * 2;
            mbar_expect_tx(&s.bar[1], bytes);
            if (FIELDS & F_BPOS) bulk_g2s(s.b_ref_pos, b.blk_ref_pos + a0, nb * 4, &s.bar[1]);
            if (FIELDS & F_BMREF) bulk_g2s(s.b_match_ref, b.blk_match_ref + a0, nb * 4, &s.bar[1]);
            if (FIELDS & F_BRPOS) bulk_g2s(s.b_read_pos, b.blk_read_pos + a0, nb * 2, &s.bar[1]);
            if (FIELDS & F_BMREAD) bulk_g2s(s.b_match_read, b.blk_match_read + a0, nb * 2, &s.bar[1]);
        }
        s.blk_off[n] = o1;  // (the bulk copy writes indices < kTile only)
        s_ti = ti;
    }
    __syncthreads();
    StageTicket t;
    t.ti = s_ti; t.full = full;
    t.plain_blocks = (t.ti.nb >= 0 && (t.ti.nb & 0x40000000)) || (!full && t.ti.nb > 0);
    if (t.ti.nb >= 0) t.ti.nb &= 0x3fffffff;
    return t;
}
template <uint32_t FIELDS>
__device__ __forceinline__ void stage_wait(TileStage &s, const DevBatch &b, const uint8_t *cls, const StageTicket &t) {
    const int tid = threadIdx.x;
    const TileInfo &ti = t.ti;
    if (t.full) {
        mbar_wait(&s.bar[0], 0);
    } else {
        for (int i = tid; i < ti.n; i += kTileThreads) {
            const int64_t r = ti.rec0 + i;
            s.blk_off[i] = b.blk_off[r];
            if (FIELDS & F_REF) s.ref_id[i] = b.ref_id[r]; if (FIELDS & F_POS) s.pos[i] = b.pos[r]; if (FIELDS & F_MREF) s.mate_ref_id[i] = b.mate_ref_id[r];
            if (FIELDS & F_MPOS) s.mate_pos[i] = b.mate_pos[r]; if (FIELDS & F_END) s.end_pos[i] = b.end_pos[r]; if (FIELDS & F_FLAG) s.flag[i] = b.flag[r];
            if (FIELDS & F_TLEN) s.total_len[i] = b.total_len[r]; if (FIELDS & F_LOWQ) s.lowphred_run[i] = b.lowphred_run[r];
            if (FIELDS & F_MAPQ) s.mapq[i] = b.mapq[r]; if (FIELDS & F_AUX) s.aux[i] = b.aux[r]; if (FIELDS & F_CLS) s.cls[i] = cls[r];
        }
    }
    if (FIELDS & F_BLOCKS) {
        if (t.plain_blocks) {
            for (int i = tid; i < ti.nb; i += kTileThreads) {
                const int64_t k = ti.blk0 + i;
                if (FIELDS & F_BPOS) s.b_ref_pos[i] = b.blk_ref_pos[k]; if (FIELDS & F_BMREF) s.b_match_ref[i] = b.blk_match_ref[k];
                if (FIELDS & F_BRPOS) s.b_read_pos[i] = b.blk_read_pos[k]; if (FIELDS & F_BMREAD) s.b_match_read[i] = b.blk_match_read[k];
            }
        } else if (t.full && ti.nb > 0) {
            mbar_wait(&s.bar[1], 0);
        }
    }
    if (!t.full || t.plain_blocks) __syncthreads();  // plain stores of other threads
}

// TileBatch view over a staged tile (global indices).
__device__ __forceinline__ TileBatch tile_view(const TileStage &s, const TileInfo &ti, const DevBatch &b) {
    TileBatch t;
    t.n_rec = b.n_rec; t.n_blk = b.n_blk;
    const uint32_t r0 = (uint32_t)ti.rec0, k0 = (uint32_t)ti.blk0;
    t.ref_id = {s.ref_id, r0}; t.pos = {s.pos, r0}; t.mate_ref_id = {s.mate_ref_id, r0}; t.mate_pos = {s.mate_pos, r0}; t.end_pos = {s.end_pos, r0};
    t.flag = {s.flag, r0}; t.total_len = {s.total_len, r0}; t.lowphred_run = {s.lowphred_run, r0};
    t.mapq = {s.mapq, r0}; t.aux = {s.aux, r0}; t.blk_off = {s.blk_off, r0};
    t.blk_ref_pos = {s.b_ref_pos, k0}; t.blk_match_ref = {s.b_match_ref, k0}; t.blk_read_pos = {s.b_read_pos, k0}; t.blk_match_read = {s.b_match_read, k0};
    return t;
}

}  // namespace sq
#endif
