// Shared device-side vocabulary of the B200 segment-graph path: the HBM-resident record batch,
// the segment (node) table and the per-record helpers every kernel uses.
// The element-level rules are `SQ_HD` (host+device) so that tests/emul can step the very same
// functions on the CPU while no GPU is attached; the product only ever runs them inside kernels.
#ifndef SQ_COMMON_CUH
#define SQ_COMMON_CUH
#include <stdint.h>

#if defined(__CUDACC__)
#define SQ_HD __host__ __device__ __forceinline__
#define SQ_HD_NOINLINE __host__ __device__ __noinline__ inline  // (inline: several translation units include it)
#else
#define SQ_HD inline
#define SQ_HD_NOINLINE inline
#endif

namespace sq {

constexpr int kMaxBlocks = 16;     // per mate (packer rejects more; keeps sorts insertion-only like std::sort's n<=16 path)
constexpr int kLocateTol = 5;      // LocateRead overhang tolerance   (SegmentGraph.cpp:1209)
constexpr int kSeedThresh = 3;     // BuildNode_STAR `thresh`          (SegmentGraph.cpp:286)
constexpr int kMateBlockLen = 15;  // synthetic mate block             (SegmentGraph.cpp:308)

// record class bits written by the classify kernel
enum : uint8_t {
    CLS_GATE = 1,      // passes the record gate (SegmentGraph.cpp:302 / 1584 / 3136)
    CLS_KEEP = 2,      // ... and is not Equal() to the previous gate-passing record (:315-318, 1597-1600)
    CLS_CONC = 4,      // kept, proper FR pair within 750 kb (:651-654) and owns >= 1 block (:655)
    CLS_PART = 8,      // CLS_CONC and partially aligned (:668-683) => PartialAlignCluster, else ConcordantCluster
    CLS_HASBLK = 16,   // kept and owns >= 1 block (feeds ReadsMain, :320-333)
    CLS_DISPL = 32,    // CLS_HASBLK and the first kept block does not start at the record position (leading block dropped)
    CLS_REST = 64,     // CLS_CONC with a mate flag and >= 2 blocks: its later blocks feed ConcordRest (:690-699)
};

// HBM-resident SoA batch (include/squid_b200.h: sqg_batch), device pointers.
struct DevBatch {
    int64_t n_rec = 0, n_blk = 0;
    const int32_t *ref_id = nullptr, *pos = nullptr, *mate_ref_id = nullptr, *mate_pos = nullptr, *end_pos = nullptr;
    const uint16_t *flag = nullptr, *total_len = nullptr, *lowphred_run = nullptr;
    const uint8_t *mapq = nullptr, *aux = nullptr;
    const uint32_t *blk_off = nullptr;
    const int32_t *blk_ref_pos = nullptr, *blk_match_ref = nullptr;
    const uint16_t *blk_read_pos = nullptr, *blk_match_read = nullptr;
};

// The same batch seen through a tile staged in shared memory: arrays indexed by the GLOBAL record / block index, backed by
// staging buffers that start at record `rec0` / block `blk0`.  The element rules are templates over the batch type, so the
// very same code classifies from HBM (DevBatch) and from a staged tile (TileBatch).
template <class T> struct OffPtr {
    const T *p; uint32_t off;  // indices stay below 2^32 (records: 2^31 per context, blocks: uint32 offsets)
    SQ_HD T operator[](int64_t i) const { return p[(uint32_t)i - off]; }
};
template <class T> SQ_HD const T *elem_ptr(const T *p, int64_t i) { return p + i; }
template <class T> SQ_HD const T *elem_ptr(const OffPtr<T> &q, int64_t i) { return q.p + ((uint32_t)i - q.off); }
struct TileBatch {
    int64_t n_rec = 0, n_blk = 0;
    OffPtr<int32_t> ref_id, pos, mate_ref_id, mate_pos, end_pos;
    OffPtr<uint16_t> flag, total_len, lowphred_run;
    OffPtr<uint8_t> mapq, aux;
    OffPtr<uint32_t> blk_off;
    OffPtr<int32_t> blk_ref_pos, blk_match_ref;
    OffPtr<uint16_t> blk_read_pos, blk_match_read;
};

struct Params {
    int32_t min_mapq, max_lowphred_len, concord_dist_pos, concord_dist_idx, read_len, n_ref;
};

// Segment table: segments tile every chromosome; chr_head(nt, c).c0..c1 are the segments of c.
// The position index answers "which segment holds position x" (LocateRead's scans, the depth cursor, the spanning-block
// fallback) in two dependent loads: the chromosome's 16-byte header, then the 16-byte entry of the bin that holds x
// (positions [k<<bin_shift, (k+1)<<bin_shift) of chromosome c are entry head[c].bin0 + k), which names the segment holding
// the bin's start together with its Position and End.  Only a position past that segment walks on, bounded by the segment
// that holds the next bin's start.  Without bins the lookups fall back to binary searches.
// The index comes in two forms with the same content: packed (head, bins: what the device reads, built by install_nodes) and
// plain (chr_first, bin_off, bin_seg: what a host-side caller such as the CPU stepping harness builds).  chr_head / bin_ent
// read either; every lookup above them is written once.
struct alignas(16) ChrHead {
    int32_t c0, c1;  // segments of the chromosome: [c0, c1), c1 == c0 when it has none
    int32_t bin0;    // its first bin entry
    int32_t end1;    // End of its last segment
};
struct alignas(16) BinEnt {
    int32_t j;         // segment holding the bin's start (the last segment of the chromosome when that is its end)
    int32_t pos, end;  // Position and End of segment j
    int32_t hi;        // segment holding the next bin's start (the last segment of the chromosome for its last bin)
};
struct NodeTable {
    int32_t n = 0, n_ref = 0;
    const int32_t *chr = nullptr, *pos = nullptr, *end = nullptr;  // end = Position + Length
    const ChrHead *head = nullptr;                                 // packed: n_ref headers
    const BinEnt *bins = nullptr;                                  //         and the bin entries
    const int32_t *chr_first = nullptr;                            // plain:  n_ref + 1
    const int32_t *bin_seg = nullptr, *bin_off = nullptr;          //         bin_seg[bin_off[c] + k] = BinEnt::j; bin_off: n_ref + 1
    int32_t bin_shift = 12;
};
// A segment with its Position and End, as a lookup returns it.
struct SegHit {
    int32_t s, pos, end;
};

// An aligned block in registers/local memory (SingleBamRec_t).
struct Blk {
    int32_t ref_id, ref_pos, match_ref, read_pos, match_read;
    bool rev;
};

SQ_HD bool flag_mapped(uint16_t f) { return !(f & 0x4); }
SQ_HD bool flag_mate_mapped(uint16_t f) { return !(f & 0x8); }
SQ_HD bool flag_rev(uint16_t f) { return f & 0x10; }
SQ_HD bool flag_mate_rev(uint16_t f) { return f & 0x20; }
SQ_HD bool flag_first(uint16_t f) { return f & 0x40; }
SQ_HD bool flag_second(uint16_t f) { return f & 0x80; }
SQ_HD bool flag_dup(uint16_t f) { return f & 0x400; }
SQ_HD bool flag_proper(uint16_t f) { return f & 0x2; }

// Record gate shared by the three passes (SegmentGraph.cpp:302, 1584, 3136).  A mapped record with
// RefID -1 is rejected at load time, so the three gates coincide.
SQ_HD bool record_gate(uint16_t flag, uint8_t mapq, uint8_t aux, int32_t ref_id, int32_t min_mapq) {
    return !((aux & (1u | 2u | 8u)) || (int32_t)mapq < min_mapq || flag_dup(flag) || !flag_mapped(flag) || ref_id < 0);
}
SQ_HD bool has_mate_block(uint16_t flag, int32_t mate_ref_id) { return flag_mate_mapped(flag) && mate_ref_id != -1; }

// first index in [lo,hi) with a[i] >= v
SQ_HD int32_t lower_bound_i32(const int32_t *a, int32_t lo, int32_t hi, int32_t v) {
    while (lo < hi) {
        int32_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// first index in [lo,hi) with a[i] > v
SQ_HD int32_t upper_bound_i32(const int32_t *a, int32_t lo, int32_t hi, int32_t v) {
    while (lo < hi) {
        int32_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Header of chromosome c over a table whose chromosomes start at chr_first[c] (n_ref + 1 entries), with its bins starting at
// bin_off[c].
SQ_HD ChrHead chr_head_value(const int32_t *chr_first, const int32_t *end, const int32_t *bin_off, int32_t c) {
    const int32_t c0 = chr_first[c], c1 = chr_first[c + 1];
    return ChrHead{c0, c1, bin_off ? bin_off[c] : 0, c1 > c0 ? end[c1 - 1] : 0};
}
SQ_HD bool has_bins(const NodeTable &nt) { return nt.bins || nt.bin_seg; }
#if defined(__CUDA_ARCH__)
SQ_HD ChrHead chr_head(const NodeTable &nt, int32_t c) {
    const int4 v = __ldg(reinterpret_cast<const int4 *>(nt.head) + c);
    return ChrHead{v.x, v.y, v.z, v.w};
}
SQ_HD BinEnt bin_ent(const NodeTable &nt, const ChrHead &, int32_t k) {
    const int4 v = __ldg(reinterpret_cast<const int4 *>(nt.bins) + k);
    return BinEnt{v.x, v.y, v.z, v.w};
}
#else
SQ_HD ChrHead chr_head(const NodeTable &nt, int32_t c) { return nt.head ? nt.head[c] : chr_head_value(nt.chr_first, nt.end, nt.bin_off, c); }
// (the plain form names no next-bin segment: the chromosome's last segment bounds the walk instead, which changes how the
// lookup steps, never what it returns)
SQ_HD BinEnt bin_ent(const NodeTable &nt, const ChrHead &h, int32_t k) {
    if (nt.bins) return nt.bins[k];
    const int32_t j = nt.bin_seg[k];
    return BinEnt{j, nt.pos[j], nt.end[j], h.c1 - 1};
}
#endif

// value of bin k of chromosome c: the segment holding position k << bin_shift (the last segment of c at the chromosome end)
SQ_HD int32_t bin_seg_value(const NodeTable &nt, int32_t c, int32_t k) {
    const ChrHead h = chr_head(nt, c);
    if (h.c1 <= h.c0) return h.c0;
    const int32_t j = upper_bound_i32(nt.end, h.c0, h.c1, k << nt.bin_shift);
    return j < h.c1 ? j : h.c1 - 1;
}
// packed entry of bin k of chromosome c (nb bins); the headers must be in place
SQ_HD BinEnt bin_ent_value(const NodeTable &nt, int32_t c, int32_t k, int32_t nb) {
    const ChrHead h = chr_head(nt, c);
    if (h.c1 <= h.c0) return BinEnt{h.c0, 0, 0, h.c0};
    const int32_t j = bin_seg_value(nt, c, k);
    return BinEnt{j, nt.pos[j], nt.end[j], k + 1 < nb ? bin_seg_value(nt, c, k + 1) : h.c1 - 1};
}

// Segment of the chromosome of header h (h.c1 > h.c0) that holds position x, clamped to its first / last segment when x lies
// outside [Position of the first, End of the last); == upper_bound_i32(nt.end, h.c0, h.c1, x), clamped to h.c1 - 1.
SQ_HD SegHit seg_at(const NodeTable &nt, const ChrHead &h, int32_t x) {
    int32_t j;
    if (x >= h.end1) j = h.c1 - 1;
    else if (has_bins(nt)) {
        const BinEnt e = bin_ent(nt, h, h.bin0 + (x < 0 ? 0 : x >> nt.bin_shift));
        if (e.end > x) return SegHit{e.j, e.pos, e.end};
        if (e.hi - e.j <= 4) {  // the tiling: each step's Position is the End before it
            int32_t q = e.end;
            j = e.j;
            for (;;) { j++; const int32_t t = nt.end[j]; if (t > x) return SegHit{j, q, t}; q = t; }
        }
        j = upper_bound_i32(nt.end, e.j + 1, e.hi + 1, x);
    } else j = upper_bound_i32(nt.end, h.c0, h.c1, x);
    return SegHit{j, nt.pos[j], nt.end[j]};
}
// first segment of the chromosome with End > v (== upper_bound_i32(nt.end, c0, c1, v)); s == c1 (Position, End unset) if none
SQ_HD SegHit seg_first_end_gt(const NodeTable &nt, const ChrHead &h, int32_t v) {
    if (h.c1 <= h.c0 || v >= h.end1) return SegHit{h.c1, 0, 0};
    return seg_at(nt, h, v);
}
// first segment of the chromosome with End >= v  (== lower_bound_i32(nt.end, c0, c1, v))
SQ_HD int32_t seg_first_end_ge(const NodeTable &nt, const ChrHead &h, int32_t v) {
    return seg_first_end_gt(nt, h, v - 1).s;
}
// last segment of the chromosome with Position <= v, c0 - 1 if none  (== upper_bound_i32(nt.pos, c0, c1, v) - 1)
SQ_HD int32_t seg_last_pos_le(const NodeTable &nt, const ChrHead &h, int32_t v) {
    if (h.c1 <= h.c0) return h.c0 - 1;
    const SegHit x = seg_at(nt, h, v);
    return x.pos <= v ? x.s : x.s - 1;  // (Position > v only for the first segment: v lies left of the chromosome's table)
}
// the same with the chromosome's segments [c0, c1) at hand
SQ_HD int32_t seg_last_pos_le(const NodeTable &nt, int32_t c, int32_t c0, int32_t c1, int32_t v) {
    return c1 <= c0 ? c0 - 1 : seg_last_pos_le(nt, chr_head(nt, c), v);
}

// Own blocks of record r sorted by read position (SortbyReadPos: std::sort on <=16 elements is an
// insertion sort, i.e. stable).  Returns the count.
template <class B>
SQ_HD int load_sorted_blocks(const B &b, int64_t r, Blk *out) {
    const uint32_t o = b.blk_off[r], n = b.blk_off[r + 1] - o;
    const int32_t rid = b.ref_id[r];
    const bool rev = flag_rev(b.flag[r]);
    int cnt = (int)n;
    if (cnt > kMaxBlocks) cnt = kMaxBlocks;
    for (int k = 0; k < cnt; k++) {
        Blk x;
        x.ref_id = rid; x.ref_pos = b.blk_ref_pos[o + k]; x.match_ref = b.blk_match_ref[o + k];
        x.read_pos = b.blk_read_pos[o + k]; x.match_read = b.blk_match_read[o + k]; x.rev = rev;
        int j = k;
        while (j > 0 && x.read_pos < out[j - 1].read_pos) { out[j] = out[j - 1]; j--; }
        out[j] = x;
    }
    return cnt;
}

}  // namespace sq
#endif
