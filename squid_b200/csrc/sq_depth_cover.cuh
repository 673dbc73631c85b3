// Per-segment depth (Support / AvgDepth numerators) and breakpoint coverage rules.
// Reference behaviour: BuildNode_STAR part D (SegmentGraph.cpp:765-826) and
// ExactBPConcordantSupport's BAM pass (SegmentGraph.cpp:3129-3166).
#ifndef SQ_DEPTH_COVER_CUH
#define SQ_DEPTH_COVER_CUH
#include "sq_common.cuh"

namespace sq {

constexpr int32_t kNoNode = 0x7fffffff;

SQ_HD bool depth_contained(const NodeTable &nt, int32_t j, int32_t chr, int32_t start, int32_t len) {  // :789, :811
    return nt.chr[j] == chr && start >= nt.pos[j] - kSeedThresh && start + len <= nt.end[j] + kSeedThresh;
}

// The merge loop at :784-803 moves a segment cursor forward only: a read is tested against the
// segment max(cursor, n(start)) where n(start) is the first segment of its chromosome that ends
// right of `start`; blocks of <= 3 bp can already be "contained" (+-3) in one of the <= 3
// segments just left of n(start), which then is where the cursor stops.  This returns that
// per-read target m; the cursor is the running maximum of m over the stream.  depth_target_hit gives the target with its
// Position and End (s == kNoNode: none).
SQ_HD SegHit depth_target_hit(const NodeTable &nt, int32_t chr, int32_t start, int32_t len) {
    const SegHit none{kNoNode, 0, 0};
    if (chr < 0 || chr >= nt.n_ref) return none;
    const ChrHead h = chr_head(nt, chr);
    const SegHit n = seg_first_end_gt(nt, h, start);  // first segment with End > start
    if (len <= kSeedThresh) {
        for (int32_t j = (n.s - 3 > h.c0 ? n.s - 3 : h.c0); j < n.s; j++)
            if (depth_contained(nt, j, chr, start, len)) return SegHit{j, nt.pos[j], nt.end[j]};
    }
    return n.s < h.c1 ? n : none;  // a start at/after the chromosome end walks the cursor off the table
}
SQ_HD int32_t depth_target(const NodeTable &nt, int32_t chr, int32_t start, int32_t len) { return depth_target_hit(nt, chr, start, len).s; }
// depth_contained for a segment on chromosome chr, with its Position and End at hand
SQ_HD bool depth_contained(const SegHit &j, int32_t start, int32_t len) {
    return start >= j.pos - kSeedThresh && start + len <= j.end + kSeedThresh;
}

// ---- ReadsOther (:781, :806-825): blocks of <= 3 bp ----------------------------------------------------------------
// ReadsOther is sorted by (chr, start) before its merge loop, so the forward-only cursor at an entry is the maximum "own"
// segment over the entries sorted before it, where own(e) = first segment ending right of its start -- or, for an entry of
// <= 3 bp, the earliest of the <= 3 segments left of that one which already contains it within +-3.  A long entry always ends
// up at its own segment.  A short entry A that some segment i left of n(start) contains is contained in EVERY segment from i
// to n(start) and is counted at max(i, own of the entries that start in [End_i, start_A)) -- at most two positions.  Those are
// recorded per segment j in a small mask while the stream is read:
//   bit d (0..2)            a long entry starts at Position_j + d
//   bit 3 + 3 d + (len-1)   a short entry of that length starts at Position_j + d         (j = first segment with End > start)
// and the short entries themselves are deferred to a tiny second pass (depth_short_node).  What the reference's own source
// does not define -- entries with the SAME (chr, start), which its unstable std::sort may order either way -- is detected:
// *unstable is set when such a tie could move A, and A is counted as if it came first.
SQ_HD int32_t depth_short_own(const NodeTable &nt, int32_t chr, int32_t c0, int32_t n, int32_t start, int32_t len) {  // earliest containing segment left of n, else n
    for (int32_t j = (n - 3 > c0 ? n - 3 : c0); j < n; j++)
        if (depth_contained(nt, j, chr, start, len)) return j;
    return n;
}
// mask bit of an entry of ReadsOther; returns the segment j whose mask gets it (or -1: none needed)
SQ_HD int32_t depth_other_mark(const NodeTable &nt, int32_t chr, int32_t start, int32_t len, uint32_t *bit) {
    *bit = 0;
    if (chr < 0 || chr >= nt.n_ref) return -1;
    const ChrHead h = chr_head(nt, chr);
    const SegHit x = seg_first_end_gt(nt, h, start);
    const int32_t n = x.s;
    if (n >= h.c1) return -1;
    const int32_t d = start - x.pos;
    if (d < 0 || d > 2) return -1;
    if (len > kSeedThresh) *bit = 1u << d;
    else { const int32_t l = len < 1 ? 1 : len; *bit = 1u << (3 + 3 * d + (l - 1)); }
    return n;
}
// segment in which the short entry (chr, start, len <= 3) of ReadsOther is counted, or kNoNode
SQ_HD int32_t depth_short_node(const NodeTable &nt, const uint32_t *mask, int32_t chr, int32_t start, int32_t len, bool *unstable) {
    if (chr < 0 || chr >= nt.n_ref) return kNoNode;
    const ChrHead h = chr_head(nt, chr);
    const int32_t c0 = h.c0, c1 = h.c1;
    const int32_t n = seg_first_end_gt(nt, h, start).s;
    const int32_t i = depth_short_own(nt, chr, c0, n, start, len);
    if (i == n) return (n < c1 && depth_contained(nt, n, chr, start, len)) ? n : kNoNode;  // as a long entry: tested at n only
    int32_t at = i;
    const int32_t jmax = n < c1 ? n : c1 - 1;
    for (int32_t j = i + 1; j <= jmax; j++) {
        const uint32_t m = mask[j];
        if (!m) continue;
        for (int32_t d = 0; d <= 2; d++) {
            const int32_t b = nt.pos[j] + d;
            if (b > start) break;
            int32_t own = -1;  // largest own segment among the entries that start at b
            if ((m >> d) & 1u) own = j;
            for (int32_t l = 3; l >= 1 && own < j; l--)
                if ((m >> (3 + 3 * d + (l - 1))) & 1u) {
                    if (b == start && l == (len < 1 ? 1 : len)) continue;  // A itself (or its exact twins: same own segment)
                    const int32_t o = depth_short_own(nt, chr, c0, j, b, l);
                    if (o > own) own = o;
                }
            if (own < 0) continue;
            if (b < start) { if (own > at) at = own; }
            else if (own > at) *unstable = true;  // a tie at the same start that would move A if the sort put it first
        }
    }
    return at;
}

// ---- breakpoint coverage ------------------------------------------------------------------------

// Pass-3 record filter (:3136-3142): gate, then keep only the right-hand record of a same-chromosome pair.
SQ_HD bool cover_qualifies(uint8_t cls, uint16_t f, int32_t rid, int32_t pos, int32_t mrid, int32_t mpos) {
    if (!(cls & CLS_GATE)) return false;
    if (flag_mate_mapped(f) && mrid == rid) {
        if (mpos > pos) return false;
        if (mpos == pos && flag_second(f)) return false;
    }
    return true;
}
SQ_HD int32_t cover_start(uint16_t f, int32_t rid, int32_t pos, int32_t mrid, int32_t mpos) {  // :3148-3155
    return (flag_mate_mapped(f) && mrid == rid) ? mpos : pos;
}
SQ_HD uint64_t chrpos_key(int32_t chr, int32_t pos) { return ((uint64_t)(uint32_t)(chr + 1) << 32) | (uint32_t)pos; }
// indBP threshold (:3157): a qualifying record passes breakpoint (chr, pos) when its start key exceeds this key.  The reference
// compares `start > pos + Concord_Dist_Pos` as ints, so with a negative -dp near a chromosome start every record of that
// chromosome passes; the key then sits just below the chromosome's position 0 (cast to uint32, the negative sum would lie above
// every record of the chromosome and stall indBP).  Sums above INT32_MAX overflow in the reference itself and are not handled.
SQ_HD uint64_t cover_pass_key(int32_t chr, int32_t pos, int32_t dist) {
    const int64_t s = (int64_t)pos + dist;
    return s < 0 ? chrpos_key(chr, 0) - 1 : chrpos_key(chr, (int32_t)s);
}

// first index in [lo,hi) with a[i] >= v (uint64 keys)
SQ_HD int64_t lower_bound_u64(const uint64_t *a, int64_t lo, int64_t hi, uint64_t v) {
    while (lo < hi) {
        int64_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
SQ_HD int64_t upper_bound_u64(const uint64_t *a, int64_t lo, int64_t hi, uint64_t v) {
    while (lo < hi) {
        int64_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

}  // namespace sq
#endif
