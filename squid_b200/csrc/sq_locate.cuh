// Read-to-segment assignment and raw edge generation for one read.
// Reference behaviour: LocateRead (SegmentGraph.cpp:1207-1293), the -1 fallback scans
// (:1405-1421, :1610-1629), RawEdgesChim (:1394-1527) and RawEdgesOther (:1601-1686),
// IsDiscordant(Edge_t) (:159-190), Edge_t canonicalisation (BPEdge.h:31-52).
//
// The reference walks the node vector linearly from a hint that is carried block to block and
// read to read.  Here every scan is replaced by its closed form over the sorted segment table
// (two binary searches give the contiguous range [lo,hi] of segments a block fits in), which makes
// one read independent of all others EXCEPT when the outcome depends on the incoming hint.  Those
// reads are detected (`sensitive`) and replayed in stream order by a tiny second pass that knows
// the true hint.
#ifndef SQ_LOCATE_CUH
#define SQ_LOCATE_CUH
#include "sq_common.cuh"

namespace sq {

enum : int { MODE_OTHER = 0, MODE_CHIM = 1 };

SQ_HD uint64_t edge_key(int32_t i, bool hi_, int32_t j, bool hj) {  // Edge_t ctor + operator<
    if (i > j) { int32_t t = i; i = j; j = t; bool h = hi_; hi_ = hj; hj = h; }
    return ((uint64_t)(uint32_t)i << 33) | ((uint64_t)(uint32_t)j << 2) | ((uint64_t)hi_ << 1) | (uint64_t)hj;
}
SQ_HD void edge_unpack(uint64_t k, int32_t &i, bool &hi_, int32_t &j, bool &hj) {
    i = (int32_t)(k >> 33); j = (int32_t)((k >> 2) & 0x7fffffffu); hi_ = (k >> 1) & 1; hj = k & 1;
}
SQ_HD bool edge_is_discordant(const NodeTable &nt, const Params &p, uint64_t k) {  // :181-190
    int32_t i, j; bool h1, h2;
    edge_unpack(k, i, h1, j, h2);
    if (nt.chr[i] != nt.chr[j]) return true;
    if (nt.pos[j] - nt.end[i] > p.concord_dist_pos && j - i > p.concord_dist_idx) return true;
    return h1 != false || h2 != true;
}

SQ_HD bool block_fits(const NodeTable &nt, int32_t j, const Blk &b) {  // :1213
    return nt.chr[j] == b.ref_id && b.ref_pos >= nt.pos[j] - kLocateTol && b.ref_pos + b.match_ref <= nt.end[j] + kLocateTol;
}

// Cursor of LocateRead's running index `i`: a concrete index, or "whatever the hint is".
struct Cursor {
    int32_t idx;
    bool known;
};

// The segment j with its Position and End, read from the table.
SQ_HD SegHit seg_hit(const NodeTable &nt, int32_t j) { return SegHit{j, nt.pos[j], nt.end[j]}; }

// One iteration of LocateRead's per-block body.  Returns the segment with its Position and End (s == -1: none); updates `cur`.
// Sets *sensitive when the outcome cannot be decided without the concrete hint.
SQ_HD SegHit locate_block(const NodeTable &nt, const Blk &b, Cursor &cur, bool hint_known, int32_t hint, bool *sensitive) {
    const SegHit none{-1, 0, 0};
    // `if(i<0 || i>=vNodes.size()) i=initialguess;`
    if (cur.known && (cur.idx < 0 || cur.idx >= nt.n)) { cur.known = hint_known; cur.idx = hint; }
    if (cur.known && block_fits(nt, cur.idx, b)) return seg_hit(nt, cur.idx);
    const int32_t c = b.ref_id;
    if (c < 0 || c >= nt.n_ref) {  // no segment can fit; the scan direction still moves the cursor
        if (!cur.known) { return none; }
        cur.idx = (nt.chr[cur.idx] < c) ? nt.n : -1;
        return none;
    }
    const ChrHead h = chr_head(nt, c);
    if (!cur.known && h.c1 > h.c0 && b.match_ref > kLocateTol) {
        // the common case in closed form: the block lies inside the segment s that holds its start, clear of both ends
        // by more than the tolerance.  Then s is the only segment it fits (lo == hi == s below) and no scan can miss it.
        const SegHit s = seg_at(nt, h, b.ref_pos);
        if (s.pos <= b.ref_pos && b.ref_pos + kLocateTol < s.end && b.ref_pos + b.match_ref - kLocateTol <= s.end) { cur.known = true; cur.idx = s.s; return s; }
    }
    // segments that fit: lo = first with End >= p+m-5, hi = last with Position <= p+5
    const int32_t lo = seg_first_end_ge(nt, h, b.ref_pos + b.match_ref - kLocateTol);
    const int32_t hi = seg_last_pos_le(nt, h, b.ref_pos + kLocateTol);
    if (cur.known) {
        const int32_t i = cur.idx;
        const bool forward = nt.chr[i] < c || (nt.chr[i] == c && nt.pos[i] <= b.ref_pos);  // :1214
        if (forward) {
            const int32_t j = i > lo ? i : lo;
            if (lo <= hi && j <= hi) { cur.idx = j; return seg_hit(nt, j); }
            cur.idx = h.c1;  // ran off the chromosome to the right
            return none;
        }
        const int32_t j = i < hi ? i : hi;
        if (lo <= hi && j >= lo) { cur.idx = j; return seg_hit(nt, j); }
        cur.idx = h.c0 - 1;
        return none;
    }
    // unknown start index (it equals the hint): decidable only if every possible start agrees
    if (lo > hi) { cur.known = false; return none; }  // nothing fits; cursor ends off-chromosome on a side we do not know
    if (lo == hi) {
        // a start left of lo on the same chromosome whose Position is already > p scans backwards and misses
        const bool trap = lo - 1 >= h.c0 && nt.pos[lo - 1] > b.ref_pos;
        if (!trap) { cur.known = true; cur.idx = lo; return seg_hit(nt, lo); }
    }
    *sensitive = true;
    return none;
}

// Clip a block located in segment j (Position, End as the lookup returned them) to it, strand-aware (:1229-1248).
SQ_HD void trim_block(const SegHit &j, Blk &b) {
    if (b.ref_pos < j.pos) {
        const int32_t d = j.pos - b.ref_pos;
        if (!b.rev) b.read_pos += d;
        b.match_ref -= d; b.match_read -= d; b.ref_pos = j.pos;
    }
    if (b.ref_pos + b.match_ref > j.end) {
        const int32_t d = b.ref_pos + b.match_ref - j.end;
        if (b.rev) b.read_pos += d;
        b.match_ref -= d; b.match_read -= d;
    }
}

SQ_HD bool list_end_discordant(const Blk *v, int n) {  // ReadRec.cpp:178-209
    for (int k = 0; k + 1 < n; k++) {
        if (v[k].ref_id != v[k + 1].ref_id || v[k].rev != v[k + 1].rev) return true;
        const bool a = v[k].ref_pos < v[k + 1].ref_pos, r = v[k].read_pos < v[k + 1].read_pos;
        if (!v[k].rev && a != r) return true;
        if (v[k].rev && a == r) return true;
    }
    return false;
}

struct ReadView {
    Blk *F; int nF;   // FirstRead, sorted by read position
    Blk *S; int nS;   // SecondMate
    int32_t first_total, second_total;
};

SQ_HD bool read_pair_discordant_nocheck(const ReadView &rv) {  // IsPairDiscordant(false), ReadRec.cpp:211-228
    if (rv.nF == 0 || rv.nS == 0) return false;
    const Blk &ff = rv.F[0], &fb = rv.F[rv.nF - 1], &sf = rv.S[0], &sb = rv.S[rv.nS - 1];
    if (ff.ref_id != sb.ref_id || ff.rev == sb.rev) return true;
    if (!ff.rev && ff.ref_pos - ff.read_pos > sb.ref_pos - (rv.second_total - sb.read_pos - sb.match_read)) return true;
    if (!sf.rev && sf.ref_pos - sf.read_pos > fb.ref_pos - (rv.first_total - fb.read_pos - fb.match_read)) return true;
    return false;
}

// Segment index the "-1" fallback lands on (:1408-1409 / :1614-1615) when started from `ffi`.
// n0 = segment containing p.  The forward scan stops one segment early when p sits exactly on a
// boundary and the scan started at or left of that segment.
SQ_HD int32_t spanning_node(const NodeTable &nt, const Blk &b, bool ffi_known, int32_t ffi, bool *sensitive) {
    const ChrHead h = chr_head(nt, b.ref_id);
    const SegHit x = seg_at(nt, h, b.ref_pos);  // n0 = last segment with Position <= p, clamped to the first
    const int32_t n0 = x.s;
    if (x.pos == b.ref_pos && n0 - 1 >= h.c0) {
        if (!ffi_known) { *sensitive = true; return n0; }
        if (ffi <= n0 - 1) return n0 - 1;
    }
    return n0;
}

// Everything RawEdgesOther / RawEdgesChim do for one read.  `emit(key)` receives one weight-1 edge.
// node_out (size nF+nS) receives tmpRead_Node.  Blocks are trimmed in place.
// Returns false (and emits nothing) when the read is hint-sensitive and the hint is not known.
template <class Emit>
SQ_HD bool read_edges(const NodeTable &nt, const Params &p, ReadView &rv, int mode, bool record_is_first,
                      bool hint_known, int32_t hint, int32_t *node_out, Emit &emit) {
    const int n = rv.nF + rv.nS;
    bool sensitive = false;
    Cursor cur;
    cur.idx = hint; cur.known = hint_known;
    for (int k = 0; k < n; k++) {
        Blk &b = k < rv.nF ? rv.F[k] : rv.S[k - rv.nF];
        const SegHit j = locate_block(nt, b, cur, hint_known, hint, &sensitive);
        if (sensitive) return false;
        node_out[k] = j.s;
        if (j.s >= 0) trim_block(j, b);
    }
    // firstfrontindex after this read (:1402-1403, :1608-1609)
    bool ffi_known = hint_known;
    int32_t ffi = hint;
    if (n > 0 && node_out[0] != -1) { ffi_known = true; ffi = node_out[0]; }
    // pre-flight the -1 fallbacks so that nothing is emitted for a sensitive read
    for (int k = 0; k < n; k++)
        if (node_out[k] == -1) {
            const Blk &b = k < rv.nF ? rv.F[k] : rv.S[k - rv.nF];
            if (b.ref_id < 0 || b.ref_id >= nt.n_ref) continue;
            (void)spanning_node(nt, b, ffi_known, ffi, &sensitive);
            if (sensitive) return false;
        }
    for (int k = 0; k < n; k++)
        if (node_out[k] == -1) {  // block spans a segment boundary: edge (i,Tail)->(i+1,Head)
            const Blk &b = k < rv.nF ? rv.F[k] : rv.S[k - rv.nF];
            if (b.ref_id < 0 || b.ref_id >= nt.n_ref) continue;
            const int32_t i = spanning_node(nt, b, ffi_known, ffi, &sensitive);
            if (i + 1 < nt.n) emit(edge_key(i, false, i + 1, true));
        }
    for (int m = 0; m < 2; m++) {  // split junctions inside each mate
        const Blk *v = m ? rv.S : rv.F;
        const int cnt = m ? rv.nS : rv.nF, base = m ? rv.nF : 0;
        for (int k = 0; k + 1 < cnt; k++) {
            const int32_t i = node_out[base + k], j = node_out[base + k + 1];
            if (i != j && i != -1 && j != -1) emit(edge_key(i, v[k].rev, j, !v[k + 1].rev));
        }
    }
    // pair edge between the last block of each mate
    if ((mode == MODE_CHIM || record_is_first) && rv.nF > 0 && rv.nS > 0 &&
        !list_end_discordant(rv.F, rv.nF) && !list_end_discordant(rv.S, rv.nS)) {
        const int32_t i = node_out[rv.nF - 1], j = node_out[n - 1];
        bool overlap = false;
        for (int k = 0; k < rv.nF; k++) if (j == node_out[k]) overlap = true;
        for (int k = 0; k < rv.nS; k++) if (i == node_out[rv.nF + k]) overlap = true;
        const int32_t d = i > j ? i - j : j - i;
        if (rv.nF > 1 && d < 3) overlap = true;
        if (rv.nS > 1 && d < 3) overlap = true;
        if (i != j && i != -1 && j != -1 && !overlap) {
            const uint64_t key = edge_key(i, rv.F[rv.nF - 1].rev, j, rv.S[rv.nS - 1].rev);
            const bool disc = edge_is_discordant(nt, p, key);
            const bool pd = read_pair_discordant_nocheck(rv);
            if (mode == MODE_OTHER ? (pd == disc) : (!disc || pd)) emit(key);
        }
    }
    return true;
}

// ---- the concordant stream (RawEdgesOther) ---------------------------------------------------------------------------
// whetherbuildedge (:1601-1605)
template <class B>
SQ_HD bool conc_builds_edges(const B &b, const Params &p, int64_t r) {
    const uint32_t o = b.blk_off[r], nb = b.blk_off[r + 1] - o;
    if (nb == 0 || !has_mate_block(b.flag[r], b.mate_ref_id[r])) return true;
    int32_t front_rp = 0x7fffffff;
    for (uint32_t k = 0; k < nb; k++) { const int32_t rp = b.blk_read_pos[o + k]; if (rp < front_rp) front_rp = rp; }
    return front_rp <= 15 || (int32_t)b.lowphred_run[r] > p.max_lowphred_len;
}
SQ_HD Blk mate_block_of(uint16_t flag, int32_t mate_ref_id, int32_t mate_pos) {  // the synthetic 15-bp mate block (:306-314, 1588-1596)
    Blk x;
    x.ref_id = mate_ref_id; x.ref_pos = mate_pos; x.read_pos = 0; x.match_ref = kMateBlockLen; x.match_read = kMateBlockLen;
    x.rev = flag_mate_rev(flag);
    return x;
}
template <class B>
SQ_HD void conc_load_read(const B &b, int64_t r, ReadView &rv, bool &is_first) {
    is_first = flag_first(b.flag[r]);
    Blk *own = is_first ? rv.F : rv.S;
    Blk *oth = is_first ? rv.S : rv.F;
    const int no = load_sorted_blocks(b, r, own);
    int nm = 0;
    if (has_mate_block(b.flag[r], b.mate_ref_id[r])) oth[nm++] = mate_block_of(b.flag[r], b.mate_ref_id[r], b.mate_pos[r]);
    if (is_first) { rv.nF = no; rv.nS = nm; rv.first_total = b.total_len[r]; rv.second_total = 0; }
    else { rv.nS = no; rv.nF = nm; rv.second_total = b.total_len[r]; rv.first_total = 0; }
}

// read_edges(MODE_OTHER, hint unknown) for a record with at most ONE own block -- nine records out of ten -- with
// everything in registers: the lists are [own] and [mate], so there are no split junctions and at most one pair edge.
// Returns -3 when the read is hint-sensitive (nothing emitted), else tmpRead_Node[0] (>= -1).  n = #blocks must be > 0.
template <class Emit>
SQ_HD int32_t read_edges_single(const NodeTable &nt, const Params &p, bool has_own, Blk own, bool has_mate, Blk mate, bool is_first,
                                int32_t own_total, Emit &emit) {
    const bool hasF = is_first ? has_own : has_mate, hasS = is_first ? has_mate : has_own;
    Blk A = hasF ? (is_first ? own : mate) : (is_first ? mate : own);  // first block in FirstRead-then-SecondMate order
    Blk Bk = is_first ? mate : own;                                     // second one (when both lists are non-empty)
    const bool two = hasF && hasS;
    bool sensitive = false;
    Cursor cur;
    cur.idx = 0; cur.known = false;
    const SegHit hA = locate_block(nt, A, cur, false, 0, &sensitive);
    if (sensitive) return -3;
    const int32_t jA = hA.s;
    if (jA >= 0) trim_block(hA, A);
    int32_t jB = -1;
    if (two) {
        const SegHit hB = locate_block(nt, Bk, cur, false, 0, &sensitive);
        if (sensitive) return -3;
        jB = hB.s;
        if (jB >= 0) trim_block(hB, Bk);
    }
    const bool ffi_known = jA != -1;  // firstfrontindex after this read (:1608-1609); the incoming one is not known
    const int32_t ffi = jA;
    const bool spanA = jA == -1 && A.ref_id >= 0 && A.ref_id < nt.n_ref, spanB = two && jB == -1 && Bk.ref_id >= 0 && Bk.ref_id < nt.n_ref;
    int32_t iA = 0, iB = 0;
    if (spanA) { iA = spanning_node(nt, A, ffi_known, ffi, &sensitive); if (sensitive) return -3; }
    if (spanB) { iB = spanning_node(nt, Bk, ffi_known, ffi, &sensitive); if (sensitive) return -3; }
    if (spanA && iA + 1 < nt.n) emit(edge_key(iA, false, iA + 1, true));
    if (spanB && iB + 1 < nt.n) emit(edge_key(iB, false, iB + 1, true));
    if (is_first && two && jA != jB && jA != -1 && jB != -1) {  // pair edge; F = [A] (own), S = [Bk] (mate)
        const uint64_t key = edge_key(jA, A.rev, jB, Bk.rev);
        const bool disc = edge_is_discordant(nt, p, key);
        bool pd;  // IsPairDiscordant(false) on the trimmed blocks, first_total = own_total, second_total = 0
        if (A.ref_id != Bk.ref_id || A.rev == Bk.rev) pd = true;
        else if (!A.rev && A.ref_pos - A.read_pos > Bk.ref_pos - (0 - Bk.read_pos - Bk.match_read)) pd = true;
        else if (!Bk.rev && Bk.ref_pos - Bk.read_pos > A.ref_pos - (own_total - A.read_pos - A.match_read)) pd = true;
        else pd = false;
        if (pd == disc) emit(key);
    }
    return jA;
}

}  // namespace sq
#endif
