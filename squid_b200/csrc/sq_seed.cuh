// Seed-segment state machine of BuildNode_STAR, restated event-driven and island-parallel.
//
// The reference (SegmentGraph.cpp:296-701) steps through every concordant alignment and keeps
// per-record state.  All of that state is either (a) a pure function of the sorted discordant
// blocks (the discordant groups and their right ends), (b) a prefix scan over the record stream
// (otherrightmost, the duplicate filter), or (c) only observable when a discordant group is
// processed.  So the stream itself is handled by data-parallel kernels (classify, scans,
// compaction of the few "coverage gap" records) and this machine runs once per discordant GROUP:
//   1. apply, lazily, what the records since the previous group did to the machine state
//      (close a pending segment at the first 0-coverage record, clear or trim the cluster windows);
//   2. run the per-group segmentation rules literally (SegmentGraph.cpp:353-612).
// ConcordantCluster / PartialAlignCluster are not materialised: they are index windows over the
// record stream (class bits CLS_CONC / CLS_PART).  Every "count the window entries that span x"
// loop of the reference is answered from the sorted stream by binary search on position (entries
// whose first kept block does not start at the record position are rare and kept in a side list).
// ConcordRest is a set, queried from a small position-sorted table of candidate blocks.
//
// ISLANDS.  A 0-coverage record empties both windows and closes the pending segment
// (:616-636); if it also lies more than ReadLen+70 bp left of the next group (or on another
// chromosome) nothing of the earlier state can influence that group except (Chr, End) of the last
// emitted segment, which is then known to be "far left".  Groups between two such cuts form an
// island; islands run in parallel, each emitting a list of SeedOps that is stitched in order.
#ifndef SQ_SEED_CUH
#define SQ_SEED_CUH
#include "sq_common.cuh"

namespace sq {

struct DiscBlock {  // bamdiscordant element (+1 zeroed sentinel at the end, SURVEY App. A-5)
    int32_t chr, pos, len;
    int32_t rev;
};
struct Group {      // discordant group [ds,de) with its chained right end (:341-348)
    int32_t ds, de, chr, right;
};
struct SeedNode {
    int32_t chr, pos, len;
};
struct SeedOp {    // seed-segment emission of one island
    int32_t kind;  // 0: push (chr,pos,len)
                   // 1: the last segment emitted before this island, if on chr, gets End = pos+len; otherwise push (chr,pos,len)
                   // 2: the current last segment gets End = pos
    int32_t chr, pos, len;
};
struct RestBlock {  // ConcordRest candidate: non-first block of a concordant record; the table is ordered by owning group
    int32_t chr, pos, end, rec;
};
constexpr int32_t kIslandSlack = 70;  // > thresh*20 + 2*thresh, see island_cut()

struct SeedInputs {
    DevBatch b;
    const uint8_t *cls;
    const uint16_t *first_len;      // per CLS_CONC record: length of its first kept block (65535: look at the block arrays)
    const int32_t *gap_rec; int32_t n_gap;  // kept records preceded by a concordant-coverage gap, ascending
    const uint64_t *gap_other;      // per gap record: otherChr/otherrightmost before the record ((chr+1)<<32|pos)
    const int32_t *pc_rec; int32_t n_pc;    // records with CLS_PART, ascending
    const int32_t *dp_rec; int32_t n_dp;    // CLS_CONC records whose first kept block does not start at the record position
    int32_t lmax;                           // max first-block length over CLS_CONC records
    int64_t n_rec;
    const DiscBlock *D; int32_t nD;
    const Group *G; int32_t nG;
    const int64_t *trigger;         // per group: first kept record past its right end, or n_rec
    const int32_t *Pchr, *Ppos; int32_t nP;  // PartAlignPos sorted
    const RestBlock *rest; const uint32_t *rest_g; int32_t n_rest;  // ConcordRest candidates binned by the group they can matter to (rest_g ascending)
    int32_t read_len;
    int64_t first_kept;
    unsigned long long *win_count = nullptr;  // (device) total number of window records the groups looked at: the machine's algorithmic input
    // range shard of one genome: groups before g_lo belong to earlier shards; when a later shard follows, the record right
    // after this batch is a 0-coverage record for the pending group (the shard planner guarantees it, sqg_plan_shards)
    int32_t g_lo = 0;
    int32_t g_hi = 0;               // groups from g_hi on are never triggered by this batch (trigger == n_rec): islands cover [g_lo, g_hi)
    bool has_next = false;
    uint64_t end_other = 0;         // otherChr/otherrightmost after the last record of the batch
    const int32_t *ccmax = nullptr; int32_t cc_tile = 0;  // per tile of cc_tile records: maximum end of its ConcordantCluster entries (sq_classify.cuh)
    int32_t dense_max_r = 0;        // > 0: sub-clusters whose margins span at most this many positions use position-indexed tables
};

struct SeedState {
    int64_t offCC;   // record-index cursor of the ConcordantCluster window
    int32_t offPC;   // cursor into pc_rec
    int32_t markedStart, markedChr;
    int32_t backChr, backEnd;
    int32_t n_out;
    int32_t last_kind;
    bool have_back;
    bool back_inherited;  // the last segment belongs to an earlier island (far left of everything here)
};

// Cooperation policy: how many lanes step one island together.  All lanes keep identical scalar
// state; only the marked loops are split across lanes and recombined with the reductions below.
struct CoopSerial {  // one lane (CPU stepping harness, tiny islands)
    static SQ_HD int lane() { return 0; }
    static SQ_HD int size() { return 1; }
    static SQ_HD int sum(int v) { return v; }
    static SQ_HD int max(int v) { return v; }
    static SQ_HD int min(int v) { return v; }
    static SQ_HD int excl_prefix_max(int v, int identity) { (void)v; return identity; }
    static SQ_HD int excl_prefix_sum(int v) { (void)v; return 0; }
    static SQ_HD void add(int32_t *p, int32_t v) { *p += v; }
    static SQ_HD void add_range(int32_t *diff, int32_t ja, int32_t jb, bool on) { if (on && ja < jb) { diff[ja] += 1; diff[jb] -= 1; } }
    static SQ_HD void sync() {}
    // unordered append: begin(cell, n) .. reserve(has, n, cell) per lane .. end(cell, n) leaves the new uniform count in n
    static SQ_HD void begin_append(int32_t *cell, int32_t n) { (void)cell; (void)n; }
    static SQ_HD int32_t reserve(bool has, int32_t &n, int32_t *cell) { (void)cell; const int32_t s = n; if (has) n++; return s; }
    static SQ_HD void end_append(int32_t *cell, int32_t &n) { (void)cell; (void)n; }
};
#if defined(__CUDACC__)
struct CoopWarp {  // 32 lanes of one warp
    static __device__ __forceinline__ int lane() { return threadIdx.x & 31; }
    static __device__ __forceinline__ int size() { return 32; }
    static __device__ __forceinline__ int sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
    static __device__ __forceinline__ int max(int v) { return __reduce_max_sync(0xffffffffu, v); }
    static __device__ __forceinline__ int min(int v) { return __reduce_min_sync(0xffffffffu, v); }
    static __device__ __forceinline__ int excl_prefix_max(int v, int identity) {
        const int l = threadIdx.x & 31;
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, v, d); if (l >= d && o > v) v = o; }
        const int e = __shfl_up_sync(0xffffffffu, v, 1);
        return l == 0 ? identity : e;
    }
    static __device__ __forceinline__ int excl_prefix_sum(int v) {
        const int l = threadIdx.x & 31;
        int incl = v;
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, incl, d); if (l >= d) incl += o; }
        return incl - v;
    }
    static __device__ __forceinline__ void add(int32_t *p, int32_t v) { atomicAdd(p, v); }
    // +1 at diff[ja], -1 at diff[jb] for the lanes with `on` (called by every lane of the warp): sorted input makes
    // neighbouring lanes hit the same two cells, so one lane per distinct index adds for its whole group
    static __device__ __forceinline__ void add_range(int32_t *diff, int32_t ja, int32_t jb, bool on) {
        on = on && ja < jb;
        const unsigned act = __ballot_sync(0xffffffffu, on);
        if (!on) return;
        const int l = threadIdx.x & 31;
        unsigned m = __match_any_sync(act, ja);
        if (l == __ffs(m) - 1) atomicAdd(&diff[ja], __popc(m));
        m = __match_any_sync(act, jb);
        if (l == __ffs(m) - 1) atomicAdd(&diff[jb], -__popc(m));
    }
    static __device__ __forceinline__ void sync() { __syncwarp(); }
    static __device__ __forceinline__ void begin_append(int32_t *cell, int32_t n) { (void)cell; (void)n; }
    static __device__ __forceinline__ int32_t reserve(bool has, int32_t &n, int32_t *cell) {  // lanes in lockstep: slots from a ballot
        (void)cell;
        const unsigned m = __ballot_sync(0xffffffffu, has);
        const int32_t s = n + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
        n += __popc(m);
        return s;
    }
    static __device__ __forceinline__ void end_append(int32_t *cell, int32_t &n) { (void)cell; (void)n; }
};
struct CoopBlock {  // every thread of the block (blockDim.x a multiple of 32): for the few islands with huge windows
    template <int OP> static __device__ __forceinline__ int reduce(int v, int identity) {
        __shared__ int wv[32];
        __shared__ int res;
        v = OP == 0 ? __reduce_add_sync(0xffffffffu, v) : (OP == 1 ? __reduce_max_sync(0xffffffffu, v) : __reduce_min_sync(0xffffffffu, v));
        if ((threadIdx.x & 31) == 0) wv[threadIdx.x >> 5] = v;
        __syncthreads();
        if (threadIdx.x < 32) {
            int x = threadIdx.x < (blockDim.x >> 5) ? wv[threadIdx.x] : identity;
            x = OP == 0 ? __reduce_add_sync(0xffffffffu, x) : (OP == 1 ? __reduce_max_sync(0xffffffffu, x) : __reduce_min_sync(0xffffffffu, x));
            if (threadIdx.x == 0) res = x;
        }
        __syncthreads();
        const int r = res;
        __syncthreads();
        return r;
    }
    static __device__ __forceinline__ int lane() { return threadIdx.x; }
    static __device__ __forceinline__ int size() { return blockDim.x; }
    static __device__ __forceinline__ int sum(int v) { return reduce<0>(v, 0); }
    static __device__ __forceinline__ int max(int v) { return reduce<1>(v, -2147483647 - 1); }
    static __device__ __forceinline__ int min(int v) { return reduce<2>(v, 2147483647); }
    static __device__ __forceinline__ int excl_prefix_max(int v, int identity) {
        __shared__ int wtot[32];
        const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
        int incl = v;
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, incl, d); if (l >= d && o > incl) incl = o; }
        int excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (l == 0) excl = identity;
        if (l == 31) wtot[w] = incl;
        __syncthreads();
        int base = identity;
        for (int k = 0; k < w; k++) if (wtot[k] > base) base = wtot[k];
        __syncthreads();
        return excl > base ? excl : base;
    }
    static __device__ __forceinline__ int excl_prefix_sum(int v) {
        __shared__ int wsum[32];
        const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
        int incl = v;
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, incl, d); if (l >= d) incl += o; }
        if (l == 31) wsum[w] = incl;
        __syncthreads();
        int base = 0;
        for (int k = 0; k < w; k++) base += wsum[k];
        __syncthreads();
        return base + incl - v;
    }
    static __device__ __forceinline__ void add(int32_t *p, int32_t v) { atomicAdd(p, v); }
    // +1 at diff[ja], -1 at diff[jb] for the lanes with `on` (called by every lane of the warp): sorted input makes
    // neighbouring lanes hit the same two cells, so one lane per distinct index adds for its whole group
    static __device__ __forceinline__ void add_range(int32_t *diff, int32_t ja, int32_t jb, bool on) {
        on = on && ja < jb;
        const unsigned act = __ballot_sync(0xffffffffu, on);
        if (!on) return;
        const int l = threadIdx.x & 31;
        unsigned m = __match_any_sync(act, ja);
        if (l == __ffs(m) - 1) atomicAdd(&diff[ja], __popc(m));
        m = __match_any_sync(act, jb);
        if (l == __ffs(m) - 1) atomicAdd(&diff[jb], -__popc(m));
    }
    static __device__ __forceinline__ void sync() { __syncthreads(); }
    // unordered append through a counter cell in the island's scratch (one atomic per warp)
    static __device__ __forceinline__ void begin_append(int32_t *cell, int32_t n) { __syncthreads(); if (threadIdx.x == 0) *cell = n; __syncthreads(); }
    static __device__ __forceinline__ int32_t reserve(bool has, int32_t &n, int32_t *cell) {
        (void)n;
        const unsigned m = __ballot_sync(0xffffffffu, has);
        if (!m) return 0;
        const int l = threadIdx.x & 31;
        int32_t base = 0;
        if (l == __ffs(m) - 1) base = atomicAdd(cell, __popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        return base + __popc(m & ((1u << l) - 1u));
    }
    static __device__ __forceinline__ void end_append(int32_t *cell, int32_t &n) { __syncthreads(); n = *(volatile int32_t *)cell; __syncthreads(); }
};
#endif

template <class W>
struct SeedMachineT {
    SeedInputs in;
    SeedState st;
    SeedOp *out; int32_t out_cap;
    int32_t *margin; int32_t margin_cap;
    int32_t *msearch = nullptr; int32_t msearch_cap = 0;  // fast (shared) memory for a copy of the sorted margins, if the caller has some
    const int32_t *ms = nullptr;                          // what the searches read: that copy, or margin itself
    int32_t error;  // 1: margin overflow, 2: output overflow

    // ---- entry accessors --------------------------------------------------------------------
    SQ_HD bool isCC(int64_t r) const { return (in.cls[r] & (CLS_CONC | CLS_PART)) == CLS_CONC; }
    SQ_HD bool isDispl(int64_t r) const { return in.cls[r] & CLS_DISPL; }
    SQ_HD int64_t nextCC(int64_t x, int64_t lim) const { while (x < lim && !isCC(x)) x++; return x < lim ? x : lim; }
    SQ_HD int32_t e_chr(int64_t r) const { return in.b.ref_id[r]; }
    // the first kept block of a window entry (a CLS_CONC record): its start is the record position unless the record is
    // displaced, its length sits in the side array phase 1 wrote -- two independent loads instead of blk_off -> block
    SQ_HD int32_t e_pos(int64_t r) const { return (in.cls[r] & CLS_DISPL) ? in.b.blk_ref_pos[in.b.blk_off[r]] : in.b.pos[r]; }
    SQ_HD int32_t e_len(int64_t r) const { const uint32_t l = in.first_len[r]; return l != 65535u ? (int32_t)l : in.b.blk_match_ref[in.b.blk_off[r]]; }
    SQ_HD int32_t e_readpos(int64_t r) const { return in.b.blk_read_pos[in.b.blk_off[r]]; }
    SQ_HD bool e_rev(int64_t r) const { return flag_rev(in.b.flag[r]); }

    // first record in [lo,hi) with (ref_id,pos) >= (c,x); unmapped records (ref_id -1) sort last
    SQ_HD int64_t lb_pos(int64_t lo, int64_t hi, int32_t c, int32_t x) const {
        while (lo < hi) {
            const int64_t m = lo + ((hi - lo) >> 1);
            const int32_t rc = in.b.ref_id[m];
            const bool less = rc >= 0 && (rc < c || (rc == c && in.b.pos[m] < x));
            if (less) lo = m + 1; else hi = m;
        }
        return lo;
    }
    SQ_HD int32_t lb_list(const int32_t *a, int32_t n, int64_t v) const {  // first i with a[i] >= v
        int32_t lo = 0, hi = n;
        while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (a[m] < v) lo = m + 1; else hi = m; }
        return lo;
    }
    // first index i in [lo,hi) of pc_rec whose record has (ref_id,pos) >= (c,x)
    SQ_HD int32_t lb_pc_pos(int32_t lo, int32_t hi, int32_t c, int32_t x) const {
        while (lo < hi) {
            const int32_t m = (lo + hi) >> 1;
            const int64_t r = in.pc_rec[m];
            const int32_t rc = in.b.ref_id[r];
            if (rc < c || (rc == c && in.b.pos[r] < x)) lo = m + 1; else hi = m;
        }
        return lo;
    }

    // ---- output ------------------------------------------------------------------------------
    SQ_HD void emit(int32_t kind, int32_t chr, int32_t pos, int32_t len) {
        if (st.n_out >= out_cap) { error = 2; return; }
        if (W::lane() == 0) { out[st.n_out].kind = kind; out[st.n_out].chr = chr; out[st.n_out].pos = pos; out[st.n_out].len = len; }
        st.last_kind = kind;
        st.n_out++;
    }
    SQ_HD void push_node(int32_t chr, int32_t pos, int32_t len) {
        emit(0, chr, pos, len);
        st.have_back = true; st.back_inherited = false; st.backChr = chr; st.backEnd = pos + len;
    }
    SQ_HD void set_back_end(int32_t e) {  // vNodes.back().Length += e - Position - Length
        if (st.n_out > 0 && st.last_kind == 0) { if (W::lane() == 0) out[st.n_out - 1].len += e - st.backEnd; }
        else emit(2, st.backChr, e, 0);
        st.backEnd = e;
    }
    SQ_HD int32_t mcap() const { return (margin_cap - 8) / 6; }     // six regions + 8 reserved cells at the end of the scratch
    SQ_HD int32_t *cell(int k) const { return margin + (margin_cap - 8) + k; }
    bool use_dense = false;   // set by the caller: every island on the device; the CPU stepping harness chooses
    int32_t n_dense = 0, n_sparse = 0;  // sub-clusters tabulated by position / through the sorted margins (statistics)
    // first index i in [lo,hi) with pred(i), else hi; the lanes split the range, the result is uniform
    template <class F> SQ_HD int32_t find_first(int32_t lo, int32_t hi, F pred) const {
        for (int32_t base = lo; base < hi; base += W::size()) {
            const int32_t i = base + W::lane();
            const int32_t m = W::min((i < hi && pred(i)) ? i : 0x7fffffff);
            if (m != 0x7fffffff) return m;
        }
        return hi;
    }
    SQ_HD void push_margin(int32_t &n, int32_t v) {  // uniform call: every lane counts, lane 0 stores
        if (n + 1 >= mcap()) { error = 1; return; }
        if (W::lane() == 0) margin[n] = v;
        n++;
    }
    // values only, so any correct sort agrees with std::sort: bitonic network over the next power of two,
    // compare-exchanges split across the lanes (the scratch is sized for the padding)
    SQ_HD void sort_margins(int32_t n) {
        int32_t m = 1;
        while (m < n) m <<= 1;
        if (m > mcap()) { error = 1; return; }
        W::sync();
        for (int32_t i = n + W::lane(); i < m; i += W::size()) margin[i] = 0x7fffffff;
        W::sync();
        for (int32_t k = 2; k <= m; k <<= 1)
            for (int32_t j = k >> 1; j > 0; j >>= 1) {
                for (int32_t i = W::lane(); i < m; i += W::size()) {
                    const int32_t l = i ^ j;
                    if (l > i) {
                        const int32_t a = margin[i], c = margin[l];
                        const bool up = (i & k) == 0;
                        if ((a > c) == up) { margin[i] = c; margin[l] = a; }
                    }
                }
                W::sync();
            }
    }

    SQ_HD void init(bool inherited_back) {
        st.offCC = 0; st.offPC = 0; st.markedStart = -1; st.markedChr = -1;
        st.have_back = inherited_back; st.back_inherited = inherited_back;
        st.backChr = -2; st.backEnd = -(1 << 30); st.n_out = 0; st.last_kind = -1; error = 0;
    }

    // (curChr, currightmost) and the 0-coverage test of :616-620 for gap record k while a group starting at (sChr,sPos) is pending
    SQ_HD bool is0(int32_t k, int32_t dChr, int32_t dRight, int32_t sChr, int32_t sPos, int32_t *curChr, int32_t *curRight) const {
        const int64_t r = in.gap_rec[k];
        const uint64_t ok = in.gap_other[k];
        const int32_t oChr = (int32_t)(ok >> 32) - 1, oRight = (int32_t)(uint32_t)ok;
        const int32_t cr = (dChr > oChr || (dChr == oChr && dRight > oRight)) ? dRight : oRight;
        const int32_t cc = dChr > oChr ? dChr : oChr;
        *curChr = cc; *curRight = cr;
        const int32_t rl = in.read_len;
        return (in.b.ref_id[r] != cc || in.b.pos[r] > cr + rl) && (cc < sChr || (cc == sChr && cr + rl < sPos));
    }
    // last 0-coverage record among the kept records of [r_lo, r_hi); -1 if none
    SQ_HD int32_t last_is0(int64_t r_lo, int64_t r_hi, int32_t dChr, int32_t dRight, int32_t sChr, int32_t sPos, int32_t *cc, int32_t *cr) const {
        if (r_hi <= r_lo) return -1;
        const int32_t a = lb_list(in.gap_rec, in.n_gap, r_lo), bnd = lb_list(in.gap_rec, in.n_gap, r_hi);
        for (int32_t k = bnd - 1; k >= a; k--) if (is0(k, dChr, dRight, sChr, sPos, cc, cr)) return k;
        return -1;
    }
    // May the machine be restarted at group g (g >= 1)?  Yes when the records between the triggers of g-1 and g
    // contain a 0-coverage record z (windows emptied, pending segment closed) and every segment emitted so far
    // ends at most currightmost(z)+3, i.e. more than 60 bp left of the leftmost position group g can look at
    // (group start - ReadLen, from the PartAlignPos window) -- or lies on another chromosome.
    SQ_HD bool island_cut(int32_t g) const {
        const int64_t r_lo = in.trigger[g - 1], r_hi = in.trigger[g];
        if (r_hi >= in.n_rec || r_hi <= r_lo) return false;
        const Group gp = in.G[g - 1], gn = in.G[g];
        int32_t cc, cr;
        const int32_t z = last_is0(r_lo, r_hi, gp.chr, gp.right, gn.chr, in.D[gn.ds].pos, &cc, &cr);
        if (z < 0) return false;
        return cc != gn.chr || (int64_t)in.D[gn.ds].pos - cr > (int64_t)in.read_len + kIslandSlack;
    }

    // skip-prefix of the :637-646 trims: first entry index >= x (below `lim`) that is not skipped
    SQ_HD int64_t trim_cc(int64_t x, int64_t lim, int32_t lchr, int32_t sChr) const {
        if (x >= lim) return lim;
        if (lchr < sChr) return lim;                     // every visible entry is on a chromosome before the pending group
        int64_t y = lb_pos(x, lim, lchr, -(1 << 30));    // entries on earlier chromosomes
        if (st.have_back && st.backChr == lchr) {
            int64_t j = lb_pos(y, lim, lchr, st.backEnd);  // non-displaced entries left of the last segment's end
            // a displaced entry (block start != record position) inside [y,j) that is not left of backEnd stops the skip
            for (int32_t k = lb_list(in.dp_rec, in.n_dp, y); k < in.n_dp && in.dp_rec[k] < j; k++) {
                const int64_t r = in.dp_rec[k];
                if (isCC(r) && e_pos(r) >= st.backEnd) { j = r; break; }
            }
            // ... and displaced entries at/after j that ARE left of backEnd are skipped too
            y = j;
            for (;;) {
                y = nextCC(y, lim);
                if (y < lim && e_chr(y) == lchr && e_pos(y) < st.backEnd) { y++; continue; }
                break;
            }
        }
        return nextCC(y, lim);
    }
    SQ_HD int32_t trim_pc(int32_t x, int32_t lim, int32_t lchr, int32_t sChr) const {
        while (x < lim) {
            const int64_t r = in.pc_rec[x];
            const int32_t c = e_chr(r);
            if (c != lchr || c < sChr || (st.have_back && c == st.backChr && e_pos(r) < st.backEnd)) { x++; continue; }
            break;
        }
        return x;
    }

    // :621-630 at a 0-coverage record whose (curChr, currightmost) is (cc, cr)
    SQ_HD void close_marked_gap(int32_t cc, int32_t cr) {
        if (st.markedStart == -1) return;
        if (cc == st.markedChr && cr > st.markedStart && cr - st.markedStart < kSeedThresh * 20 && st.have_back && st.markedStart == st.backEnd)
            set_back_end(st.backEnd + (cr - st.markedStart));
        else if (cc == st.markedChr && cr > st.markedStart && cr - st.markedStart >= kSeedThresh * 20)
            push_node(st.markedChr, st.markedStart, cr - st.markedStart);
        st.markedStart = -1; st.markedChr = -1;
    }

    // Lazy replay of steps :616-646 for the kept records in [r_lo, r_hi) while the group starting at (sChr,sPos) is pending.
    SQ_HD void replay_between(int64_t r_lo, int64_t r_hi, int32_t dChr, int32_t dRight, int32_t sChr, int32_t sPos, bool do_trim) {
        if (r_hi <= r_lo) return;
        const int32_t a = lb_list(in.gap_rec, in.n_gap, r_lo), bnd = lb_list(in.gap_rec, in.n_gap, r_hi);
        int32_t cc, cr;
        int32_t f = -1, z = -1;
        for (int32_t k = a; k < bnd; k++) if (is0(k, dChr, dRight, sChr, sPos, &cc, &cr)) { f = k; break; }
        if (f >= 0) {
            close_marked_gap(cc, cr);
            if (!do_trim) return;
            for (int32_t k = bnd - 1; k >= f; k--) if (is0(k, dChr, dRight, sChr, sPos, &cc, &cr)) { z = k; break; }
            const int64_t zr = in.gap_rec[z];
            st.offCC = zr;  // :633-636 at record z: both windows emptied; z's own block is pushed afterwards
            st.offPC = lb_list(in.pc_rec, in.n_pc, zr);
            r_lo = zr + 1;
        }
        if (!do_trim) return;
        // :637-646 for the kept records in [r_lo, r_hi): a prefix skip whose predicate is that of the LAST kept record
        int64_t last = r_hi - 1;
        while (last >= r_lo && !(in.cls[last] & CLS_KEEP)) last--;
        if (last < r_lo) return;
        const int32_t lchr = in.b.ref_id[last];
        // entries visible to that record are those pushed before it, i.e. from records < last
        const int64_t x = trim_cc(st.offCC, last, lchr, sChr);
        if (x > st.offCC) st.offCC = x;
        const int32_t y = trim_pc(st.offPC, lb_list(in.pc_rec, in.n_pc, last), lchr, sChr);
        if (y > st.offPC) st.offPC = y;
    }

    // number of ConcordantCluster + PartialAlignCluster window entries spanning brk +- thresh (:457-469); lanes split the ranges
    SQ_HD int32_t window_coverage(int32_t chrG, int32_t brk, int64_t rg, int32_t szPC) const {
        const int32_t thresh = kSeedThresh;
        int32_t cov = 0;
        // an entry spans iff pos < brk-thresh and pos+len >= brk+thresh, hence pos in [brk+thresh-lmax, brk-thresh)
        const int32_t pmin = brk + thresh - in.lmax, pmax = brk - thresh;
        if (st.offCC < rg) {
            const int64_t lo = lb_pos(st.offCC, rg, chrG, pmin), hi = lb_pos(lo, rg, chrG, pmax);
            for (int64_t r = lo + W::lane(); r < hi; r += W::size())
                if (isCC(r) && !isDispl(r) && in.b.ref_id[r] == chrG) {
                    const int32_t p0 = e_pos(r);
                    if (p0 + e_len(r) >= brk + thresh && p0 < pmax) cov++;
                }
        }
        if (st.offPC < szPC) {
            const int32_t lo = lb_pc_pos(st.offPC, szPC, chrG, pmin), hi = lb_pc_pos(lo, szPC, chrG, pmax);
            for (int32_t i = lo + W::lane(); i < hi; i += W::size()) {
                const int64_t r = in.pc_rec[i];
                if (!isDispl(r) && in.b.ref_id[r] == chrG) {
                    const int32_t p0 = e_pos(r);
                    if (p0 + e_len(r) >= brk + thresh && p0 < pmax) cov++;
                }
            }
        }
        // displaced entries of either window
        const int64_t w0 = st.offCC < rg ? st.offCC : rg;
        const int64_t wp = st.offPC < szPC ? (int64_t)in.pc_rec[st.offPC] : rg;
        const int32_t k0 = lb_list(in.dp_rec, in.n_dp, w0 < wp ? w0 : wp), k1 = lb_list(in.dp_rec, in.n_dp, rg);
        for (int32_t k = k0 + W::lane(); k < k1; k += W::size()) {
            const int64_t r = in.dp_rec[k];
            if (in.b.ref_id[r] != chrG) continue;
            const bool part = in.cls[r] & CLS_PART;
            if (part ? (r < wp) : (r < st.offCC)) continue;
            const int32_t p0 = e_pos(r);
            if (p0 + e_len(r) >= brk + thresh && p0 < pmax) cov++;
        }
        return W::sum(cov);
    }

    // The ConcordRest candidates of group g: a block that starts in [start_g - ReadLen, right_g + ReadLen) belongs to g alone (the
    // next group starts at least ReadLen right of right_g), and nothing a break of g looks at starts outside that range.
    SQ_HD void rest_range(int32_t g, int32_t *lo_out, int32_t *hi_out) const {
        int32_t lo = 0, hi = in.n_rest;
        while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (in.rest_g[m] < (uint32_t)g) lo = m + 1; else hi = m; }
        int32_t lo2 = lo, hi2 = in.n_rest;
        while (lo2 < hi2) { const int32_t m = (lo2 + hi2) >> 1; if (in.rest_g[m] <= (uint32_t)g) lo2 = m + 1; else hi2 = m; }
        *lo_out = lo; *hi_out = lo2;
    }
    // :420-434 for one PartialAlignCluster entry: the margin position it contributes, if any
    SQ_HD bool pc_margin_value(int64_t r, int32_t chrG, int32_t m0, int32_t curEndPos, int32_t *v) const {
        const int32_t thresh = kSeedThresh;
        if (e_chr(r) != chrG) return false;
        const int32_t p0 = e_pos(r), p1 = p0 + e_len(r);
        const bool rv = e_rev(r);
        if (e_readpos(r) > 15 && p0 > m0 - thresh && p0 < curEndPos + thresh) {
            if (rv && p1 > m0 - thresh && p1 < curEndPos + thresh) { *v = p1; return true; }
            if (!rv) { *v = p0; return true; }
            return false;
        }
        if (rv && p0 > m0 - thresh && p0 < curEndPos + thresh) { *v = p0; return true; }
        if (!rv && p1 > m0 - thresh && p1 < curEndPos + thresh) { *v = p1; return true; }
        return false;
    }
    // Lanes split the candidate list [lo,hi) of `list` (pc_rec or dp_rec indices); the margins are sorted (or histogrammed)
    // afterwards, so only the multiset matters: unordered append.  `from_dp`: take displaced PART entries (dp list) /
    // non-displaced entries (pc list).
    SQ_HD void pc_margins(const int32_t *list, int32_t lo, int32_t hi, bool from_dp, int32_t chrG, int32_t m0, int32_t curEndPos, int32_t &nM) {
        if (hi <= lo) return;
        const int32_t cap = mcap() - 1;
        W::begin_append(cell(0), nM);
        for (int32_t base = lo; base < hi; base += W::size()) {
            const int32_t i = base + W::lane();
            int32_t v = 0;
            bool has = false;
            if (i < hi) {
                const int64_t r = list[i];
                const uint8_t c = in.cls[r];
                if (from_dp ? (c & CLS_PART) != 0 : !(c & CLS_DISPL)) has = pc_margin_value(r, chrG, m0, curEndPos, &v);
            }
            const int32_t at = W::reserve(has, nM, cell(0));
            if (has && at < cap) margin[at] = v;
        }
        W::end_append(cell(0), nM);
        if (nM >= cap) error = 1;
    }

    // ---- per-break tables ------------------------------------------------------------------------------------------
    // For every entry of the sorted MarginPositions array the break loop (:440-504) needs srsupport, peleftfor,
    // perightrev, the spanning coverage of the windows + discordant blocks, and the ConcordRest coverage.  None of them
    // depends on what the loop emits, so they are tabulated up front: interval-shaped contributions go into difference
    // arrays (two binary searches in the margin array each) that are prefix-summed, instead of rescanning the window
    // for each candidate break.
    SQ_HD int32_t m_upper(int32_t nM, int32_t v) const {  // first index with margin > v
        int32_t lo = 0, hi = nM;
        while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (ms[m] <= v) lo = m + 1; else hi = m; }
        return lo;
    }
    SQ_HD int32_t m_lower(int32_t nM, int32_t v) const {  // first index with margin >= v
        int32_t lo = 0, hi = nM;
        while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (ms[m] < v) lo = m + 1; else hi = m; }
        return lo;
    }
    SQ_HD void add_range(int32_t *diff, int32_t ja, int32_t jb) { if (ja < jb) { W::add(&diff[ja], 1); W::add(&diff[jb], -1); } }
    // a block [p0,p1) spans break b iff p0 < b-thresh and p1 >= b+thresh  <=>  p0+thresh < b <= p1-thresh
    SQ_HD void add_span(int32_t *diff, int32_t nM, int32_t p0, int32_t p1) { add_range(diff, m_upper(nM, p0 + kSeedThresh), m_upper(nM, p1 - kSeedThresh)); }
    // U independent searches stepped together (the loads of one step do not depend on each other)
    template <int U>
    SQ_HD void m_upper_n(int32_t nM, const int32_t *v, int32_t *res) const {
        int32_t lo[U], hi[U];
#pragma unroll
        for (int u = 0; u < U; u++) { lo[u] = 0; hi[u] = nM; }
        for (int32_t span = nM; span > 0; span >>= 1) {
#pragma unroll
            for (int u = 0; u < U; u++)
                if (lo[u] < hi[u]) { const int32_t m = (lo[u] + hi[u]) >> 1; if (ms[m] <= v[u]) lo[u] = m + 1; else hi[u] = m; }
        }
#pragma unroll
        for (int u = 0; u < U; u++) res[u] = lo[u];
    }
    // add_span for the first kept blocks of up to U window records r0 + u*stride (u < U, r < hi) that satisfy `want`
    // (class bits: value after masking with CONC|PART|DISPL), on chromosome chrG
    template <int U>
    SQ_HD void add_span_records(int32_t *diff, int32_t nM, int64_t r0, int64_t stride, int64_t hi, uint8_t want, int32_t chrG) {
        uint8_t c[U]; uint32_t fl[U]; int32_t rc[U], ps[U];
#pragma unroll
        for (int u = 0; u < U; u++) {  // all loads of all records independent of each other (`want` excludes displaced records)
            const int64_t r = r0 + u * stride;
            const bool inr = r < hi;
            c[u] = inr ? in.cls[r] : (uint8_t)0; fl[u] = inr ? in.first_len[r] : 0u; rc[u] = inr ? in.b.ref_id[r] : -1; ps[u] = inr ? in.b.pos[r] : 0;
        }
        bool ok[U]; int32_t v[2 * U], j[2 * U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            ok[u] = (c[u] & (CLS_CONC | CLS_PART | CLS_DISPL)) == want && rc[u] == chrG;
            const int32_t p0 = ps[u];
            int32_t l = (int32_t)fl[u];
            if (ok[u] && fl[u] == 65535u) l = in.b.blk_match_ref[in.b.blk_off[r0 + u * stride]];
            v[2 * u] = p0 + kSeedThresh; v[2 * u + 1] = p0 + l - kSeedThresh;
        }
        m_upper_n<2 * U>(nM, v, j);
#pragma unroll
        for (int u = 0; u < U; u++) W::add_range(diff, j[2 * u], j[2 * u + 1], ok[u]);
    }
    SQ_HD void scan_inplace(int32_t *a, int32_t n) {
        W::sync();
        int32_t carry = 0;
        for (int32_t base = 0; base < n; base += W::size()) {
            const int32_t i = base + W::lane();
            const int32_t v = i < n ? a[i] : 0;
            const int32_t ex = W::excl_prefix_sum(v);
            if (i < n) a[i] = carry + ex + v;
            carry += W::sum(v);
        }
        W::sync();
    }
    SQ_HD void tabulate_breaks(int32_t g, int32_t nM, int32_t ds, int32_t de, int32_t chrG, int32_t sPos, int64_t rg, int32_t szPC) {
        const int32_t thresh = kSeedThresh, RL = in.read_len, cap = mcap();
        int32_t *t_sr = margin + cap, *t_pl = margin + 2 * cap, *t_pr = margin + 3 * cap, *t_cov = margin + 4 * cap, *t_rest = margin + 5 * cap;
        const DiscBlock *D = in.D;
        W::sync();
        for (int32_t i = W::lane(); i <= nM; i += W::size()) { t_pl[i] = 0; t_pr[i] = 0; t_cov[i] = 0; t_rest[i] = 0; }
        for (int32_t i = W::lane(); i < nM; i += W::size()) {  // srsupport: margins within +-thresh (:445-448)
            const int32_t brk = ms[i];
            t_sr[i] = m_lower(nM, brk + thresh) - m_upper(nM, brk - thresh);
        }
        W::sync();
        for (int32_t k = ds + W::lane(); k < de; k += W::size()) {
            const int32_t p0 = D[k].pos, p1 = p0 + D[k].len;
            if (!D[k].rev) add_range(t_pl, m_upper(nM, p1), m_lower(nM, p1 + RL));        // end < b < end+ReadLen   (:450)
            else add_range(t_pr, m_upper(nM, p0 - RL), m_lower(nM, p0));                // pos-ReadLen < b < pos   (:452)
            if (D[k].chr == chrG) add_span(t_cov, nM, p0, p1);                            // :462-464
        }
        const int32_t bmin = ms[0], bmax = ms[nM - 1];
        const int32_t pmin = bmin + thresh - in.lmax, pmax = bmax - thresh;  // block starts that can span some break
        if (st.offCC < rg) {  // ConcordantCluster window (:457-461)
            const int64_t lo = lb_pos(st.offCC, rg, chrG, pmin), hi = lb_pos(lo, rg, chrG, pmax);
            constexpr int U = 4;
            for (int64_t base = lo; base < hi; base += (int64_t)W::size() * U)
                add_span_records<U>(t_cov, nM, base + W::lane(), W::size(), hi, CLS_CONC, chrG);
        }
        if (st.offPC < szPC) {  // PartialAlignCluster window (:465-469)
            const int32_t lo = lb_pc_pos(st.offPC, szPC, chrG, pmin), hi = lb_pc_pos(lo, szPC, chrG, pmax);
            for (int32_t base = lo; base < hi; base += W::size()) {
                const int32_t i = base + W::lane();
                bool on = false;
                int32_t ja = 0, jb = 0;
                if (i < hi) {
                    const int64_t r = in.pc_rec[i];
                    if (!isDispl(r) && in.b.ref_id[r] == chrG) { on = true; const int32_t p0 = e_pos(r); ja = m_upper(nM, p0 + kSeedThresh); jb = m_upper(nM, p0 + e_len(r) - kSeedThresh); }
                }
                W::add_range(t_cov, ja, jb, on);
            }
        }
        {   // displaced entries of either window
            const int64_t w0 = st.offCC < rg ? st.offCC : rg;
            const int64_t wp = st.offPC < szPC ? (int64_t)in.pc_rec[st.offPC] : rg;
            const int32_t k0 = lb_list(in.dp_rec, in.n_dp, w0 < wp ? w0 : wp), k1 = lb_list(in.dp_rec, in.n_dp, rg);
            for (int32_t k = k0 + W::lane(); k < k1; k += W::size()) {
                const int64_t r = in.dp_rec[k];
                if (in.b.ref_id[r] != chrG) continue;
                const bool part = in.cls[r] & CLS_PART;
                if (part ? (r < wp) : (r < st.offCC)) continue;
                const int32_t p0 = e_pos(r);
                add_span(t_cov, nM, p0, p0 + e_len(r));
            }
        }
        {   // ConcordRest (:471-473): blocks of records before rg that start at/after group start - ReadLen
            const int32_t lo_pos = sPos - RL;
            int32_t lo, lo2;
            rest_range(g, &lo, &lo2);
            for (int32_t base = lo; base < lo2; base += W::size()) {
                const int32_t k = base + W::lane();
                bool on = false;
                int32_t ja = 0, jb = 0;
                if (k < lo2) {
                    const RestBlock e = in.rest[k];
                    if (e.rec < rg && e.pos >= lo_pos && e.pos < pmax) { on = true; ja = m_upper(nM, e.pos + kSeedThresh); jb = m_upper(nM, e.end - kSeedThresh); }
                }
                W::add_range(t_rest, ja, jb, on);
            }
        }
        scan_inplace(t_pl, nM); scan_inplace(t_pr, nM); scan_inplace(t_cov, nM); scan_inplace(t_rest, nM);
    }

    // ---- the same tables indexed by POSITION -----------------------------------------------------------------------
    // When the margins of a sub-cluster span a modest position range [P_lo, P_lo + R) -- the rule for every island that sits in
    // a highly expressed gene, where the windows hold hundreds of thousands of records and the margins thousands of partial-
    // alignment ends -- nothing needs the sorted margin array: H[x] counts the margins at position x, the interval-shaped
    // contributions are +1/-1 at clamped position offsets (no binary searches), one prefix sum per table turns them into
    // values, and the candidate breaks (the positions that pass the support and coverage tests of :455-475, none of which
    // depends on what the break loop emits) are compacted in increasing order for the short sequential pass.
    SQ_HD int32_t didx(int32_t x, int32_t P_lo, int32_t R) const { const int32_t i = x - P_lo; return i < 0 ? 0 : (i > R ? R : i); }
    // returns the number of candidate breaks; CAND = (position, support) pairs
    SQ_HD int32_t tabulate_dense(int32_t g, int32_t nM, int32_t P_lo, int32_t R, int32_t ds, int32_t de, int32_t chrG, int32_t sPos, int64_t rg, int32_t szPC, int32_t *CAND) {
        const int32_t thresh = kSeedThresh, RL = in.read_len;
        int32_t *H = margin + mcap(), *PL = H + (R + 2), *PR = PL + (R + 2), *COV = PR + (R + 2), *REST = COV + (R + 2);
        const DiscBlock *D = in.D;
        W::sync();
        for (int32_t i = W::lane(); i < 5 * (R + 2); i += W::size()) H[i] = 0;
        W::sync();
        for (int32_t i = W::lane(); i < nM; i += W::size()) W::add(&H[margin[i] - P_lo], 1);
        for (int32_t k = ds + W::lane(); k < de; k += W::size()) {
            const int32_t p0 = D[k].pos, p1 = p0 + D[k].len;
            if (!D[k].rev) add_range(PL, didx(p1 + 1, P_lo, R), didx(p1 + RL, P_lo, R));            // end < b < end+ReadLen   (:450)
            else add_range(PR, didx(p0 - RL + 1, P_lo, R), didx(p0, P_lo, R));                      // pos-ReadLen < b < pos   (:452)
            if (D[k].chr == chrG) add_range(COV, didx(p0 + thresh + 1, P_lo, R), didx(p1 - thresh + 1, P_lo, R));   // :462-464
        }
        const int32_t bmin = P_lo, bmax = P_lo + R - 1;
        const int32_t pmin = bmin + thresh - in.lmax, pmax = bmax - thresh;  // block starts that can span some break
        // The window walks add +1/-1 at a handful of offsets over and over (sorted stream: hundreds of records per position in an
        // expressed gene), and atomics on one address in HBM/L2 scratch complete one after the other.  When the caller has fast
        // (shared) memory for them, the walks accumulate there and the sums are folded into the tables afterwards.
        int32_t *COVw = COV, *RESTw = REST;
        if (msearch && R + 2 <= msearch_cap) {
            COVw = msearch;
            if (2 * (R + 2) <= msearch_cap) RESTw = msearch + (R + 2);
            for (int32_t i = W::lane(); i < (RESTw != REST ? 2 : 1) * (R + 2); i += W::size()) msearch[i] = 0;
            W::sync();
        }
        if (st.offCC < rg) {  // ConcordantCluster window (:457-461); every record of [lo,hi) lies on chrG (sorted stream, rg is the group's trigger)
            const int64_t lo = lb_pos(st.offCC, rg, chrG, pmin), hi = lb_pos(lo, rg, chrG, pmax);
            constexpr int U = 8;
            for (int64_t base = lo; base < hi; base += (int64_t)W::size() * U) {
                uint8_t c[U]; uint32_t fl[U]; int32_t ps_[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int64_t r = base + (int64_t)u * W::size() + W::lane();
                    const bool inr = r < hi;
                    c[u] = inr ? in.cls[r] : (uint8_t)0; fl[u] = inr ? in.first_len[r] : 0u; ps_[u] = inr ? in.b.pos[r] : 0;
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const bool ok = (c[u] & (CLS_CONC | CLS_PART | CLS_DISPL)) == CLS_CONC;
                    int32_t l = (int32_t)fl[u];
                    if (ok && fl[u] == 65535u) l = in.b.blk_match_ref[in.b.blk_off[base + (int64_t)u * W::size() + W::lane()]];
                    W::add_range(COVw, didx(ps_[u] + thresh + 1, P_lo, R), didx(ps_[u] + l - thresh + 1, P_lo, R), ok);
                }
            }
        }
        if (st.offPC < szPC) {  // PartialAlignCluster window (:465-469)
            const int32_t lo = lb_pc_pos(st.offPC, szPC, chrG, pmin), hi = lb_pc_pos(lo, szPC, chrG, pmax);
            for (int32_t base = lo; base < hi; base += W::size()) {
                const int32_t i = base + W::lane();
                bool on = false;
                int32_t ja = 0, jb = 0;
                if (i < hi) {
                    const int64_t r = in.pc_rec[i];
                    if (!isDispl(r) && in.b.ref_id[r] == chrG) { on = true; const int32_t p0 = e_pos(r); ja = didx(p0 + thresh + 1, P_lo, R); jb = didx(p0 + e_len(r) - thresh + 1, P_lo, R); }
                }
                W::add_range(COVw, ja, jb, on);
            }
        }
        {   // displaced entries of either window
            const int64_t w0 = st.offCC < rg ? st.offCC : rg;
            const int64_t wp = st.offPC < szPC ? (int64_t)in.pc_rec[st.offPC] : rg;
            const int32_t k0 = lb_list(in.dp_rec, in.n_dp, w0 < wp ? w0 : wp), k1 = lb_list(in.dp_rec, in.n_dp, rg);
            for (int32_t k = k0 + W::lane(); k < k1; k += W::size()) {
                const int64_t r = in.dp_rec[k];
                if (in.b.ref_id[r] != chrG) continue;
                const bool part = in.cls[r] & CLS_PART;
                if (part ? (r < wp) : (r < st.offCC)) continue;
                const int32_t p0 = e_pos(r);
                add_range(COV, didx(p0 + thresh + 1, P_lo, R), didx(p0 + e_len(r) - thresh + 1, P_lo, R));
            }
        }
        {   // ConcordRest (:471-473): blocks of records before rg that start at/after group start - ReadLen
            const int32_t lo_pos = sPos - RL;
            int32_t lo, lo2;
            rest_range(g, &lo, &lo2);
            for (int32_t base = lo; base < lo2; base += W::size()) {
                const int32_t k = base + W::lane();
                bool on = false;
                int32_t ja = 0, jb = 0;
                if (k < lo2) {
                    const RestBlock e = in.rest[k];
                    if (e.rec < rg && e.pos >= lo_pos && e.pos < pmax) { on = true; ja = didx(e.pos + thresh + 1, P_lo, R); jb = didx(e.end - thresh + 1, P_lo, R); }
                }
                W::add_range(RESTw, ja, jb, on);
            }
        }
        if (COVw != COV) {  // fold the fast accumulators into the tables (the discordant blocks and displaced entries went there directly)
            W::sync();
            for (int32_t i = W::lane(); i <= R; i += W::size()) { COV[i] += COVw[i]; if (RESTw != REST) REST[i] += RESTw[i]; }
            W::sync();
        }
        scan_inplace(PL, R); scan_inplace(PR, R); scan_inplace(COV, R); scan_inplace(REST, R);
        // candidate breaks, in increasing position
        int32_t nC = 0;
        for (int32_t base = 0; base < R; base += W::size()) {
            const int32_t i = base + W::lane();
            bool is = false;
            int32_t sup = 0;
            if (i < R && H[i] > 0) {
                int32_t sr = 0;  // margins within +-thresh (:445-448)
                for (int32_t d = -(thresh - 1); d <= thresh - 1; d++) { const int32_t q = i + d; if (q >= 0 && q < R) sr += H[q]; }
                const int32_t pl = PL[i], pr = PR[i];
                if (sr > 3 || sr + pl > 4 || sr + pr > 4) {
                    int32_t coverage = COV[i];
                    int32_t rest = coverage - sr; if (rest < 0) rest = 0;
                    if (sr > rest + 2) { coverage += REST[i]; rest = coverage - sr; if (rest < 0) rest = 0; }
                    if (sr > rest + 2) { is = true; sup = sr + (pl > pr ? pl : pr); }
                }
            }
            const int32_t tot = W::sum(is ? 1 : 0);
            if (tot == 0) continue;
            const int32_t at = nC + W::excl_prefix_sum(is ? 1 : 0);
            if (is) { CAND[2 * at] = P_lo + i; CAND[2 * at + 1] = sup; }
            nC += tot;
        }
        W::sync();
        return nC;
    }

    struct BreakCtx { int32_t lastCurser, lastSupport, curStartPos, curEndPos; bool isClusternSplit; };
    // :476-497 for a break position that passed the support and coverage tests
    SQ_HD void accept_break(int32_t brk, int32_t sup, int32_t chrG, int32_t dpos, BreakCtx &c) {
        const int32_t thresh = kSeedThresh;
        if (c.lastCurser == -1 && brk - c.curStartPos < thresh * 20) {
            st.markedStart = c.curStartPos; st.markedChr = chrG;
        } else if ((c.lastCurser == -1 || brk - c.lastCurser < thresh * 20) && sup > c.lastSupport) {
            c.lastCurser = brk; c.lastSupport = sup;
        } else if (brk - c.lastCurser >= thresh * 20) {
            c.isClusternSplit = true;
            if (dpos - c.curStartPos > thresh * 20 && c.lastCurser - dpos > thresh * 20) {
                push_node(chrG, c.curStartPos, dpos - c.curStartPos);
                c.curStartPos = dpos;
            }
            push_node(chrG, c.curStartPos, c.lastCurser - c.curStartPos);
            c.curStartPos = c.lastCurser; c.curEndPos = c.lastCurser;
            st.markedStart = c.lastCurser; st.markedChr = chrG;
            c.lastCurser = brk;
        }
    }

    // flag1/flag2 of the two walks at :536-601 for an entry (c,p0,p1); dc = first discordant block not covered yet
    SQ_HD bool walk_ok(bool first_walk, int32_t chrG, int32_t dc, int32_t c, int32_t p0, int32_t p1) const {
        const DiscBlock *D = in.D;
        const int32_t RL = in.read_len;
        if (first_walk) {
            if (c > chrG) return false;
            if (dc != in.nD && c == D[dc].chr && p1 + RL >= D[dc].pos) return false;
            if (st.have_back && (c > st.backChr || (c == st.backChr && p0 >= st.backEnd))) return false;
            return true;
        }
        return dc == in.nD || c < D[dc].chr || (c == D[dc].chr && p1 + RL < D[dc].pos);
    }
    // maximum end over the ConcordantCluster entries of records [a, b) (all on one chromosome): whole tiles from the per-tile
    // table of the classification pass, the ragged ends (and the rare tiles that hold several chromosomes) by walking
    SQ_HD int32_t cc_end_max_walk(int64_t a, int64_t b) const {
        int32_t m = -(1 << 30);
        for (int64_t r = a + W::lane(); r < b; r += W::size())
            if (isCC(r)) { const int32_t e = e_pos(r) + e_len(r); if (e > m) m = e; }
        return m;  // lane-local
    }
    SQ_HD int32_t cc_end_max(int64_t a, int64_t b) const {
        int32_t m = -(1 << 30);
        if (b <= a) return m;
        const int64_t T = in.cc_tile;
        int64_t ta = T > 0 ? (a + T - 1) / T : 0, tb = T > 0 ? b / T : 0;
        if (!in.ccmax || T <= 0 || ta >= tb) m = cc_end_max_walk(a, b);
        else {
            int32_t v = cc_end_max_walk(a, ta * T); if (v > m) m = v;
            v = cc_end_max_walk(tb * T, b); if (v > m) m = v;
            for (int64_t t = ta + W::lane(); t < tb; t += W::size()) {
                int32_t q = in.ccmax[t];
                if (q == 0x7fffffff) {  // several chromosomes in the tile: this lane walks it
                    q = -(1 << 30);
                    for (int64_t r = t * T; r < (t + 1) * T; r++) if (isCC(r)) { const int32_t e = e_pos(r) + e_len(r); if (e > q) q = e; }
                }
                if (q > m) m = q;
            }
        }
        return W::max(m);
    }
    // Advance st.offCC over the maximal prefix of window entries that pass walk_ok; returns the largest end consumed.
    SQ_HD int32_t consume_cc(int64_t rg, int32_t chrG, int32_t dc, bool first_walk) {
        constexpr int U = 4;
        const int32_t NEG = -(1 << 30);
        const int chunk = W::size() * U;
        int32_t mx = NEG;
        int64_t x = st.offCC;
        if (first_walk && x < rg && in.b.ref_id[x] == chrG) {
            // Every entry of [offCC, rg) lies on chrG (sorted stream; :529-530 skipped the earlier chromosomes).  An entry that
            // starts left of T = min(next discordant block - ReadLen - lmax, end of the last segment) passes walk_ok whatever
            // its length, so up to the first record at or right of T only the maximum end matters: no per-chunk reductions.
            int64_t T = (int64_t)1 << 40;
            const DiscBlock *D = in.D;
            if (dc != in.nD && D[dc].chr == chrG) T = (int64_t)D[dc].pos - in.read_len - in.lmax;
            bool any_ok = true;
            if (st.have_back) {
                if (st.backChr < chrG) any_ok = false;               // c > backChr for every entry
                else if (st.backChr == chrG && st.backEnd < T) T = st.backEnd;
            }
            if (any_ok && T > in.b.pos[x]) {
                int64_t xs = T >= ((int64_t)1 << 31) ? rg : lb_pos(x, rg, chrG, (int32_t)T);
                // displaced entries start elsewhere than their record: the first one in [x, xs) that fails ends the prefix
                for (int32_t k = lb_list(in.dp_rec, in.n_dp, x); k < in.n_dp && in.dp_rec[k] < xs; k++) {
                    const int64_t r = in.dp_rec[k];
                    if (!isCC(r)) continue;
                    const int32_t p0 = e_pos(r);
                    if (!walk_ok(true, chrG, dc, e_chr(r), p0, p0 + e_len(r))) { xs = r; break; }
                }
                if (xs > x) {
                    const int32_t m = cc_end_max(x, xs);
                    if (m > mx) mx = m;
                    x = xs;
                }
            }
        }
        while (x < rg) {
            uint8_t c[U]; uint32_t fl[U]; int32_t rc[U], ps[U];
#pragma unroll
            for (int u = 0; u < U; u++) {  // entry index inside the chunk: u*size + lane (stream order)
                const int64_t r = x + u * W::size() + W::lane();
                const bool inr = r < rg;
                c[u] = inr ? in.cls[r] : (uint8_t)0; fl[u] = inr ? in.first_len[r] : 0u; rc[u] = inr ? in.b.ref_id[r] : -1; ps[u] = inr ? in.b.pos[r] : 0;
            }
            int32_t p1[U]; bool cc[U], ok[U];
            int fb = chunk;
#pragma unroll
            for (int u = 0; u < U; u++) {
                cc[u] = (c[u] & (CLS_CONC | CLS_PART)) == CLS_CONC;
                ok[u] = false; p1[u] = NEG;
                if (cc[u]) {
                    const int64_t r = x + u * W::size() + W::lane();
                    const bool plain = !(c[u] & CLS_DISPL) && fl[u] != 65535u;  // else: through the block arrays
                    const int32_t p0 = plain ? ps[u] : e_pos(r);
                    p1[u] = p0 + (plain ? (int32_t)fl[u] : e_len(r));
                    ok[u] = walk_ok(first_walk, chrG, dc, rc[u], p0, p1[u]);
                    if (!ok[u] && u * W::size() + W::lane() < fb) fb = u * W::size() + W::lane();
                }
            }
            const int first_bad = W::min(fb);
            int32_t m = NEG;
#pragma unroll
            for (int u = 0; u < U; u++) if (cc[u] && ok[u] && u * W::size() + W::lane() < first_bad && p1[u] > m) m = p1[u];
            m = W::max(m);
            if (m > mx) mx = m;
            if (first_bad < chunk) { st.offCC = x + first_bad; return mx; }
            x += chunk;
        }
        st.offCC = rg;
        return mx;
    }
    SQ_HD int32_t consume_pc(int32_t szPC, int32_t chrG, int32_t dc, bool first_walk) {
        int32_t mx = -(1 << 30);
        int32_t x = st.offPC;
        while (x < szPC) {
            const int32_t i = x + W::lane();
            const bool in_w = i < szPC;
            bool ok = false;
            int32_t p1 = -(1 << 30);
            if (in_w) { const int64_t r = in.pc_rec[i]; const int32_t p0 = e_pos(r); p1 = p0 + e_len(r); ok = walk_ok(first_walk, chrG, dc, e_chr(r), p0, p1); }
            const int first_bad = W::min((in_w && !ok) ? W::lane() : W::size());
            const int32_t m = W::max((in_w && ok && W::lane() < first_bad) ? p1 : -(1 << 30));
            if (m > mx) mx = m;
            if (first_bad < W::size()) { st.offPC = x + first_bad; return mx; }
            x += W::size();
        }
        st.offPC = szPC;
        return mx;
    }
    // close-out of the pending segment at the 0-coverage position concord0pos (:572-580)
    SQ_HD void close_marked(int32_t concord0pos, int32_t &curStartPos) {
        const int32_t thresh = kSeedThresh;
        if (st.back_inherited) {
            // the last segment was emitted by an earlier island: whether it is on markedChr (extend it) or not (push a
            // new one) is decided when the islands are stitched; either way the last segment becomes (markedChr, concord0pos)
            if (concord0pos > st.markedStart) {
                emit(concord0pos < st.markedStart + thresh * 20 ? 1 : 0, st.markedChr, st.markedStart, concord0pos - st.markedStart);
                st.have_back = true; st.back_inherited = false; st.backChr = st.markedChr; st.backEnd = concord0pos;
            }
        } else if (concord0pos > st.markedStart && concord0pos < st.markedStart + thresh * 20 && st.have_back && st.backChr == st.markedChr)
            set_back_end(concord0pos);
        else if (concord0pos > st.markedStart)
            push_node(st.markedChr, st.markedStart, concord0pos - st.markedStart);
        curStartPos = concord0pos;
        st.markedChr = -1; st.markedStart = -1;
    }
    // The loop at :570-601.  Every iteration first tests whether the stream shows a 0-coverage position right after
    // concord0pos (then the pending segment is closed there), else consumes one entry of each window that is still more
    // than ReadLen left of the next discordant block.  While the (sparse) PartialAlignCluster window still moves the
    // iterations are stepped one by one; afterwards only the ConcordantCluster window advances and the iterations are
    // evaluated a chunk at a time with a prefix maximum of the consumed ends.
    SQ_HD void extend_to_zero_coverage(int64_t rg, int32_t szPC, int32_t dc, int32_t recChr, int32_t recPos, int32_t concord0pos, int32_t &curStartPos) {
        const int32_t RL = in.read_len;
        bool first = true;
        for (;;) {  // phase 1: literal iterations while the PartialAlignCluster front is consumable
            const bool ccEmpty = !(st.offCC < rg), pcEmpty = !(st.offPC < szPC);
            if (!first && ccEmpty && pcEmpty) return;  // `while(... .size()!=offset ...)` fails
            bool f2 = false;
            int32_t pc_c = 0, pc_p0 = 0, pc_p1 = 0;
            if (!pcEmpty) {
                const int64_t r = in.pc_rec[st.offPC];
                pc_c = e_chr(r); pc_p0 = e_pos(r); pc_p1 = pc_p0 + e_len(r);
                f2 = walk_ok(false, 0, dc, pc_c, pc_p0, pc_p1);
            }
            if (!f2) break;  // the PartialAlignCluster front is stuck (or the window is empty) from now on
            first = false;
            int32_t cc_c = 0, cc_p0 = 0, cc_p1 = 0;
            if (!ccEmpty) { cc_c = e_chr(st.offCC); cc_p0 = e_pos(st.offCC); cc_p1 = cc_p0 + e_len(st.offCC); }
            if (st.markedStart != -1 && (recChr > st.markedChr || recPos > concord0pos + RL) &&
                (ccEmpty || cc_c != st.markedChr || cc_p0 > concord0pos + RL) && (pc_c != st.markedChr || pc_p0 > concord0pos)) {
                close_marked(concord0pos, curStartPos);
                return;
            }
            if (!ccEmpty && walk_ok(false, 0, dc, cc_c, cc_p0, cc_p1)) { if (cc_p1 > concord0pos) concord0pos = cc_p1; st.offCC = nextCC(st.offCC + 1, rg); }
            if (pc_p1 > concord0pos) concord0pos = pc_p1;
            st.offPC++;
        }
        // phase 2: the PartialAlignCluster front is fixed
        const bool pcEmpty = !(st.offPC < szPC);
        int32_t pc_c = -1, pc_p0 = 0;
        if (!pcEmpty) { pc_c = e_chr(in.pc_rec[st.offPC]); pc_p0 = e_pos(in.pc_rec[st.offPC]); }
        const bool marked = st.markedStart != -1;
        int64_t x = st.offCC;
        for (;;) {
            if (x >= rg) {  // ConcordantCluster window exhausted
                st.offCC = rg;
                if (!first && pcEmpty) return;
                if (marked && (recChr > st.markedChr || recPos > concord0pos + RL) && (pcEmpty || pc_c != st.markedChr || pc_p0 > concord0pos))
                    close_marked(concord0pos, curStartPos);
                return;  // neither window can move
            }
            const int64_t r = x + W::lane();
            const bool cc = r < rg && isCC(r);
            int32_t c = 0, p0 = 0, p1 = -(1 << 30);
            bool f1 = false;
            if (cc) { c = e_chr(r); p0 = e_pos(r); p1 = p0 + e_len(r); f1 = walk_ok(false, 0, dc, c, p0, p1); }
            // concord0pos seen by this lane's iteration = everything consumed by the lanes before it
            int32_t mi = W::excl_prefix_max(cc ? p1 : -(1 << 30), -(1 << 30));
            if (concord0pos > mi) mi = concord0pos;
            const bool close_i = cc && marked && (recChr > st.markedChr || recPos > mi + RL) && (c != st.markedChr || p0 > mi + RL) &&
                                 (pcEmpty || pc_c != st.markedChr || pc_p0 > mi);
            const bool stop_i = cc && (close_i || !f1);
            const int fs = W::min(stop_i ? W::lane() : W::size());
            if (fs < W::size()) {
                const int32_t m_at = W::max(W::lane() == fs ? mi : -(1 << 30));
                const int32_t cl_at = W::max((W::lane() == fs && close_i) ? 1 : 0);
                st.offCC = x + fs;
                concord0pos = m_at;
                if (cl_at) close_marked(concord0pos, curStartPos);
                return;
            }
            const int32_t m = W::max(cc ? p1 : -(1 << 30));
            if (m > concord0pos) concord0pos = m;
            if (W::max(cc ? 1 : 0)) first = false;
            x += W::size();
        }
    }

    // Lines :353-612 for group g, reached at trigger record rg.
    SQ_HD void process_group(int32_t g, int64_t rg) {
        const int32_t thresh = kSeedThresh, RL = in.read_len;
        const Group grp = in.G[g];
        int32_t ds = grp.ds; const int32_t de = grp.de, chrG = grp.chr, nextright = grp.right;
        const DiscBlock *D = in.D;
        const int32_t recChr = in.b.ref_id[rg], recPos = in.b.pos[rg];
        int32_t curEndPos = 0, curStartPos = 0, disStartPos = -1, disEndPos = -1, disCount = -1;
        bool isClusternSplit = false;
        if (st.markedStart != -1 && chrG != st.markedChr) { st.markedChr = -1; st.markedStart = -1; }
        const int32_t szPC = lb_list(in.pc_rec, in.n_pc, rg);
        // :365-368 skip cluster entries of earlier chromosomes
        {
            const int64_t lo = lb_pos(0, rg, chrG, -(1 << 30));
            if (lo > st.offCC) st.offCC = lo;
            st.offCC = nextCC(st.offCC, rg);
            while (st.offPC < szPC && e_chr(in.pc_rec[st.offPC]) < chrG) st.offPC++;
        }
        // :369-372 whole window stale?
        if (st.offCC < rg) {
            int64_t lb = rg - 1;
            while (!isCC(lb)) lb--;
            if (D[ds].pos > e_pos(lb) + e_len(lb) + RL) st.offCC = rg;
        }
        if (st.offPC < szPC) {
            const int64_t lb = in.pc_rec[szPC - 1];
            if (D[ds].pos > e_pos(lb) + e_len(lb) + RL) st.offPC = szPC;
        }
#ifdef __CUDA_ARCH__
        if (in.win_count && W::lane() == 0 && rg > st.offCC) atomicAdd(in.win_count, (unsigned long long)(rg - st.offCC));
#endif
        // :375-385
        curStartPos = D[ds].pos;
        {
            const bool hc = st.offCC < rg, hp = st.offPC < szPC;
            int64_t t = -1;
            if (hc && hp) {
                const int64_t a = st.offCC, bq = in.pc_rec[st.offPC];
                const bool a_lt = e_chr(a) != e_chr(bq) ? e_chr(a) < e_chr(bq) : e_pos(a) < e_pos(bq);
                t = a_lt ? a : bq;
            } else if (hc) t = st.offCC;
            else if (hp) t = in.pc_rec[st.offPC];
            if (t >= 0 && (e_chr(t) < chrG || (e_chr(t) == chrG && e_pos(t) < D[ds].pos))) curStartPos = e_pos(t);
        }
        if (st.markedStart > curStartPos) curStartPos = st.markedStart;
        // :392-393 PartAlignPos window of this group
        int32_t ps, pe;
        {
            const int32_t v = D[ds].pos - RL;
            int32_t lo = 0, hi = in.nP;
            while (lo < hi) { int32_t m = (lo + hi) >> 1; if (in.Pchr[m] < chrG || (in.Pchr[m] == chrG && in.Ppos[m] < v)) lo = m + 1; else hi = m; }
            ps = lo;
            hi = in.nP;  // first entry from ps on that leaves (chrG, < nextright + ReadLen); the list is sorted by (chr, pos)
            while (lo < hi) { int32_t m = (lo + hi) >> 1; if (in.Pchr[m] == chrG && in.Ppos[m] < nextright + RL) lo = m + 1; else hi = m; }
            pe = lo;
        }
        while (ds != de) {
            if (ds != 0 && D[ds].chr != D[ds - 1].chr && st.offCC >= rg && st.offPC >= szPC) curStartPos = D[ds].pos;
            isClusternSplit = false;
            int32_t nM = 0;
            int32_t dc;
            const int32_t m0 = D[ds].pos;  // MarginPositions.front() while still unsorted
            {   // :400-416, the loops over the discordant blocks and PartAlignPos split across the lanes (only the multiset of
                // margins matters).  First loop: blocks from ds up to one that the next block does not touch.
                const int32_t dcb = find_first(ds, de - 1, [&](int32_t k) { return D[k + 1].pos > D[k].pos + D[k].len; });
                const bool broke = dcb < de - 1;
                int32_t mx = -(1 << 30);
                for (int32_t k = ds + W::lane(); k <= dcb; k += W::size()) { const int32_t e = D[k].pos + D[k].len; if (e > mx) mx = e; }
                mx = W::max(mx);
                if (mx > curEndPos) curEndPos = mx;
                disStartPos = curStartPos > D[ds].pos ? curStartPos : D[ds].pos;
                disEndPos = curEndPos;
                disCount = broke ? dcb - ds : de - ds;
                dc = broke ? dcb : de;
                int32_t dend = de;  // margins of the blocks [ds, dend)
                if (broke) { const int32_t lim = curEndPos + thresh; dend = find_first(dcb + 1, de, [&](int32_t k) { return !(D[k].pos < lim); }); dc = dend; }
                int32_t pce = ps;   // PartAlignPos entries [ps, pce): sorted by position inside the group's window
                { int32_t lo = ps, hi = pe; const int32_t lim = curEndPos + thresh; while (lo < hi) { const int32_t m = (lo + hi) >> 1; if (in.Ppos[m] < lim) lo = m + 1; else hi = m; } pce = lo; }
                const int32_t n_fixed = 2 * (dend - ds) + (pce - ps);
                if (n_fixed + 1 >= mcap()) { error = 1; return; }
                for (int32_t k = ds + W::lane(); k < dend; k += W::size()) { margin[2 * (k - ds)] = D[k].pos; margin[2 * (k - ds) + 1] = D[k].pos + D[k].len; }
                for (int32_t k = ps + W::lane(); k < pce; k += W::size()) margin[2 * (dend - ds) + (k - ps)] = in.Ppos[k];
                nM = n_fixed;
            }
            if (st.offPC < szPC) {  // :420-434; an entry contributes only if its block start lies in (m0-thresh-lmax, curEndPos+thresh)
                const int32_t lo = lb_pc_pos(st.offPC, szPC, chrG, m0 - thresh - in.lmax), hi = lb_pc_pos(lo, szPC, chrG, curEndPos + thresh);
                pc_margins(in.pc_rec, lo, hi, false, chrG, m0, curEndPos, nM);
                const int64_t wp = in.pc_rec[st.offPC];
                if (in.n_dp > 0 && !error) pc_margins(in.dp_rec, lb_list(in.dp_rec, in.n_dp, wp), lb_list(in.dp_rec, in.n_dp, rg), true, chrG, m0, curEndPos, nM);
            }
            if (error) return;
            W::sync();
            BreakCtx bc;
            bc.lastCurser = -1; bc.lastSupport = 0; bc.curStartPos = curStartPos; bc.curEndPos = curEndPos; bc.isClusternSplit = false;
            bool dense = false;
            int32_t P_lo = 0, R = 0;
            if (use_dense && in.dense_max_r > 0) {  // position range of the margins: small enough for position-indexed tables?
                int32_t mn = 0x7fffffff, mx = -(1 << 30);
                for (int32_t i = W::lane(); i < nM; i += W::size()) { const int32_t v = margin[i]; if (v < mn) mn = v; if (v > mx) mx = v; }
                mn = W::min(mn); mx = W::max(mx);
                const int64_t r64 = (int64_t)mx - mn + 1;
                // (a wide range with a handful of margins is cheaper through the sorted margins: the tables cost O(R))
                if (r64 <= in.dense_max_r && r64 <= 16 * (int64_t)nM + 4096 && 5 * (r64 + 2) + 2 * (r64 < nM ? r64 : (int64_t)nM) + 2 <= 5 * (int64_t)mcap()) { dense = true; P_lo = mn; R = (int32_t)r64; }
            }
            if (dense) n_dense++; else n_sparse++;
            if (dense) {
                int32_t *CAND = margin + mcap() + 5 * (R + 2);
                const int32_t nC = tabulate_dense(g, nM, P_lo, R, ds, de, chrG, in.D[grp.ds].pos, rg, szPC, CAND);
                for (int32_t ic = 0; ic < nC; ic++) {
                    const int32_t brk = CAND[2 * ic];
                    if (st.have_back && st.backChr == chrG && brk - st.backEnd < thresh * 20) continue;
                    accept_break(brk, CAND[2 * ic + 1], chrG, D[ds].pos, bc);
                }
            } else {
                sort_margins(nM);
                if (error) return;
                ms = margin;
                if (nM <= msearch_cap) {  // the sorted margins are searched twice per window entry: keep them close
                    for (int32_t i = W::lane(); i < nM; i += W::size()) msearch[i] = margin[i];
                    W::sync();
                    ms = msearch;
                }
                tabulate_breaks(g, nM, ds, de, chrG, in.D[grp.ds].pos, rg, szPC);
                const int32_t *t_sr = margin + mcap(), *t_pl = margin + 2 * mcap(), *t_pr = margin + 3 * mcap(), *t_cov = margin + 4 * mcap(), *t_rest = margin + 5 * mcap();
                for (int32_t ib = 0; ib < nM;) {
                    const int32_t brk = ms[ib];
                    if (st.have_back && st.backChr == chrG && brk - st.backEnd < thresh * 20) { ib++; continue; }
                    const int32_t sr = t_sr[ib], pl = t_pl[ib], pr = t_pr[ib];
                    if (sr > 3 || sr + pl > 4 || sr + pr > 4) {
                        int32_t coverage = t_cov[ib];
                        int32_t rest = coverage - sr; if (rest < 0) rest = 0;
                        if (sr > rest + 2) {
                            coverage += t_rest[ib];
                            rest = coverage - sr; if (rest < 0) rest = 0;
                        }
                        if (sr > rest + 2) accept_break(brk, sr + (pl > pr ? pl : pr), chrG, D[ds].pos, bc);
                    }
                    int32_t j = ib;
                    while (j < nM && ms[j] == brk) j++;
                    if (j < nM) ib = j; else break;
                }
            }
            int32_t lastCurser = bc.lastCurser;
            curStartPos = bc.curStartPos; curEndPos = bc.curEndPos; isClusternSplit = bc.isClusternSplit;
            if (lastCurser != -1 && (!isClusternSplit || st.backEnd != lastCurser)) {  // :505-516
                isClusternSplit = true;
                if (D[ds].pos - curStartPos > thresh * 20 && lastCurser - D[ds].pos > thresh * 20) {
                    push_node(chrG, curStartPos, D[ds].pos - curStartPos);
                    curStartPos = D[ds].pos;
                }
                push_node(chrG, curStartPos, lastCurser - curStartPos);
                curStartPos = lastCurser; curEndPos = lastCurser;
                st.markedStart = lastCurser; st.markedChr = chrG;
            }
            // :518-527 dense discordant group without a clear break: the whole span is one segment
            if (disStartPos != -1 && !isClusternSplit &&
                (disCount > 5 || (int64_t)disCount * RL > 4 * (int64_t)(disEndPos - disStartPos))) {
                const int32_t lastChr = D[de - 1].chr;
                if (st.have_back && st.backChr == lastChr && disEndPos - st.backEnd < thresh * 20) set_back_end(disEndPos);
                else push_node(lastChr, disStartPos, disEndPos - disStartPos);
                curStartPos = disEndPos; curEndPos = disEndPos;
                st.markedStart = disEndPos; st.markedChr = chrG;
            }
            // :529-532
            while (st.offCC < rg && e_chr(st.offCC) < chrG) st.offCC = nextCC(st.offCC + 1, rg);
            while (st.offPC < szPC && e_chr(in.pc_rec[st.offPC]) < chrG) st.offPC++;
            { const int32_t lim = curEndPos; dc = find_first(ds, de, [&](int32_t k) { return !(D[k].pos + D[k].len <= lim); }); }
            // :536-567 walk the windows up to the end of the last inserted segment, tracking the 0-coverage position.
            // Each window gives up its maximal prefix of entries that lie left of the last segment's end and more than
            // ReadLen left of the next discordant block; the two windows do not influence each other here.
            int32_t concord0pos = curStartPos;
            {
                const int32_t a = consume_cc(rg, chrG, dc, true), bq = consume_pc(szPC, chrG, dc, true);
                if (a > concord0pos) concord0pos = a;
                if (bq > concord0pos) concord0pos = bq;
            }
            // :570-601 extend the last segment to the next 0-coverage position if the stream already shows one
            extend_to_zero_coverage(rg, szPC, dc, recChr, recPos, concord0pos, curStartPos);
            ds = dc;
            if (error) return;
        }
    }

    // One island: groups [ga, gb).  `inherited_back`: some earlier island has emitted a segment.
    // Returns the first group that was NOT processed (gb, or earlier if the stream ended first).
    SQ_HD int32_t run_island(int32_t ga, int32_t gb, bool inherited_back) {
        init(inherited_back);
        int32_t dChr = 0, dRight = 0;
        int64_t r_prev = in.first_kept;
        if (ga > 0) { dChr = in.G[ga - 1].chr; dRight = in.G[ga - 1].right; r_prev = in.trigger[ga - 1]; }
        int32_t g = ga;
        for (; g < gb; g++) {
            const int64_t rg = in.trigger[g];
            const Group grp = in.G[g];
            if (rg >= in.n_rec) break;
            replay_between(r_prev, rg, dChr, dRight, grp.chr, in.D[grp.ds].pos, true);
            process_group(g, rg);
            if (error) return g;
            dChr = grp.chr; dRight = grp.right;
            r_prev = rg;
        }
        // tail: a pending segment is closed by the first 0-coverage record that follows, while the next group
        // (or, once the stream ends before it, still that group) is pending
        if (g < in.nG) {
            const Group grp = in.G[g];
            const int64_t r_hi = in.trigger[g] < in.n_rec ? in.trigger[g] : in.n_rec;
            replay_between(r_prev, r_hi, dChr, dRight, grp.chr, in.D[grp.ds].pos, false);
            if (in.has_next && in.trigger[g] >= in.n_rec && st.markedStart != -1) {
                // range shard: the pending segment is closed by the first record of the next shard, a 0-coverage record
                // whose (curChr, currightmost) is the maximum of the last group's right end and the batch's final other key
                const uint64_t e = in.end_other < (1ull << 32) ? (1ull << 32) : in.end_other;
                const int32_t oChr = (int32_t)(e >> 32) - 1, oRight = (int32_t)(uint32_t)e;
                const int32_t cr = (dChr > oChr || (dChr == oChr && dRight > oRight)) ? dRight : oRight;
                const int32_t cc = dChr > oChr ? dChr : oChr;
                close_marked_gap(cc, cr);
            }
        }
        // after the very last group the reference compares against the element one past the end of bamdiscordant
        // (zero sentinel): the 0-coverage test can never hold there, nothing to do.
        return g;
    }
};

typedef SeedMachineT<CoopSerial> SeedMachine;

// Stitch island op lists (in island order) into the seed-segment list.  Host side (sizes are tiny).
template <class Vec>
inline void stitch_ops(const SeedOp *ops, int32_t n_ops, Vec &seeds) {
    for (int32_t i = 0; i < n_ops; i++) {
        const SeedOp &o = ops[i];
        if (o.kind == 0) seeds.push_back(SeedNode{o.chr, o.pos, o.len});
        else if (o.kind == 1) {
            if (!seeds.empty() && seeds.back().chr == o.chr) seeds.back().len = o.pos + o.len - seeds.back().pos;
            else seeds.push_back(SeedNode{o.chr, o.pos, o.len});
        } else if (!seeds.empty()) seeds.back().len = o.pos - seeds.back().pos;
    }
}

}  // namespace sq
#endif
