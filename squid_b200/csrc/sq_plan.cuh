// The range-shard planner of host/plan.cpp on the resident batch (sqg_plan_shards_resident): the same cuts, from per-record rules
// and device scans instead of a host walk.  host/plan.cpp scans the stream once and, for every record past its target, tests
// the conditions of a clean cut by walking back from it.  All of a cut at c except the first record `lo` of the shard that
// would end at c is a property of c alone:
//   A  c is the first record of its chromosome, or pos[c] lies more than ReadLen + kIslandSlack + 200 right of the largest
//      plan_reach (GetEndPosition, end of the last block, position) of the earlier records of its chromosome;
//   B  c is kept, owns a block and its first block starts at pos[c] (CLS_KEEP, CLS_HASBLK, not CLS_DISPL);
//   C  the discordant groups are clear of k2(c), the second-to-last kept record before c, and of c (plan_groups_clear);
//   D  k2(c) and u(c), the last record before c that updates otherrightmost (CLS_CONC with a mate flag, i.e. classify_record's
//      other_key != 0), lie inside plan.cpp's look-back window of kPlanLookBack records.
// The walk back from c then finds both inside the shard iff min(k2(c), u(c)) >= lo.  So a candidate is the pair
// (c, min(k2(c), u(c))), and plan.cpp's greedy over the stream is plan_greedy over the candidates.  plan.cpp stops at the first
// record with ref_id < 0; no such record passes the gate (B), and in a sorted batch (the classification pass refuses any
// other) all of them follow the last mapped record, so the candidates end there too.
#ifndef SQ_PLAN_CUH
#define SQ_PLAN_CUH
#include "sq_classify.cuh"
#include "sq_seed.cuh"

namespace sq {

constexpr int32_t kPlanMargin = 200;            // plan.cpp: P.margin
constexpr int64_t kPlanLookBack = 1 << 20;      // plan.cpp: records the walk back from a cut looks at
constexpr uint64_t kPlanNoCand = ~0ull;

// (ref_id, reach) as one key ordered lexicographically -- ref_id + 1 < 2^31 above reach + 2^31 < 2^33 -- so that over a sorted
// stream the prefix maximum is the largest reach on the latest chromosome; 0 = no record
SQ_HD uint64_t plan_reach_key(int32_t ref_id, int64_t reach) { return ((uint64_t)(uint32_t)(ref_id + 1) << 33) | (uint64_t)(reach + (1ll << 31)); }
SQ_HD int32_t plan_key_chr(uint64_t key) { return (int32_t)(key >> 33) - 1; }
SQ_HD int64_t plan_key_reach(uint64_t key) { return (int64_t)(key & ((1ull << 33) - 1)) - (1ll << 31); }

// how far right record r reaches for condition A
template <class B>
SQ_HD int64_t plan_reach(const B &b, int64_t r) {
    int64_t e = b.end_pos[r];
    const uint32_t o0 = b.blk_off[r], o1 = b.blk_off[r + 1];
    if (o1 > o0) {
        const int64_t x = (int64_t)b.blk_ref_pos[o1 - 1] + b.blk_match_ref[o1 - 1];
        if (x > e) e = x;
    }
    if ((int64_t)b.pos[r] > e) e = b.pos[r];
    return e;
}

SQ_HD bool plan_updates_other(uint8_t cls, uint16_t flag) { return (cls & CLS_CONC) && (flag_first(flag) || flag_second(flag)); }

// C: the first group not clear of (c2, p2) on the left must be clear of (ci, pi) on the right (group right ends increase)
SQ_HD bool plan_groups_clear(const Group *G, const DiscBlock *D, int32_t nG, int32_t c2, int32_t p2, int32_t ci, int32_t pi, int32_t read_len) {
    int32_t lo = 0, hi = nG;
    while (lo < hi) {
        const int32_t m = lo + ((hi - lo) >> 1);
        const bool left = G[m].chr < c2 || (G[m].chr == c2 && (int64_t)G[m].right + read_len + kPlanMargin < p2);
        if (left) lo = m + 1; else hi = m;
    }
    if (lo == nG) return true;
    const Group x = G[lo];
    const int64_t start = D[x.ds].pos;
    return x.chr > ci || (x.chr == ci && start - read_len - kPlanMargin > pi);
}

// The lo-free part of a cut at c: min(k2(c), u(c)), or -1 when c is no candidate.  `before` = exclusive prefix maximum of
// plan_reach_key at c; keep_excl[r] / upd_excl[r] = last kept / otherrightmost-updating record before r (-1: none).
template <class B>
SQ_HD int64_t plan_candidate(const B &b, const Params &p, uint8_t cls_c, uint64_t before, const int32_t *keep_excl, const int32_t *upd_excl,
                             const Group *G, const DiscBlock *D, int32_t nG, int64_t c) {
    if ((cls_c & (CLS_KEEP | CLS_HASBLK | CLS_DISPL)) != (CLS_KEEP | CLS_HASBLK)) return -1;  // B
    const int32_t ci = b.ref_id[c], pi = b.pos[c];
    if (plan_key_chr(before) == ci && (int64_t)pi - plan_key_reach(before) <= (int64_t)p.read_len + kIslandSlack + kPlanMargin) return -1;  // A
    const int64_t k1 = keep_excl[c], k2 = k1 >= 0 ? keep_excl[k1] : -1, u = upd_excl[c];
    if (k2 < 0 || u < 0 || c - k2 >= kPlanLookBack || c - u >= kPlanLookBack) return -1;  // D
    if (!plan_groups_clear(G, D, nG, b.ref_id[k2], b.pos[k2], ci, pi, p.read_len)) return -1;  // C
    return k2 < u ? k2 : u;
}
SQ_HD uint64_t plan_pack(int64_t c, int64_t m) { return ((uint64_t)c << 32) | (uint32_t)m; }

// plan.cpp's greedy over the candidates (packed (c, min(k2, u)), ascending c) of a stream of n records: writes cuts[0..k] with
// cuts[0] = 0 and cuts[k] = n, returns k <= n_shards.  Shard k ends at the first candidate c >= max(cut k-1 + 1, n / n_shards * k)
// whose look-back stays inside it.
inline int32_t plan_greedy(const uint64_t *cand, int64_t n_cand, int64_t n, int32_t n_shards, int64_t *cuts) {
    int32_t made = 0;
    cuts[0] = 0;
    int64_t target = n_shards > 1 ? n / n_shards : n;
    for (int64_t i = 0; i < n_cand && made + 1 < n_shards; i++) {
        const int64_t c = (int64_t)(cand[i] >> 32), m = (int64_t)(uint32_t)cand[i];
        if (c >= target && c > cuts[made] && m >= cuts[made]) {
            cuts[++made] = c;
            const int64_t nominal = n / n_shards * (int64_t)(made + 1);
            target = c + 1 > nominal ? c + 1 : nominal;
        }
    }
    cuts[made + 1] = n;
    return made + 1;
}

#if defined(__CUDACC__)
struct PlanIsCand { __device__ bool operator()(uint64_t x) const { return x != kPlanNoCand; } };

// inputs of the three exclusive scans: (ref_id, reach), "kept", "updates otherrightmost"
__global__ void k_plan_prep(DevBatch b, const uint8_t *cls, uint64_t *reach, int32_t *keep, int32_t *upd) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= b.n_rec) return;
    const uint8_t k = cls[r];
    reach[r] = plan_reach_key(b.ref_id[r], plan_reach(b, r));
    keep[r] = (k & CLS_KEEP) ? (int32_t)r : -1;
    upd[r] = plan_updates_other(k, b.flag[r]) ? (int32_t)r : -1;
}

__global__ void k_plan_cands(DevBatch b, Params p, const uint8_t *cls, const uint64_t *reach_excl, const int32_t *keep_excl, const int32_t *upd_excl,
                             const Group *G, const DiscBlock *D, int32_t nG, uint64_t *cand) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= b.n_rec) return;
    const int64_t m = plan_candidate(b, p, cls[c], reach_excl[c], keep_excl, upd_excl, G, D, nG, c);
    cand[c] = m < 0 ? kPlanNoCand : plan_pack(c, m);
}

// blk_off of a kept record range, rebased to start at 0 (src: the range's n + 1 offsets, copied out of the batch first)
__global__ void k_keep_offsets(uint32_t *dst, const uint32_t *src, int64_t n1, uint32_t base) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n1) dst[i] = src[i] - base;
}
#endif

}  // namespace sq
#endif
