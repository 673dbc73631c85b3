#include "prepass.h"

#include <algorithm>
#include <cstdlib>
#include <thread>
#include <omp.h>
#include <chrono>
#include <cstdio>

namespace sqh {
namespace {
// one chimeric read as index ranges over the flat block arrays of sqg_chimeric: FirstRead = [f0,f1), SecondMate = [f1,s1)
struct View {
    const sqg_chimeric &c;
    uint32_t f0, f1, s1;
    int32_t chr(uint32_t k) const { return c.blk_ref_id[k]; }
    int32_t pos(uint32_t k) const { return c.blk_ref_pos[k]; }
    int32_t rpos(uint32_t k) const { return c.blk_read_pos[k]; }
    int32_t mref(uint32_t k) const { return c.blk_match_ref[k]; }
    int32_t mread(uint32_t k) const { return c.blk_match_read[k]; }
    bool rev(uint32_t k) const { return c.blk_is_reverse[k] != 0; }
};
bool end_disc(const View &v, uint32_t a, uint32_t b) {  // ReadRec.cpp:178-209 on blocks [a,b)
    for (uint32_t i = a; i + 1 < b; i++) {
        if (v.chr(i) != v.chr(i + 1) || v.rev(i) != v.rev(i + 1)) return true;
        const bool x = v.pos(i) < v.pos(i + 1), r = v.rpos(i) < v.rpos(i + 1);
        if (!v.rev(i) && x != r) return true;
        if (v.rev(i) && x == r) return true;
    }
    return false;
}
bool pair_disc(const View &v, int32_t ft, int32_t st_) {  // ReadRec.cpp:211-228 with needcheck=true
    if (v.f0 == v.f1 || v.f1 == v.s1) return false;
    if (end_disc(v, v.f0, v.f1) || end_disc(v, v.f1, v.s1)) return true;
    const uint32_t ff = v.f0, fb = v.f1 - 1, sf = v.f1, sb = v.s1 - 1;
    if (v.chr(ff) != v.chr(sb) || v.rev(ff) == v.rev(sb)) return true;
    if (!v.rev(ff) && v.pos(ff) - v.rpos(ff) > v.pos(sb) - (st_ - v.rpos(sb) - v.mread(sb))) return true;
    if (!v.rev(sf) && v.pos(sf) - v.rpos(sf) > v.pos(fb) - (ft - v.rpos(fb) - v.mread(fb))) return true;
    return false;
}

// ---- std::sort, run on several threads -----------------------------------------------------------------------------
// The order in which equal (RefID,RefPos) blocks leave the reference's `sort(bamdiscordant)` (SegmentGraph.cpp:264) is
// observable (SURVEY.md App. A-11), so the pre-pass must produce exactly libstdc++'s std::sort permutation.  std::sort
// is introsort: quicksort partitions (median of first+1 / middle / last-1 moved to the front, unguarded Hoare partition
// around it, recursion on the right part, loop on the left) down to ranges of 16, heap sort when the depth budget
// 2*floor(log2 n) runs out, and a final insertion sort.  Two facts make it parallel without changing a single outcome:
//   * after a partition the two parts never interact again (the final insertion pass is stable and never moves an element
//     across a partition boundary), so they can be finished by different threads;
//   * the Hoare partition itself has a closed form.  With L = positions (ascending) whose element is not < pivot and
//     R = positions (descending) whose element is not > pivot, the loop swaps L[i] <-> R[i] for i < m, m = #{i : L[i] < R[i]},
//     and returns L[m] if that lies left of R[m-1], else R[m-1]; every scan of the loop only ever looks at positions no
//     earlier swap has touched.  So big ranges are partitioned by all threads together (collect L and R per chunk, pair
//     them up, swap in parallel).
// tests/test_cpu_host_twin.py checks this routine against std::sort (ties, sorted, reversed and organ-pipe inputs).
inline bool sk_lt(const SortKey &x, const SortKey &y) { return x.key < y.key; }
inline void median_to_first(SortKey *first, SortKey *last) {  // std::__move_median_to_first(first, first+1, mid, last-1)
    SortKey *mid = first + (last - first) / 2, *a = first + 1, *c = last - 1;
    if (sk_lt(*a, *mid)) {
        if (sk_lt(*mid, *c)) std::swap(*first, *mid);
        else if (sk_lt(*a, *c)) std::swap(*first, *c);
        else std::swap(*first, *a);
    } else if (sk_lt(*a, *c)) std::swap(*first, *a);
    else if (sk_lt(*mid, *c)) std::swap(*first, *c);
    else std::swap(*first, *mid);
}
void sort_loop(SortKey *first, SortKey *last, int depth) {  // std::__introsort_loop
    while (last - first > 16) {
        if (depth == 0) { std::partial_sort(first, last, last, sk_lt); break; }
        --depth;
        median_to_first(first, last);
        SortKey *lo = first + 1, *hi = last;  // std::__unguarded_partition(first+1, last, first)
        for (;;) {
            while (sk_lt(*lo, *first)) ++lo;
            --hi;
            while (sk_lt(*first, *hi)) --hi;
            if (!(lo < hi)) break;
            std::swap(*lo, *hi);
            ++lo;
        }
        sort_loop(lo, last, depth);
        last = lo;
    }
}
inline void insertion_sort(SortKey *first, SortKey *last) {  // what the final insertion pass does to one partition
    for (SortKey *i = first + 1; i < last; ++i) {
        const SortKey v = *i;
        SortKey *j = i;
        while (j > first && sk_lt(v, *(j - 1))) { *j = *(j - 1); --j; }
        *j = v;
    }
}
// Closed-form Hoare partition of [first+1, last) around *first, all threads together.  Returns the cut.
// One scan: thread t writes the positions of its chunk [a_t, b_t) that belong to L / R into Lg / Rg starting at a_t (a chunk
// cannot hold more of them than it has elements); rank i of the whole list lives at Lg[a_t + i - cl[t]] for the t with
// cl[t] <= i < cl[t+1].
struct Ranked {  // access by rank to the per-chunk position lists
    const std::vector<uint32_t> &g; const std::vector<size_t> &cum, &start; int T;
    int chunk_of(size_t i) const { int lo = 0, hi = T - 1; while (lo < hi) { const int m = (lo + hi + 1) >> 1; if (cum[(size_t)m] <= i) lo = m; else hi = m - 1; } return lo; }
    uint32_t at(size_t i) const { const int t = chunk_of(i); return g[start[(size_t)t] + (i - cum[(size_t)t])]; }
};
SortKey *partition_parallel(SortKey *first, SortKey *last, int T, std::vector<uint32_t> &Lg, std::vector<uint32_t> &Rg) {
    SortKey *base = first + 1;
    const size_t n = (size_t)(last - base);
    const SortKey piv = *first;
    std::vector<size_t> cl((size_t)T + 1, 0), cr((size_t)T + 1, 0), st((size_t)T + 1, 0);
    if (Lg.size() < n) { Lg.resize(n); Rg.resize(n); }
    for (int t = 0; t <= T; t++) st[(size_t)t] = n * (size_t)t / (size_t)T;
#pragma omp parallel num_threads(T)
    {
        const int t = omp_get_thread_num();
        const size_t a = st[(size_t)t], b = st[(size_t)t + 1];
        size_t wl = a, wr = a;
        for (size_t i = a; i < b; i++) {
            const uint64_t k = base[i].key;
            if (!(k < piv.key)) Lg[wl++] = (uint32_t)i;
            if (!(piv.key < k)) Rg[wr++] = (uint32_t)i;   // ascending here; R[i] of the text is rank nR-1-i
        }
        cl[(size_t)t + 1] = wl - a; cr[(size_t)t + 1] = wr - a;
    }
    for (int q = 0; q < T; q++) { cl[(size_t)q + 1] += cl[(size_t)q]; cr[(size_t)q + 1] += cr[(size_t)q]; }
    const size_t nL = cl[(size_t)T], nR = cr[(size_t)T];
    const Ranked L{Lg, cl, st, T}, R{Rg, cr, st, T};
    // m = #{i : L[i] < R[i]}: the predicate is monotone in i
    size_t lo = 0, hi = std::min(nL, nR);
    while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (L.at(mid) < R.at(nR - 1 - mid)) lo = mid + 1; else hi = mid; }
    const size_t m = lo;
#pragma omp parallel num_threads(T)
    {
        const int t = omp_get_thread_num();
        const size_t i0 = m * (size_t)t / (size_t)T, i1 = m * (size_t)(t + 1) / (size_t)T;
        if (i0 < i1) {
            int tl = L.chunk_of(i0), tr = R.chunk_of(nR - 1 - i0);  // walk the chunks instead of searching per element
            for (size_t i = i0; i < i1; i++) {
                while (cl[(size_t)tl + 1] <= i) tl++;
                const size_t j = nR - 1 - i;
                while (cr[(size_t)tr] > j) tr--;
                std::swap(base[Lg[st[(size_t)tl] + (i - cl[(size_t)tl])]], base[Rg[st[(size_t)tr] + (j - cr[(size_t)tr])]]);
            }
        }
    }
    size_t cut;
    if (m == 0) cut = L.at(0);
    else cut = (m < nL && L.at(m) < R.at(nR - m)) ? L.at(m) : R.at(nR - m);  // R[m-1] is ascending rank nR-m
    return base + cut;
}
void sort_like_std(SortKey *first, SortKey *last, int threads) {
    if (first == last) return;
    int lg = 0;
    for (size_t n = (size_t)(last - first); n > 1; n >>= 1) lg++;
    struct Range { SortKey *a, *b; int depth; };
    const int T = std::max(1, std::min(threads, 32));
    const ptrdiff_t kBig = 1 << 15;  // ranges above this are partitioned by all threads together
    std::vector<Range> big, small;
    big.push_back(Range{first, last, 2 * lg});
    std::vector<uint32_t> Lg, Rg;
    while (!big.empty()) {
        Range r = big.back();
        big.pop_back();
        if (T == 1 || r.b - r.a <= kBig || r.depth == 0) { small.push_back(r); continue; }
        median_to_first(r.a, r.b);
        SortKey *cut = partition_parallel(r.a, r.b, T, Lg, Rg);
        big.push_back(Range{r.a, cut, r.depth - 1});
        big.push_back(Range{cut, r.b, r.depth - 1});
    }
    // the remaining partitions: sequential introsort loop + their share of the final insertion sort, one task each
    // (no barriers inside: this loop may use every core even while the caller's thread spins on the GPU)
    std::sort(small.begin(), small.end(), [](const Range &x, const Range &y) { return x.b - x.a > y.b - y.a; });  // largest first
#pragma omp parallel for num_threads(std::max(T, std::min(2 * T, omp_get_num_procs()))) schedule(dynamic, 1)
    for (long long i = 0; i < (long long)small.size(); i++) {
        sort_loop(small[(size_t)i].a, small[(size_t)i].b, small[(size_t)i].depth);
        insertion_sort(small[(size_t)i].a, small[(size_t)i].b);
    }
}
}  // namespace
void sort_keys_like_std(SortKey *first, SortKey *last, int threads) { sort_like_std(first, last, threads); }

// test hook: does sort_like_std reproduce std::sort's permutation (payload included) on n keys drawn from [0,range)?
extern "C" int sqh_selftest_sort(int64_t n, uint64_t seed, uint64_t range, int pattern, int fanout) {
    std::vector<SortKey> a((size_t)n), b;
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1;
    for (int64_t i = 0; i < n; i++) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        uint64_t v = range ? x % range : 0;
        if (pattern == 1) v = (uint64_t)i / 3;                 // sorted with ties
        else if (pattern == 2) v = (uint64_t)(n - i) / 3;      // reversed with ties
        else if (pattern == 3) v = (uint64_t)std::min(i, n - 1 - i);  // organ pipe
        a[(size_t)i] = SortKey{v, (uint32_t)i};
    }
    b = a;
    std::sort(a.begin(), a.end(), sk_lt);
    sort_like_std(b.data(), b.data() + b.size(), fanout == 0 ? 1 : (fanout < 0 ? omp_get_num_procs() : fanout));
    for (size_t i = 0; i < a.size(); i++) if (a[i].key != b[i].key || a[i].k != b[i].k) return 0;
    return 1;
}

// test hook: milliseconds sort_like_std needs for n random keys from [0,range) on `threads` threads
extern "C" double sqh_time_sort(int64_t n, uint64_t seed, uint64_t range, int threads) {
    std::vector<SortKey> a((size_t)n);
    uint64_t x = seed * 0x9E3779B97F4A7C15ull + 1;
    for (int64_t i = 0; i < n; i++) { x ^= x << 13; x ^= x >> 7; x ^= x << 17; a[(size_t)i] = SortKey{range ? x % range : 0, (uint32_t)i}; }
    const auto t0 = std::chrono::steady_clock::now();
    sort_like_std(a.data(), a.data() + a.size(), threads <= 0 ? omp_get_num_procs() : threads);
    return 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

void chimeric_prepass(const sqg_chimeric &c, int32_t n_ref, int32_t read_len, ChimPrepass &out) {
    const bool timing = getenv("SQH_TIMING") != nullptr;
    auto T0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *w) { if (timing) { auto t = std::chrono::steady_clock::now(); fprintf(stderr, "[prepass] %s %.1f ms\n", w, 1e3 * std::chrono::duration<double>(t - T0).count()); T0 = t; } };
    // buffers are reused from call to call (thread-local scratch, `out` keeps its capacity): at a few hundred thousand reads
    // allocation, first-touch page faults and value-initialisation cost as much as the work itself
    out.part_chr.clear(); out.part_pos.clear(); out.groups.clear();
    typedef SortKey DB;  // key = (RefID,RefPos) packed, k = block index
    // The read loop (:206-262) is split into contiguous chunks of reads, one per thread; chunk results are concatenated in
    // order.  The only coupling between reads is `bamdiscordant.back()` at :257: a chunk that has not pushed a discordant
    // block yet defers that test until the chunks before it are known.
    const int local_ranks = getenv("LOCAL_WORLD_SIZE") ? std::max(1, atoi(getenv("LOCAL_WORLD_SIZE"))) : 1;  // one process per GPU shares the host
    // half the cores, split between the processes of the node: the calling threads spin on their GPUs meanwhile (and NCCL has
    // its own), and an oversubscribed OpenMP team pays for every barrier
    int cores = std::max(local_ranks == 1 ? 1 : 2, omp_get_num_procs() / 2 / local_ranks);
    if (getenv("SQH_PREPASS_THREADS")) cores = std::max(1, atoi(getenv("SQH_PREPASS_THREADS")));  // tuning hook
    int T = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)cores, 16, c.n_reads / 4096 + 1}));
    if (getenv("SQH_PREPASS_CHUNKS")) T = std::max(1, atoi(getenv("SQH_PREPASS_CHUNKS")));  // test hook: force the chunked path on small inputs
    struct Chunk { std::vector<DB> dis; std::vector<std::pair<int, int>> part; std::vector<uint32_t> pend; };
    static thread_local std::vector<Chunk> tl_chunks;
    static thread_local std::vector<DB> tl_dis;
    std::vector<Chunk> &chunks = tl_chunks;  // (references: the OpenMP workers must see the caller's instances, not their own)
    std::vector<DB> &dis = tl_dis;
    if (chunks.size() < (size_t)T) chunks.resize((size_t)T);
    for (Chunk &ch : chunks) { ch.dis.clear(); ch.part.clear(); ch.pend.clear(); }
    auto same_block = [&](uint32_t l, uint32_t b) {  // SingleBamRec_t::Same(): every field incl. IsFirstRead; b is a SecondMate block
        const uint32_t *ro = c.read_off;
        int64_t lo = 0, hi = c.n_reads;  // read owning block l
        while (lo < hi) { const int64_t m2 = (lo + hi) >> 1; if (ro[m2 + 1] <= l) lo = m2 + 1; else hi = m2; }
        const bool l_first = l - ro[lo] < c.n_first[lo];
        return c.blk_ref_id[l] == c.blk_ref_id[b] && c.blk_ref_pos[l] == c.blk_ref_pos[b] && c.blk_read_pos[l] == c.blk_read_pos[b] &&
               c.blk_match_read[l] == c.blk_match_read[b] && c.blk_match_ref[l] == c.blk_match_ref[b] &&
               (c.blk_is_reverse[l] != 0) == (c.blk_is_reverse[b] != 0) && l_first == false;
    };
#pragma omp parallel for num_threads(T) schedule(static, 1)
    for (int t = 0; t < T; t++) {
        Chunk &ch = chunks[(size_t)t];
        std::vector<DB> &dis = ch.dis;
        std::vector<std::pair<int, int>> &part = ch.part;
        auto push_dis = [&](uint32_t k) { dis.push_back(DB{((uint64_t)(uint32_t)c.blk_ref_id[k] << 32) | (uint32_t)c.blk_ref_pos[k], k}); };
        const int64_t i0 = c.n_reads * t / T, i1 = c.n_reads * (t + 1) / T;
        for (int64_t i = i0; i < i1; i++) {
            const uint32_t o = c.read_off[i], e = c.read_off[i + 1], nf = c.n_first[i];
            const View v{c, o, o + nf, e};
            const int32_t ft = c.first_total_len[i], st_ = c.second_total_len[i];
            const bool fl = c.first_lowphred[i], sl = c.second_lowphred[i], mf = c.multi_filter[i];
            const bool fempty = v.f0 == v.f1, sempty = v.f1 == v.s1;
            const bool single = (fempty || sempty) && !mf;
            if (end_disc(v, v.f0, v.f1) || end_disc(v, v.f1, v.s1) || single || pair_disc(v, ft, st_)) {  // :208-213
                for (uint32_t k = o; k < e; k++) push_dis(k);
                continue;
            }
            bool fin = false, sin = false;
            for (int m = 0; m < 2; m++) {  // blocks of one mate more than 750 kb apart (:217-239)
                const uint32_t a = m ? v.f1 : v.f0, b = m ? v.s1 : v.f1;
                int64_t prev = -1;
                for (uint32_t k = a; k + 1 < b; k++)
                    if (std::abs(v.pos(k) - v.pos(k + 1)) > 750000) {
                        if (prev != (int64_t)k) push_dis(k);
                        push_dis(k + 1);
                        prev = k + 1;
                        if (k + 1 == b - 1) (m ? sin : fin) = true;
                    }
            }
            if (!fempty && !sempty && std::abs(v.pos(v.f1 - 1) - v.pos(v.s1 - 1)) > 750000) {  // :240-249
                if (!fin) { push_dis(v.f1 - 1); fin = true; }
                if (!sin) { push_dis(v.s1 - 1); sin = true; }
            }
            if (!fin && !sin) {  // soft-clipped ends of otherwise concordant chimeric reads (:250-259)
                if (!fempty && v.rpos(v.f0) > 15 && !fl) part.push_back({v.chr(v.f0), v.rev(v.f0) ? v.pos(v.f0) + v.mref(v.f0) : v.pos(v.f0)});
                if (!fempty) { const uint32_t b = v.f1 - 1; if (ft - v.rpos(b) - v.mread(b) > 15 && !fl) part.push_back({v.chr(b), v.rev(b) ? v.pos(b) : v.pos(b) + v.mref(b)}); }
                if (!sempty && v.rpos(v.f1) > 15 && !sl) part.push_back({v.chr(v.f1), v.rev(v.f1) ? v.pos(v.f1) + v.mref(v.f1) : v.pos(v.f1)});
                if (!sempty) {
                    const uint32_t b = v.s1 - 1;
                    if (st_ - v.rpos(b) - v.mread(b) > 15 && !sl) {
                        // `!bamdiscordant.back().Same(SecondMate.back())` (:257); back() of an empty vector is UB in the
                        // reference, we read it as "not the same".
                        if (dis.empty()) ch.pend.push_back(b);  // decided when the earlier chunks are known
                        else if (!same_block(dis.back().k, b)) part.push_back({v.chr(b), v.rev(b) ? v.pos(b) : v.pos(b) + v.mref(b)});
                    }
                }
            }
        }
    }
    std::vector<std::pair<int, int>> part((size_t)n_ref, std::make_pair(0, 0));  // resize()d then appended (:203-204)
    {
        size_t nd = 0, np = part.size();
        std::vector<size_t> off((size_t)T + 1, 0);
        for (int t = 0; t < T; t++) { const Chunk &ch = chunks[(size_t)t]; off[(size_t)t + 1] = off[(size_t)t] + ch.dis.size(); np += ch.part.size() + ch.pend.size(); }
        nd = off[(size_t)T];
        if (dis.size() != nd) dis.resize(nd);
        part.reserve(np);
        for (int t = 0; t < T; t++) {
            const Chunk &ch = chunks[(size_t)t];
            for (uint32_t b : ch.pend) {  // `bamdiscordant.back()` as the earlier chunks left it
                int q = t - 1;
                while (q >= 0 && chunks[(size_t)q].dis.empty()) q--;
                if (q < 0 || !same_block(chunks[(size_t)q].dis.back().k, b)) part.push_back({c.blk_ref_id[b], c.blk_is_reverse[b] ? c.blk_ref_pos[b] : c.blk_ref_pos[b] + c.blk_match_ref[b]});
            }
            part.insert(part.end(), ch.part.begin(), ch.part.end());
        }
#pragma omp parallel for num_threads(T) schedule(static, 1)
        for (int t = 0; t < T; t++) std::copy(chunks[(size_t)t].dis.begin(), chunks[(size_t)t].dis.end(), dis.begin() + (ptrdiff_t)off[(size_t)t]);
    }
    lap("reads");
    std::sort(part.begin(), part.end(), [](std::pair<int, int> a, std::pair<int, int> b) { return a.first == b.first ? a.second < b.second : a.first < b.first; });
    // Same unstable std::sort, same ordering relation, same input sequence as :264 => the same permutation, including
    // the order among equal (RefID,RefPos) which the sub-cluster walk observes (SURVEY.md App. A-11).  The packed key
    // compares exactly like operator< of SingleBamRec_t (RefID, RefPos are non-negative here).
    lap("part sort");
    sort_like_std(dis.data(), dis.data() + dis.size(), std::min(cores, 16));
    lap("disc sort");
    out.part_chr.reserve(part.size()); out.part_pos.reserve(part.size());
    for (auto &p : part) { out.part_chr.push_back(p.first); out.part_pos.push_back(p.second); }
    if (out.disc.capacity() < dis.size() + 1) {
        out.disc.clear();
        out.disc.reserve(dis.size() + 1 + dis.size() / 8);  // head room: the storage survives slightly larger inputs
    }
    if (out.disc.size() != dis.size() + 1) out.disc.resize(dis.size() + 1);
    {   // gather the sorted blocks (random access into the caller's arrays)
        const long long nd = (long long)dis.size();
#pragma omp parallel for num_threads(std::min(cores, 16)) schedule(static)
        for (long long i = 0; i < nd; i++) {
            const uint32_t k = dis[(size_t)i].k;
            out.disc[(size_t)i] = sq::DiscBlock{c.blk_ref_id[k], c.blk_ref_pos[k], c.blk_match_ref[k], c.blk_is_reverse[k] ? 1 : 0};
        }
    }
    const int32_t n = (int32_t)dis.size();
    out.disc[dis.size()] = sq::DiscBlock{0, 0, 0, 0};  // what *cend() reads (SURVEY App. A-5)
    // :341-348 chain while the next block starts within ReadLen of the running right end.  In sorted order the running right
    // end of a group equals the maximum end over ALL earlier blocks of the chromosome (the previous group ended more than
    // ReadLen left of this one), so block e opens a group iff it is the first of its chromosome or starts at/after that
    // prefix maximum + ReadLen: a prefix maximum per chunk of blocks, chunks in parallel.
    {
        int TG = n > (1 << 16) ? std::min(cores, 16) : 1;
        if (getenv("SQH_PREPASS_CHUNKS")) TG = std::max(1, std::min(n, atoi(getenv("SQH_PREPASS_CHUNKS"))));  // test hook
        struct Tail { int32_t chr, mx; bool any; };
        std::vector<Tail> tail((size_t)TG);
        std::vector<std::vector<std::pair<int32_t, int32_t>>> brk((size_t)TG);  // (block index that opens a group, right end of the group before it)
#pragma omp parallel num_threads(TG)
        {
            const int t = omp_get_thread_num();
            const int32_t a = (int32_t)((int64_t)n * t / TG), b = (int32_t)((int64_t)n * (t + 1) / TG);
            Tail tl{-1, 0, false};  // last chromosome of the chunk and the maximum end seen on it inside the chunk
            for (int32_t e = a; e < b; e++) {
                const sq::DiscBlock &d = out.disc[(size_t)e];
                if (!tl.any || d.chr != tl.chr) { tl.chr = d.chr; tl.mx = d.pos + d.len; tl.any = true; }
                else tl.mx = std::max(tl.mx, d.pos + d.len);
            }
            tail[(size_t)t] = tl;
#pragma omp barrier
            // carry into this chunk: maximum end over the earlier chunks on the chromosome they end with
            int32_t cchr = -1, cmx = 0;
            bool cany = false;
            for (int q = 0; q < t; q++) {
                const Tail &x = tail[(size_t)q];
                if (!x.any) continue;
                if (cany && x.chr == cchr) {
                    // the chunk may hold earlier chromosomes too; its tail maximum is about its LAST chromosome only, which
                    // equals cchr here, so the maxima combine
                    cmx = std::max(cmx, x.mx);
                    // ... unless the chunk changed chromosome and came back (impossible in sorted order)
                } else { cchr = x.chr; cmx = x.mx; cany = true; }
            }
            int32_t rchr = cchr, rmx = cmx;
            bool rany = cany;
            for (int32_t e = a; e < b; e++) {
                const sq::DiscBlock &d = out.disc[(size_t)e];
                const bool opens = !rany || d.chr != rchr || d.pos >= rmx + read_len;
                if (opens) brk[(size_t)t].push_back({e, rany ? rmx : 0});
                if (!rany || d.chr != rchr) { rchr = d.chr; rmx = d.pos + d.len; rany = true; }
                else rmx = std::max(rmx, d.pos + d.len);
            }
            if (t == TG - 1) tail[(size_t)t] = Tail{rchr, rmx, rany};  // the true running state at the end of the list
        }
        size_t ng = 0;
        for (auto &v : brk) ng += v.size();
        out.groups.reserve(ng);
        int32_t prev_start = -1;
        for (auto &v : brk)
            for (auto &pr : v) {
                if (prev_start >= 0) out.groups.push_back(sq::Group{prev_start, pr.first, out.disc[(size_t)prev_start].chr, pr.second});
                prev_start = pr.first;
            }
        if (prev_start >= 0) out.groups.push_back(sq::Group{prev_start, n, out.disc[(size_t)prev_start].chr, tail[(size_t)TG - 1].mx});
    }
    lap("groups");
}
}  // namespace sqh

// test / tuning hook: milliseconds of the `iters`-th consecutive pre-pass of the same reads (buffers warm, as in a context)
extern "C" double sqh_time_prepass(const sqg_chimeric *c, int32_t n_ref, int32_t read_len, int iters) {
    sqh::ChimPrepass pre;
    double ms = 0;
    for (int i = 0; i < iters; i++) {
        const auto t0 = std::chrono::steady_clock::now();
        sqh::chimeric_prepass(*c, n_ref, read_len, pre);
        ms = 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
    return ms;
}
