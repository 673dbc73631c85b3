// TEST TOOLING — CPU stepping harness for the device-side rules.
//
// There is no GPU in the development container, so this program steps the SAME `SQ_HD`
// element functions the CUDA kernels call (squid_b200/csrc/*.cuh) over plain loops, with
// std::sort / running maxima standing in for the device-wide sort and scan primitives.  It exists
// to debug the data-parallel restatement against the reference-built oracle before spending GPU
// time; it is NOT a product path (the product library has no CPU fallback and never links this).
// Dumps use the oracle harness's file names so the same comparison script reads both.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_set>
#include <vector>

#include "host/chimeric.h"
#include "host/prepass.h"
#include "sq_classify.cuh"
#include "sq_depth_cover.cuh"
#include "sq_locate.cuh"
#include "sq_seed.cuh"

using namespace sq;

static std::string outdir;
static void dump_i32(const std::string &name, const std::vector<int32_t> &v) {
    FILE *f = fopen((outdir + "/" + name).c_str(), "wb");
    if (!f) { fprintf(stderr, "cannot write %s\n", name.c_str()); exit(2); }
    if (!v.empty()) fwrite(v.data(), 4, v.size(), f);
    fclose(f);
}

struct EdgeVec {
    std::vector<uint64_t> *v;
    void operator()(uint64_t k) { v->push_back(k); }
};

int main(int argc, char **argv) {
    if (argc < 4) { fprintf(stderr, "usage: %s conc.sqmb chim.sqmb outdir [bps.bin]\n", argv[0]); return 2; }
    outdir = argv[3];
    sqh::HostConfig cfg;
    if (getenv("SQ_EMUL_DP")) cfg.concord_dist_pos = atoi(getenv("SQ_EMUL_DP"));  // -dp (Concord_Dist_Pos)
    if (getenv("SQ_EMUL_DI")) cfg.concord_dist_idx = atoi(getenv("SQ_EMUL_DI"));  // -di (Concord_Dist_Idx)
    SqmbView conc, chim;
    if (!conc.open(argv[1]) || !chim.open(argv[2])) { fprintf(stderr, "cannot open inputs\n"); return 2; }
    std::vector<sqh::Read> reads;
    sqh::load_chimeric(chim, cfg, reads);
    std::unordered_set<std::string> names;
    names.insert("");  // the pre-sized empty strings of ChimName (SURVEY App. A-3)
    for (auto &r : reads) names.insert(r.qname);
    sqh::PackedBatch pb;
    std::string err;
    if (sqh::pack_concordant(conc, cfg, names, pb, err)) { fprintf(stderr, "%s\n", err.c_str()); return 2; }
    sqh::PackedChimeric pc;
    pc.from_reads(reads);
    sqg_chimeric cview = pc.view();
    sqg_batch hb = pb.view();
    const int32_t n_ref = (int32_t)conc.n_ref;
    sqh::ChimPrepass pre;
    sqh::chimeric_prepass(cview, n_ref, cfg.read_len, pre);

    DevBatch b;
    b.n_rec = hb.n_rec; b.n_blk = hb.n_blk; b.ref_id = hb.ref_id; b.pos = hb.pos; b.mate_ref_id = hb.mate_ref_id; b.mate_pos = hb.mate_pos;
    b.end_pos = hb.end_pos; b.flag = hb.flag; b.total_len = hb.total_len; b.lowphred_run = hb.lowphred_run; b.mapq = hb.mapq; b.aux = hb.aux;
    b.blk_off = hb.blk_off; b.blk_ref_pos = hb.blk_ref_pos; b.blk_match_ref = hb.blk_match_ref; b.blk_read_pos = hb.blk_read_pos; b.blk_match_read = hb.blk_match_read;
    Params p;
    p.min_mapq = cfg.min_mapq; p.max_lowphred_len = cfg.max_lowphred_len; p.concord_dist_pos = cfg.concord_dist_pos;
    p.concord_dist_idx = cfg.concord_dist_idx; p.read_len = cfg.read_len; p.n_ref = n_ref;
    const int64_t n = b.n_rec;

    // ---- classify + scans ----
    std::vector<uint8_t> cls(n);
    std::vector<uint16_t> first_len(n, 0);
    std::vector<uint64_t> other_excl(n);
    const int32_t cc_tile = getenv("SQ_EMUL_CC_TILE") ? atoi(getenv("SQ_EMUL_CC_TILE")) : 512;  // 0: no per-tile maxima (plain walks)
    std::vector<int32_t> ccmax(cc_tile > 0 ? (size_t)((n + cc_tile - 1) / cc_tile) + 1 : 1, kNoCcEnd);
    {
        int64_t prev = -1;
        uint64_t run = 1ull << 32;
        for (int64_t r = 0; r < n; r++) {
            ClassifyOut o = classify_record(b, p, r, prev);
            cls[r] = o.cls;
            first_len[r] = (uint16_t)(o.first_len < 65535 ? o.first_len : 65535);
            other_excl[r] = run;
            if (cc_tile > 0) {
                int32_t &m = ccmax[(size_t)(r / cc_tile)];
                const int64_t t0 = r / cc_tile * cc_tile, t1 = std::min<int64_t>(t0 + cc_tile, n) - 1;
                if (b.ref_id[t0] < 0 || b.ref_id[t0] != b.ref_id[t1]) m = kCcWalkTile;
                else if (o.cc_end > m) m = o.cc_end;
            }
            if (o.other_key > run) run = o.other_key;
            if (o.cls & CLS_GATE) prev = r;
        }
    }
    std::vector<int32_t> gap, pcrec, dprec;
    std::vector<uint64_t> gap_other;
    int32_t lmax = 0;
    int64_t first_kept = n;
    for (int64_t r = 0; r < n; r++) {
        if (!(cls[r] & CLS_KEEP)) continue;
        if (first_kept == n) first_kept = r;
        const int32_t oc = (int32_t)(other_excl[r] >> 32) - 1, orr = (int32_t)(uint32_t)other_excl[r];
        if (b.ref_id[r] != oc || b.pos[r] > orr + p.read_len) { gap.push_back((int32_t)r); gap_other.push_back(other_excl[r]); }
        if (cls[r] & CLS_PART) pcrec.push_back((int32_t)r);
        if ((cls[r] & CLS_CONC) && (cls[r] & CLS_DISPL)) dprec.push_back((int32_t)r);
        if (cls[r] & CLS_CONC) lmax = std::max(lmax, b.blk_match_ref[b.blk_off[r]]);
    }
    if (getenv("SQ_EMUL_CLASSIFY")) {  // phase 1's outputs, in the layouts of sqg_classify_dump; then stop
        outdir = getenv("SQ_EMUL_CLASSIFY");
        dump_i32("cls_i32.bin", std::vector<int32_t>(cls.begin(), cls.end()));
        dump_i32("first_len_i32.bin", std::vector<int32_t>(first_len.begin(), first_len.end()));
        dump_i32("gap_rec_i32.bin", gap);
        std::vector<int32_t> go;
        for (uint64_t k : gap_other) { go.push_back((int32_t)(k >> 32)); go.push_back((int32_t)(uint32_t)k); }
        dump_i32("gap_key_2xi32.bin", go);
        dump_i32("pc_rec_i32.bin", pcrec);
        dump_i32("dp_rec_i32.bin", dprec);
        dump_i32("lmax_first_kept_i32.bin", std::vector<int32_t>{lmax, (int32_t)first_kept});
        return 0;
    }
    const int32_t nD = (int32_t)pre.disc.size() - 1, nG = (int32_t)pre.groups.size();
    std::vector<int64_t> trig(nG);
    for (int32_t g = 0; g < nG; g++) {
        const Group &G = pre.groups[g];
        int64_t lo = 0, hi = n;
        while (lo < hi) {
            int64_t m = (lo + hi) >> 1;
            const bool past = b.ref_id[m] < 0 || G.chr < b.ref_id[m] || (G.chr == b.ref_id[m] && G.right < b.pos[m]);
            if (!past) lo = m + 1; else hi = m;
        }
        while (lo < n && !(cls[lo] & CLS_KEEP)) lo++;
        trig[g] = lo;
    }
    // ConcordRest candidates, binned by group: a non-first block of a concordant record belongs to the last group whose
    // (start - ReadLen) lies at or left of it, if it starts left of that group's right end + ReadLen
    std::vector<RestBlock> rest;
    std::vector<uint32_t> rest_g;
    {
        std::vector<std::pair<uint32_t, RestBlock>> tmp;
        for (int64_t r = 0; r < n; r++) {
            if (!(cls[r] & CLS_CONC) || !(b.flag[r] & 0xC0)) continue;
            for (uint32_t k = b.blk_off[r] + 1; k < b.blk_off[r + 1]; k++) {
                const int32_t c = b.ref_id[r], q = b.blk_ref_pos[k];
                int32_t gi = -1;
                for (int32_t g = 0; g < nG; g++) {
                    const Group &G = pre.groups[g];
                    const int32_t s0 = pre.disc[G.ds].pos - p.read_len;
                    if (G.chr < c || (G.chr == c && s0 <= q)) gi = g; else break;
                }
                if (gi < 0 || pre.groups[gi].chr != c || q >= pre.groups[gi].right + p.read_len) continue;
                tmp.push_back({(uint32_t)gi, RestBlock{c, q, q + b.blk_match_ref[k], (int32_t)r}});
            }
        }
        std::stable_sort(tmp.begin(), tmp.end(), [](const std::pair<uint32_t, RestBlock> &a, const std::pair<uint32_t, RestBlock> &c) { return a.first < c.first; });
        for (auto &x : tmp) { rest_g.push_back(x.first); rest.push_back(x.second); }
    }

    // ---- seed machine ----
    SeedMachine sm;
    sm.in.b = b; sm.in.cls = cls.data(); sm.in.first_len = first_len.data(); sm.in.gap_other = gap_other.data();
    sm.in.gap_rec = gap.data(); sm.in.n_gap = (int32_t)gap.size();
    sm.in.pc_rec = pcrec.data(); sm.in.n_pc = (int32_t)pcrec.size();
    sm.in.D = pre.disc.data(); sm.in.nD = nD; sm.in.G = pre.groups.data(); sm.in.nG = nG;
    sm.in.trigger = trig.data();
    sm.in.Pchr = pre.part_chr.data(); sm.in.Ppos = pre.part_pos.data(); sm.in.nP = (int32_t)pre.part_chr.size();
    sm.in.rest = rest.data(); sm.in.rest_g = rest_g.data(); sm.in.n_rest = (int32_t)rest.size();
    sm.in.read_len = p.read_len;
    if (cc_tile > 0) { sm.in.ccmax = ccmax.data(); sm.in.cc_tile = cc_tile; }
    sm.in.dp_rec = dprec.data(); sm.in.n_dp = (int32_t)dprec.size(); sm.in.lmax = lmax; sm.in.n_rec = n; sm.in.first_kept = first_kept;
    std::vector<int32_t> margin(6 * 2 * (4 * (size_t)nD + 2 * pre.part_chr.size() + 2 * pcrec.size() + 64) + 8 + (getenv("SQ_EMUL_DENSE") ? 6 * 2 * (size_t)atoi(getenv("SQ_EMUL_DENSE")) : 0));
    sm.margin = margin.data(); sm.margin_cap = (int32_t)margin.size();
    if (getenv("SQ_EMUL_DENSE")) { sm.use_dense = true; sm.in.dense_max_r = atoi(getenv("SQ_EMUL_DENSE")); }  // position-indexed break tables (heavy islands on the device)
    // islands: cut before group g when the machine provably restarts there
    std::vector<int32_t> isl_start(1, 0);
    const bool one_island = getenv("SQ_EMUL_ONE_ISLAND") != nullptr;
    for (int32_t g = 1; g < nG && !one_island; g++) if (sm.island_cut(g)) isl_start.push_back(g);
    const int32_t nI = (int32_t)isl_start.size();
    isl_start.push_back(nG);
    std::vector<std::vector<SeedOp>> ops(nI);
    std::vector<int32_t> gdone(nI, 0);
    auto run = [&](int32_t i, bool inherited) {
        ops[i].assign(4 * (size_t)(pre.groups[isl_start[i + 1] - 1].de - pre.groups[isl_start[i]].ds) + 16, SeedOp{});
        sm.out = ops[i].data(); sm.out_cap = (int32_t)ops[i].size();
        gdone[i] = sm.run_island(isl_start[i], isl_start[i + 1], inherited);
        if (sm.error) { fprintf(stderr, "seed machine error %d\n", sm.error); exit(3); }
        ops[i].resize(sm.st.n_out);
    };
    // sequential prefix: until some island has emitted a segment the machine truly has no last segment
    int32_t ip = 0;
    for (; ip < nI; ip++) { run(ip, false); if (!ops[ip].empty()) { ip++; break; } }
    // the rest is order independent: run it backwards to prove it
    for (int32_t i = nI - 1; i >= ip; i--) run(i, true);
    std::vector<SeedNode> seeds;
    int32_t g_done = nG;
    for (int32_t i = 0; i < nI; i++) {
        stitch_ops(ops[i].data(), (int32_t)ops[i].size(), seeds);
        if (gdone[i] < isl_start[i + 1]) { g_done = gdone[i]; break; }
    }
    fprintf(stderr, "emul: %d groups, %d islands, %zu seeds, lmax %d, %zu displaced, sub-clusters dense %d sparse %d\n", nG, nI, seeds.size(), lmax, dprec.size(), sm.n_dense, sm.n_sparse);
    {
        std::vector<int32_t> s;
        for (auto &x : seeds) { s.push_back(x.chr); s.push_back(x.pos); s.push_back(x.len); }
        dump_i32("seeds_i32.bin", s);
    }
    // break index for the depth streams (:338-339)
    int64_t r_break = n;  // exclusive bound of records that feed ReadsMain/ReadsOther
    if (g_done == nG && nG > 0) {
        int64_t r = trig[nG - 1] + 1;
        while (r < n && !(cls[r] & CLS_KEEP)) r++;
        r_break = r < n ? r + 1 : n;
    }
    // ---- normalise + tile (SegmentGraph.cpp:19-38, 714-761) ----
    std::sort(seeds.begin(), seeds.end(), [](const SeedNode &a, const SeedNode &c) { return a.chr != c.chr ? a.chr < c.chr : (a.pos != c.pos ? a.pos < c.pos : a.len < c.len); });
    std::vector<SeedNode> norm;
    for (auto &s : seeds) {
        if (norm.empty() || norm.back().chr != s.chr || norm.back().pos + norm.back().len <= s.pos) norm.push_back(s);
        else norm.back().len = std::max(norm.back().pos + norm.back().len, s.pos + s.len) - norm.back().pos;
    }
    std::vector<int32_t> nchr, npos, nend;
    if (const char *nf = getenv("SQ_EMUL_NODES")) {  // an injected table (the graph-reload seam): int32 rows chr, pos, len
        FILE *f = fopen(nf, "rb");
        if (!f) { fprintf(stderr, "cannot open %s\n", nf); return 2; }
        int32_t row[3];
        while (fread(row, 4, 3, f) == 3) { nchr.push_back(row[0]); npos.push_back(row[1]); nend.push_back(row[1] + row[2]); }
        fclose(f);
    } else {
        size_t k = 0;
        for (int32_t c = 0; c < n_ref; c++) {
            int32_t cur = 0;
            bool any = false;
            for (; k < norm.size() && norm[k].chr == c; k++) {
                int32_t s = norm[k].pos, e = norm[k].pos + norm[k].len;
                if (s - cur > 100) { nchr.push_back(c); npos.push_back(cur); nend.push_back(s); }
                else s = cur;
                nchr.push_back(c); npos.push_back(s); nend.push_back(e);
                cur = e; any = true;
            }
            if (!any || cur != conc.ref_len[c]) { nchr.push_back(c); npos.push_back(cur); nend.push_back(conc.ref_len[c]); }
        }
    }
    const int32_t N = (int32_t)nchr.size();
    std::vector<int32_t> chr_first(n_ref + 1, N);
    for (int32_t i = N - 1; i >= 0; i--) chr_first[nchr[i]] = i;
    for (int32_t c = n_ref - 1; c >= 0; c--) if (chr_first[c] == N && c + 1 <= n_ref) chr_first[c] = chr_first[c + 1];
    NodeTable nt;
    nt.n = N; nt.n_ref = n_ref; nt.chr = nchr.data(); nt.pos = npos.data(); nt.end = nend.data(); nt.chr_first = chr_first.data();
    // coarse position index, as sqg_api.cu builds it (a small shift makes every branch of seg_at run on the test cases)
    std::vector<int32_t> bin_off(n_ref + 1, 0), bin_seg;
    nt.bin_shift = getenv("SQ_EMUL_BIN_SHIFT") ? atoi(getenv("SQ_EMUL_BIN_SHIFT")) : 12;
    if (nt.bin_shift > 0) {
        for (int32_t c = 0; c < n_ref; c++) bin_off[c + 1] = bin_off[c] + (conc.ref_len[c] >> nt.bin_shift) + 1;
        bin_seg.resize(bin_off[n_ref]);
        nt.bin_off = bin_off.data();
        for (int32_t c = 0; c < n_ref; c++)
            for (int32_t k = 0; k < bin_off[c + 1] - bin_off[c]; k++) bin_seg[bin_off[c] + k] = bin_seg_value(nt, c, k);
        nt.bin_seg = bin_seg.data();
    }

    // ---- depth ----
    std::vector<int32_t> cnt(3 * (size_t)N, 0), sum(3 * (size_t)N, 0);
    for (int32_t k = 0; k < nD; k++) {
        const DiscBlock &d = pre.disc[k];
        const int32_t c0 = chr_first[d.chr], c1 = chr_first[d.chr + 1];
        int32_t j = seg_last_pos_le(nt, d.chr, c0, c1, d.pos);
        if (j >= c0 && d.pos >= nt.pos[j] && d.pos + d.len <= nt.end[j]) { cnt[j]++; sum[j] += d.len; }
    }
    bool other_nonempty = false;
    std::vector<uint32_t> omask((size_t)N + 1, 0);
    struct ShortBlk { int32_t chr, start, len; };
    std::vector<ShortBlk> shorts;
    int64_t n_unstable = 0;
    {
        int32_t cursor = 0;
        for (int64_t r = 0; r < r_break; r++) {
            if (!(cls[r] & CLS_HASBLK)) continue;
            const uint32_t o = b.blk_off[r];
            const int32_t c = b.ref_id[r];
            const int32_t m = depth_target(nt, c, b.blk_ref_pos[o], b.blk_match_ref[o]);
            if (m > cursor) cursor = m;
            if (cursor != kNoNode && cursor < N && depth_contained(nt, cursor, c, b.blk_ref_pos[o], b.blk_match_ref[o])) {
                cnt[N + cursor]++; sum[N + cursor] += b.blk_match_ref[o];
            }
            for (uint32_t k = o + 1; k < b.blk_off[r + 1]; k++) {
                other_nonempty = true;
                const int32_t st = b.blk_ref_pos[k], l = b.blk_match_ref[k];
                uint32_t bit;
                const int32_t jm = depth_other_mark(nt, c, st, l, &bit);
                if (jm >= 0) omask[jm] |= bit;
                if (l <= kSeedThresh) { shorts.push_back(ShortBlk{c, st, l}); continue; }  // second pass, once the masks are complete
                const int32_t m2 = depth_target(nt, c, st, l);
                if (m2 != kNoNode && depth_contained(nt, m2, c, st, l)) { cnt[2 * N + m2]++; sum[2 * N + m2] += l; }
            }
        }
        std::vector<int32_t> short_node(shorts.size());
        for (size_t q = 0; q < shorts.size(); q++) {
            bool un = false;
            short_node[q] = depth_short_node(nt, omask.data(), shorts[q].chr, shorts[q].start, shorts[q].len, &un);
            if (un) n_unstable++;
        }
        if (n_unstable == 0 || getenv("SQ_EMUL_NO_OTHER_SORT")) {
            for (size_t q = 0; q < shorts.size(); q++)
                if (short_node[q] != kNoNode) { cnt[2 * N + short_node[q]]++; sum[2 * N + short_node[q]] += shorts[q].len; }
        } else {
            // Some short block ties with an entry of the same (chr, start) that would move it: the reference's answer is the order
            // in which its unstable std::sort (:781) leaves the ties.  Same input order, same comparator, same library: sort
            // ReadsOther for real and walk the cursor = running maximum of the entries' own segments.
            std::vector<std::pair<int, std::pair<int, int>>> RO;
            for (int64_t r = 0; r < r_break; r++) {
                if (!(cls[r] & CLS_HASBLK)) continue;
                for (uint32_t k = b.blk_off[r] + 1; k < b.blk_off[r + 1]; k++) RO.push_back(std::make_pair(b.ref_id[r], std::make_pair(b.blk_ref_pos[k], b.blk_match_ref[k])));
            }
            std::sort(RO.begin(), RO.end(), [](std::pair<int, std::pair<int, int>> a, std::pair<int, std::pair<int, int>> c) { if (a.first != c.first) return a.first < c.first; else return (a.second).first < (c.second).first; });
            int32_t cursor = -1;
            for (const auto &e : RO) {
                const int32_t c = e.first, st = e.second.first, l = e.second.second;
                const int32_t own = depth_target(nt, c, st, l);  // long: n(start); short: earliest containing segment, else n(start)
                if (own == kNoNode) { cursor = kNoNode; continue; }
                if (own > cursor) cursor = own;
                if (l <= kSeedThresh && cursor != kNoNode && cursor < N && depth_contained(nt, cursor, c, st, l)) { cnt[2 * N + cursor]++; sum[2 * N + cursor] += l; }
            }
        }
        fprintf(stderr, "emul: %zu short ReadsOther blocks, %lld order-dependent\n", shorts.size(), (long long)n_unstable);
    }
    {
        std::vector<int32_t> a;
        std::vector<double> d;
        for (int32_t i = 0; i < N; i++) {
            a.push_back(nchr[i]); a.push_back(npos[i]); a.push_back(nend[i] - npos[i]);
            a.push_back(cnt[i] + cnt[N + i] + cnt[2 * N + i]);
            double dep = (double)sum[i];
            dep += (double)sum[N + i];
            if (other_nonempty) { dep += (double)sum[2 * N + i]; dep = 1.0 * dep / (nend[i] - npos[i]); }
            d.push_back(dep);
        }
        dump_i32("nodes_i32.bin", a);
        dump_i32("depth_cnt3_i32.bin", cnt);
        dump_i32("depth_sum3_i32.bin", sum);
        FILE *f = fopen((outdir + "/nodes_f64.bin").c_str(), "wb");
        fwrite(d.data(), 8, d.size(), f);
        fclose(f);
    }

    // ---- edges: chimeric reads (RawEdgesChim) then the concordant stream (RawEdgesOther) ----
    std::vector<uint64_t> keys;
    EdgeVec emit{&keys};
    auto run_stream = [&](int mode, int64_t count, auto &&load, auto &&store, auto &&builds) {
        // pass A: every read on its own, hint unknown; pass B: replay the sensitive ones in order with the true hint
        std::vector<int32_t> res0(count, -2);  // -2 = read does not touch the hint
        std::vector<char> sens(count, 0);
        for (int64_t i = 0; i < count; i++) {
            if (!builds(i)) continue;
            Blk F[kMaxBlocks + 1], S[kMaxBlocks + 1];
            ReadView rv; rv.F = F; rv.S = S;
            bool is_first;
            load(i, rv, is_first);
            int32_t node[2 * kMaxBlocks + 2];
            if (rv.nF + rv.nS == 0) continue;
            std::vector<uint64_t> tmp;
            EdgeVec e2{&tmp};
            const int n_own = is_first ? rv.nF : rv.nS, n_mate = is_first ? rv.nS : rv.nF;
            if (mode == MODE_OTHER && n_own <= 1 && !getenv("SQ_EMUL_NO_FAST_EDGES")) {  // the register fast path of the stream kernel
                const Blk own = n_own ? (is_first ? rv.F[0] : rv.S[0]) : Blk{}, mate = n_mate ? (is_first ? rv.S[0] : rv.F[0]) : Blk{};
                const int32_t r0 = read_edges_single(nt, p, n_own > 0, own, n_mate > 0, mate, is_first, is_first ? rv.first_total : rv.second_total, e2);
                if (r0 != -3) { keys.insert(keys.end(), tmp.begin(), tmp.end()); res0[i] = r0; }
                else sens[i] = 1;
                continue;
            }
            if (read_edges(nt, p, rv, mode, is_first, false, 0, node, e2)) {
                keys.insert(keys.end(), tmp.begin(), tmp.end());
                res0[i] = node[0];
                store(i, rv);
            } else sens[i] = 1;
        }
        int32_t hint = 0;
        for (int64_t i = 0; i < count; i++) {
            if (sens[i]) {
                Blk F[kMaxBlocks + 1], S[kMaxBlocks + 1];
                ReadView rv; rv.F = F; rv.S = S;
                bool is_first;
                load(i, rv, is_first);
                int32_t node[2 * kMaxBlocks + 2];
                bool ok = read_edges(nt, p, rv, mode, is_first, true, hint, node, emit);
                if (!ok) { fprintf(stderr, "sensitive with known hint?!\n"); exit(4); }
                store(i, rv);
                res0[i] = node[0];
            }
            if (res0[i] >= 0) hint = res0[i];
        }
    };
    // chimeric
    run_stream(MODE_CHIM, cview.n_reads,
        [&](int64_t i, ReadView &rv, bool &is_first) {
            const uint32_t o = cview.read_off[i], e = cview.read_off[i + 1], nf = cview.n_first[i];
            rv.nF = 0; rv.nS = 0;
            for (uint32_t k = o; k < e; k++) {
                Blk x; x.ref_id = cview.blk_ref_id[k]; x.ref_pos = cview.blk_ref_pos[k]; x.match_ref = cview.blk_match_ref[k];
                x.read_pos = cview.blk_read_pos[k]; x.match_read = cview.blk_match_read[k]; x.rev = cview.blk_is_reverse[k];
                if (k - o < nf) rv.F[rv.nF++] = x; else rv.S[rv.nS++] = x;
            }
            rv.first_total = cview.first_total_len[i]; rv.second_total = cview.second_total_len[i];
            is_first = true;
        },
        [&](int64_t i, ReadView &rv) {
            uint32_t k = cview.read_off[i];
            for (int m = 0; m < 2; m++)
                for (int q = 0; q < (m ? rv.nS : rv.nF); q++, k++) {
                    const Blk &x = m ? rv.S[q] : rv.F[q];
                    cview.blk_ref_pos[k] = x.ref_pos; cview.blk_match_ref[k] = x.match_ref; cview.blk_read_pos[k] = x.read_pos; cview.blk_match_read[k] = x.match_read;
                }
        },
        [&](int64_t) { return true; });
    // concordant stream
    auto load_conc = [&](int64_t r, ReadView &rv, bool &is_first) {
        Blk *own = flag_first(b.flag[r]) ? rv.F : rv.S;
        Blk *oth = flag_first(b.flag[r]) ? rv.S : rv.F;
        const int no = load_sorted_blocks(b, r, own);
        int nm = 0;
        if (has_mate_block(b.flag[r], b.mate_ref_id[r])) {
            Blk x; x.ref_id = b.mate_ref_id[r]; x.ref_pos = b.mate_pos[r]; x.read_pos = 0; x.match_ref = kMateBlockLen; x.match_read = kMateBlockLen;
            x.rev = flag_mate_rev(b.flag[r]);
            oth[nm++] = x;
        }
        is_first = flag_first(b.flag[r]);
        if (is_first) { rv.nF = no; rv.nS = nm; rv.first_total = b.total_len[r]; rv.second_total = 0; }
        else { rv.nS = no; rv.nF = nm; rv.second_total = b.total_len[r]; rv.first_total = 0; }
    };
    run_stream(MODE_OTHER, n, load_conc, [&](int64_t, ReadView &) {},
        [&](int64_t r) {
            if (!(cls[r] & CLS_KEEP)) return false;
            // whetherbuildedge (:1601-1605)
            const uint32_t o = b.blk_off[r], nb = b.blk_off[r + 1] - o;
            const bool mate = has_mate_block(b.flag[r], b.mate_ref_id[r]);
            if (nb == 0 || !mate) return true;
            int32_t front_rp = 0x7fffffff;
            for (uint32_t k = 0; k < nb; k++) front_rp = std::min<int32_t>(front_rp, b.blk_read_pos[o + k]);
            return front_rp <= 15 || (int32_t)b.lowphred_run[r] > p.max_lowphred_len;
        });
    std::sort(keys.begin(), keys.end());
    {
        std::vector<int32_t> e;
        for (size_t i = 0; i < keys.size();) {
            size_t j = i;
            while (j < keys.size() && keys[j] == keys[i]) j++;
            int32_t a, c; bool h1, h2;
            edge_unpack(keys[i], a, h1, c, h2);
            e.push_back(a); e.push_back(c); e.push_back(h1); e.push_back(h2); e.push_back((int32_t)(j - i));
            i = j;
        }
        dump_i32("edges_i32.bin", e);
    }
    {
        std::vector<int32_t> a;
        for (int64_t i = 0; i < cview.n_reads; i++)
            for (uint32_t k = cview.read_off[i]; k < cview.read_off[i + 1]; k++) {
                a.push_back((int32_t)i); a.push_back(k - cview.read_off[i] >= cview.n_first[i]); a.push_back(cview.blk_ref_id[k]); a.push_back(cview.blk_ref_pos[k]);
                a.push_back(cview.blk_read_pos[k]); a.push_back(cview.blk_match_ref[k]); a.push_back(cview.blk_match_read[k]); a.push_back(cview.blk_is_reverse[k]);
            }
        dump_i32("chim_after_edges.bin", a);
    }
    // ---- breakpoint coverage on a supplied sorted BP list ----
    if (argc > 4) {
        std::vector<int32_t> bp;
        FILE *f = fopen(argv[4], "rb");
        if (!f) { fprintf(stderr, "cannot open %s\n", argv[4]); return 2; }
        int32_t x;
        while (fread(&x, 4, 1, f) == 1) bp.push_back(x);
        fclose(f);
        const int64_t K = (int64_t)bp.size() / 2;
        std::vector<uint64_t> bpkey(K);
        for (int64_t k = 0; k < K; k++) bpkey[k] = chrpos_key(bp[2 * k], bp[2 * k + 1]);
        // prefix max of qualifying keys, r0 per BP, chain, count
        std::vector<uint64_t> M(n);
        uint64_t run = 0;
        std::vector<char> q(n);
        std::vector<uint64_t> key(n);
        for (int64_t r = 0; r < n; r++) {
            q[r] = cover_qualifies(cls[r], b.flag[r], b.ref_id[r], b.pos[r], b.mate_ref_id[r], b.mate_pos[r]);
            key[r] = q[r] ? chrpos_key(b.ref_id[r], cover_start(b.flag[r], b.ref_id[r], b.pos[r], b.mate_ref_id[r], b.mate_pos[r])) : 0;
            if (key[r] > run) run = key[r];
            M[r] = run;
        }
        std::vector<int64_t> t(K);
        int64_t tp = -1;
        for (int64_t k = 0; k < K; k++) {
            const uint64_t T = cover_pass_key(bp[2 * k], bp[2 * k + 1], p.concord_dist_pos);
            int64_t r0 = upper_bound_u64(M.data(), 0, n, T);
            int64_t c = r0 > tp ? r0 : tp + 1;
            while (c < n && !(q[c] && key[c] > T)) c++;
            t[k] = c; tp = c < n ? c : n;
        }
        std::vector<int32_t> cov(K, 0);
        for (int64_t r = 0; r < n; r++) {
            if (!q[r]) continue;
            const uint64_t ks = key[r], ke = chrpos_key(b.ref_id[r], b.end_pos[r]);
            for (int64_t k = lower_bound_u64(bpkey.data(), 0, K, ks); k < K && bpkey[k] < ke; k++)
                if (r < t[k]) cov[k]++;
        }
        dump_i32("cov_i32.bin", cov);
    }
    return 0;
}
