// TEST INFRASTRUCTURE — CPU restatement ("port") of the reference's segment-graph construction path.
//
// This file is the oracle of SURVEY.md §8c option (B): a plain, single-threaded, record-by-record
// restatement of what the reference does, written from the cited lines of /root/reference/src (nothing is
// copied).  It deliberately keeps the reference's STREAMING structure (one pass per BAM read-through,
// explicit cluster vectors, heap, linear LocateRead scans) and therefore shares no algorithmic shortcut with
// the CUDA path (which is event-driven over scans and binary searches).  Only tests/, __graft_entry__.smoke()
// and bench.py's cpu_baseline leg may load it; the product never does.
//
// PINNING.  The restatement is pinned against the reference itself: oracle/_ref/squid_ref is the reference's own
// sources compiled against shims, and tests/test_cpu_oracle.py requires this file to reproduce its dumps bit for
// bit on the committed golden cases (tests/golden/) and on fresh fuzzed cases whenever oracle/_ref is present.
// The reference ships no golden vectors or tests of its own (SURVEY.md §4).
//
// Entry point: sqo_run() reads two SQMB files (include/sqmb_format.h) and writes the same dump files as
// oracle/ref_harness.cpp (nodes_i32.bin, nodes_f64.bin, edges_i32.bin, chim_loaded.bin, chim_after_edges.bin,
// readlen.bin) plus cov_i32.bin for a supplied sorted breakpoint list.  sqo_edges_on_nodes() runs the same BuildEdges on
// a segment table the caller supplies.
#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/sqmb_format.h"

namespace {

struct Opt {  // src/Config.cpp:18-28
    bool phred33 = true;
    int max_lowphred = 10, min_phred = 4, min_mapq = 255, dist_pos = 50000, dist_idx = 20, read_len = 0;
};

struct Blk {  // SingleBamRec_t, src/SingleBamRec.h:25-61
    int chr, pos, rpos, mref, mread;
    int mapq;
    bool rev, first;
};
static bool blk_lt(const Blk &a, const Blk &b) { return a.chr != b.chr ? a.chr < b.chr : a.pos < b.pos; }   // operator<
static bool blk_gt(const Blk &a, const Blk &b) { return a.chr != b.chr ? a.chr > b.chr : a.pos > b.pos; }   // operator>
static bool blk_same(const Blk &a, const Blk &b) {                                                           // Same()
    return a.chr == b.chr && a.pos == b.pos && a.rpos == b.rpos && a.mread == b.mread && a.mref == b.mref && a.rev == b.rev && a.first == b.first;
}

struct Rd {  // ReadRec_t, src/ReadRec.h:35-58
    std::string name;
    std::vector<Blk> F, S;
    int ft = 0, st = 0;
    bool fl = false, sl = false, mf = false;
};

struct Aln {  // the BamAlignment members the path reads
    int chr, pos, mchr, mpos, flag, mapq;
    bool xa, has_ih;
    int ih;
    std::string name, seq, qual;
    std::vector<std::pair<char, int>> cig;
    bool mapped() const { return !(flag & 4); }
    bool mate_mapped() const { return !(flag & 8); }
    bool rev() const { return flag & 16; }
    bool mate_rev() const { return flag & 32; }
    bool first() const { return flag & 64; }
    bool second() const { return flag & 128; }
    bool dup() const { return flag & 1024; }
    bool proper() const { return flag & 2; }
    int end() const {  // BamTools GetEndPosition(): pos + M,D,N,=,X
        int e = pos;
        for (auto &c : cig) if (c.first == 'M' || c.first == 'D' || c.first == 'N' || c.first == '=' || c.first == 'X') e += c.second;
        return e;
    }
};

static Aln fetch(const SqmbView &v, uint64_t r) {  // what the BamReader shim hands to the reference, restated
    static const char OPS[] = "MIDNSHP=X";
    Aln a;
    a.chr = v.ref_id[r]; a.pos = v.pos[r]; a.mchr = v.mate_ref_id[r]; a.mpos = v.mate_pos[r]; a.flag = v.flag[r]; a.mapq = v.mapq[r];
    a.xa = v.aux[r] & 1; a.has_ih = v.aux[r] & 2; a.ih = v.ih[r];
    a.name = "q" + std::to_string(v.name_id[r]);
    if (v.aux[r] & 4) a.name += (a.flag & 128) ? "/2" : "/1";
    int lseq = 0;
    for (uint32_t c = v.cigar_off[r]; c < v.cigar_off[r + 1]; c++) {
        const int op = v.cigar[c] & 15, len = v.cigar[c] >> 4;
        a.cig.push_back({OPS[op], len});
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) lseq += len;
    }
    if (v.seq_off[r] >= 0) {
        const uint8_t *b = v.blob + v.seq_off[r];
        uint32_t l;
        memcpy(&l, b, 4);
        a.seq.assign((const char *)b + 4, l); a.qual.assign((const char *)b + 4 + l, l);
    } else {
        a.seq.assign(lseq, 'C'); a.qual.assign(lseq, 'I');
        for (int i = 0; i < lseq && i < (int)v.lowrun[r]; i++) a.qual[i] = '#';
        if (v.polya[r]) {
            int rp = 0, k = 0;
            for (size_t c = 0; c < a.cig.size(); c++) {
                const char t = a.cig[c].first;
                if (t == 'S') rp += a.cig[c].second;
                else if (t == 'M' || t == '=') {
                    int span = 0;
                    size_t d = c;
                    for (; d < a.cig.size() && a.cig[d].first != 'S' && a.cig[d].first != 'H' && a.cig[d].first != 'N'; d++)
                        if (a.cig[d].first != 'D') span += a.cig[d].second;
                    if (k < 4 && (v.polya[r] >> k & 1)) for (int i = rp; i < rp + span && i < lseq; i++) a.seq[i] = 'A';
                    if (k < 4 && (v.polya[r] >> (4 + k) & 1)) for (int i = rp; i < rp + span && i < lseq; i++) a.seq[i] = 'T';
                    rp += span; k++; c = d - 1;
                }
            }
        }
    }
    return a;
}

// ReadRec_t::ReadRec_t(BamAlignment), src/ReadRec.cpp:10-88
static Rd decode(const Aln &a, const Opt &o) {
    Rd r;
    r.name = a.name;
    if (r.name.size() >= 2 && (r.name.substr(r.name.size() - 2) == "/1" || r.name.substr(r.name.size() - 2) == "/2")) r.name.resize(r.name.size() - 2);  // :12-13
    int total = 0;
    for (auto &c : a.cig) if (strchr("MSHI=X", c.first)) total += c.second;  // :16-18
    int best = 0, run = 0;
    const char thr = (char)((o.phred33 ? 33 : 64) + o.min_phred);  // :19-38
    for (char q : a.qual) { run = q < thr ? run + 1 : 0; best = std::max(best, run); }
    const bool low = best > o.max_lowphred;
    if (a.first()) { r.ft = total; r.st = 0; r.fl = low; } else { r.st = total; r.ft = 0; r.sl = low; }  // :39-44
    int rp = 0, gp = a.pos, hard = 0;
    for (size_t i = 0; i < a.cig.size(); i++) {  // :46-87
        const char t = a.cig[i].first;
        if (t == 'S' || t == 'H') { rp += a.cig[i].second; if (t == 'H') hard += a.cig[i].second; }
        else if (t == 'M' || t == '=') {
            int sr = 0, sg = 0;
            size_t j = i;
            for (; j < a.cig.size() && a.cig[j].first != 'S' && a.cig[j].first != 'H' && a.cig[j].first != 'N'; j++) {
                if (a.cig[j].first != 'D') sr += a.cig[j].second;
                if (a.cig[j].first != 'I') sg += a.cig[j].second;
            }
            int na = 0, nt = 0;
            for (int k = rp - hard; k < rp + sr - hard; k++) {
                if (k < 0 || k >= (int)a.seq.size()) continue;
                if (a.seq[k] == 'a' || a.seq[k] == 'A') na++; else if (a.seq[k] == 't' || a.seq[k] == 'T') nt++;
            }
            if (1.0 * na / sr < 0.75 && 1.0 * nt / sr < 0.75) {  // :72
                Blk b{a.chr, gp, a.rev() ? total - rp - sr : rp, sg, sr, a.mapq, a.rev(), a.first()};
                (a.first() ? r.F : r.S).push_back(b);
            }
            rp += sr; gp += sg; i = j - 1;
        } else if (t == 'N') gp += a.cig[i].second;
    }
    return r;
}

static void sort_rpos(Rd &r) {  // SortbyReadPos, :143-146
    auto c = [](const Blk &x, const Blk &y) { return x.rpos < y.rpos; };
    std::sort(r.F.begin(), r.F.end(), c); std::sort(r.S.begin(), r.S.end(), c);
}
static bool end_disc(const std::vector<Blk> &v) {  // IsEndDiscordant, :178-209
    for (size_t i = 0; i + 1 < v.size(); i++) {
        if (v[i].chr != v[i + 1].chr || v[i].rev != v[i + 1].rev) return true;
        if (!v[i].rev && (v[i].pos < v[i + 1].pos) != (v[i].rpos < v[i + 1].rpos)) return true;
        if (v[i].rev && (v[i].pos < v[i + 1].pos) == (v[i].rpos < v[i + 1].rpos)) return true;
    }
    return false;
}
static bool single_anch(const Rd &r) { return (r.F.empty() || r.S.empty()) && !r.mf; }  // :171-176
static bool pair_disc(const Rd &r, bool check) {  // IsPairDiscordant, :211-228
    if (r.F.empty() || r.S.empty()) return false;
    if (check && (end_disc(r.F) || end_disc(r.S))) return true;
    if (r.F.front().chr != r.S.back().chr || r.F.front().rev == r.S.back().rev) return true;
    if (!r.F.front().rev && r.F.front().pos - r.F.front().rpos > r.S.back().pos - (r.st - r.S.back().rpos - r.S.back().mread)) return true;
    if (!r.S.front().rev && r.S.front().pos - r.S.front().rpos > r.F.back().pos - (r.ft - r.F.back().rpos - r.F.back().mread)) return true;
    return false;
}
static bool lists_eq(const std::vector<Blk> &x, const std::vector<Blk> &y) {
    if (x.size() != y.size()) return false;
    for (size_t i = 0; i < x.size(); i++) if (x[i].chr != y[i].chr || x[i].pos != y[i].pos || x[i].mref != y[i].mref) return false;
    return true;
}
static bool rd_equal(const Rd &a, const Rd &b) {  // Equal, :119-141
    return (lists_eq(a.F, b.F) && lists_eq(a.S, b.S)) || (lists_eq(a.F, b.S) && lists_eq(a.S, b.F));
}
static bool front_lt(const Rd &a, const Rd &b) {  // FrontSmallerThan, :90-117
    const Blk *x, *y;
    if (!a.F.empty() && !b.F.empty()) { x = &a.F[0]; y = &b.F[0]; }
    else if (!a.S.empty() && !b.S.empty()) { x = &a.S[0]; y = &b.S[0]; }
    else if (!a.F.empty() && !b.S.empty()) { x = &a.F[0]; y = &b.S[0]; }
    else if (!a.S.empty() && !b.F.empty()) { x = &a.S[0]; y = &b.F[0]; }
    else return false;
    return x->chr != y->chr ? x->chr < y->chr : x->pos < y->pos;
}

// BuildChimericSBamRecord, src/ReadRec.cpp:329-413
static std::vector<Rd> load_chim(const SqmbView &v, Opt &o) {
    std::vector<Rd> all;
    std::vector<int> sample;
    for (uint64_t r = 0; r < v.n_rec; r++) {
        Aln a = fetch(v, r);
        if (!a.mapped() || a.dup()) continue;
        Rd d = decode(a, o);
        if (sample.size() < 5) sample.push_back(std::max(d.ft, d.st));
        all.push_back(d);
    }
    std::sort(all.begin(), all.end(), [](const Rd &x, const Rd &y) { return x.name < y.name; });
    std::vector<Rd> m;
    for (Rd &d : all) {
        if (m.empty() || d.name != m.back().name) { m.push_back(d); continue; }
        Rd &t = m.back();
        if (t.ft == 0 && d.ft != 0) { t.ft = d.ft; t.fl = d.fl; }
        if (t.st == 0 && d.st != 0) { t.st = d.st; t.sl = d.sl; }
        t.F.insert(t.F.end(), d.F.begin(), d.F.end()); t.S.insert(t.S.end(), d.S.begin(), d.S.end());
    }
    for (Rd &d : m) sort_rpos(d);
    if (!sample.empty()) { std::sort(sample.begin(), sample.end()); o.read_len = sample[sample.size() / 2]; }
    std::sort(m.begin(), m.end(), front_lt);
    std::vector<Rd> out;
    for (Rd &d : m) {
        if (out.empty() || d.F.empty() || out.back().F.empty() || d.F[0].chr != out.back().F[0].chr || d.F[0].pos != out.back().F[0].pos) { out.push_back(d); continue; }
        bool dup = false;
        for (size_t k = out.size(); k-- > 0;) {
            if (out[k].F.empty() || d.F[0].chr != out[k].F[0].chr || d.F[0].pos != out[k].F[0].pos) break;
            if (rd_equal(d, out[k])) { dup = true; break; }
        }
        if (!dup) out.push_back(d);
    }
    return out;
}

struct Node { int chr, pos, len, support; double depth; };
struct Edge { int a, b; bool ha, hb; int w; };
static Edge mk_edge(int i, bool hi, int j, bool hj, int w = 1) {  // Edge_t ctor, src/BPEdge.h:31-52
    if (i > j) return Edge{j, i, hj, hi, w};
    return Edge{i, j, hi, hj, w};
}
static bool edge_lt(const Edge &x, const Edge &y) {  // BPEdge.h:59-70
    if (x.a != y.a) return x.a < y.a;
    if (x.b != y.b) return x.b < y.b;
    if (x.ha != y.ha) return (int)x.ha < (int)y.ha;
    if (x.hb != y.hb) return (int)x.hb < (int)y.hb;
    return false;
}

struct Graph {
    Opt o;
    std::vector<int> ref_len;
    std::vector<Node> nodes;
    std::vector<Edge> edges;

    bool gate(const Aln &a, const std::vector<std::string> &chim_names, bool need_chr) const {  // SegmentGraph.cpp:302 / 1584 / 3136
        int ihv = a.has_ih ? a.ih : 0;
        if (a.xa || ihv > 1 || a.mapq < o.min_mapq || a.dup() || !a.mapped()) return false;
        if (need_chr && a.chr == -1) return false;
        return !std::binary_search(chim_names.begin(), chim_names.end(), a.name);
    }
    static std::vector<std::string> names_of(const std::vector<Rd> &chim) {  // :196-201 (pre-sized vector => one "" entry)
        std::vector<std::string> n(chim.size());
        for (auto &r : chim) n.push_back(r.name);
        std::sort(n.begin(), n.end());
        n.erase(std::unique(n.begin(), n.end()), n.end());
        return n;
    }
    static void add_mate_block(const Aln &a, Rd &r) {  // :307-314
        if (!(a.mate_mapped() && a.mchr != -1)) return;
        Blk m{a.mchr, a.mpos, 0, 15, 15, 60, a.mate_rev(), false};
        (a.first() ? r.S : r.F).push_back(m);
    }
    // The per-record preamble of BuildNode_STAR for one concordant record (:297-333 gate, Equal against the previous
    // gate-passing record `last`, own blocks; :649-689 concordance and partial alignment).  Shared by build_nodes and sqo_classify.
    struct RecClass {
        Aln a;
        Rd rd, tmp;  // rd: the record's own blocks in CIGAR order; tmp: sorted by read position, with the mate block (:305-314)
        bool gate = false, keep = false, conc = false, part_f = false, part_s = false;
        const std::vector<Blk> &own() const { return (a.first() && !rd.F.empty()) ? rd.F : rd.S; }  // :320-333
        bool has_blk() const { return (a.first() && !rd.F.empty()) || !rd.S.empty(); }
        const std::vector<Blk> *other_own() const { return a.first() ? &rd.F : (a.second() ? &rd.S : nullptr); }  // :657-663
    };
    void classify(const SqmbView &conc, uint64_t ri, const std::vector<std::string> &names, Rd &last, RecClass &c) const {
        c = RecClass();
        c.a = fetch(conc, ri);
        const Aln &a = c.a;
        c.gate = gate(a, names, true);
        if (!c.gate) return;
        c.rd = decode(a, o);
        c.tmp = c.rd;
        sort_rpos(c.tmp);
        add_mate_block(a, c.tmp);
        if (rd_equal(last, c.tmp)) return;
        last = c.tmp;
        c.keep = true;
        bool concordant = false;  // :651-654
        if (a.mapped() && a.mate_mapped() && a.mchr != -1 && a.chr == a.mchr && a.proper()) {
            if (a.rev() && !a.mate_rev() && a.pos >= a.mpos && a.pos - a.mpos <= 750000) concordant = true;
            else if (!a.rev() && a.mate_rev() && a.mpos >= a.pos && a.mpos - a.pos <= 750000) concordant = true;
        }
        c.conc = concordant && c.rd.F.size() + c.rd.S.size() > 0;
        if (!c.conc) return;
        const Rd &t = c.tmp;  // :668-683
        c.part_f = a.first() && !t.fl && (t.F.front().rpos > 15 || t.ft - t.F.back().rpos - t.F.back().mread > 15);
        c.part_s = a.second() && !t.sl && (t.S.front().rpos > 15 || t.st - t.S.back().rpos - t.S.back().mread > 15);
    }

    bool edge_disc(const Edge &e) const {  // IsDiscordant(Edge_t), :181-190
        if (nodes[e.a].chr != nodes[e.b].chr) return true;
        if (nodes[e.b].pos - nodes[e.a].pos - nodes[e.a].len > o.dist_pos && e.b - e.a > o.dist_idx) return true;
        return e.ha != false || e.hb != true;
    }

    // ---- BuildNode_STAR, SegmentGraph.cpp:192-831 ---------------------------------------------------------------
    void build_nodes(const SqmbView &conc, const std::vector<Rd> &chim) {
        const int RL = o.read_len, thresh = 3;
        const std::vector<std::string> names = names_of(chim);
        std::vector<std::pair<int, int>> part(ref_len.size());  // :203-204
        std::vector<Blk> dis;
        for (const Rd &r : chim) {  // :207-261
            if (end_disc(r.F) || end_disc(r.S) || single_anch(r) || pair_disc(r, true)) {
                for (auto &b : r.F) dis.push_back(b);
                for (auto &b : r.S) dis.push_back(b);
                continue;
            }
            bool fin = false, sin = false;
            for (int m = 0; m < 2; m++) {
                const std::vector<Blk> &v = m ? r.S : r.F;
                int prev = -1;
                for (int i = 0; i + 1 < (int)v.size(); i++)
                    if (std::abs(v[i].pos - v[i + 1].pos) > 750000) {
                        if (prev != i) dis.push_back(v[i]);
                        dis.push_back(v[i + 1]);
                        prev = i + 1;
                        if (i + 1 == (int)v.size() - 1) (m ? sin : fin) = true;
                    }
            }
            if (!r.F.empty() && !r.S.empty() && std::abs(r.F.back().pos - r.S.back().pos) > 750000) {
                if (!fin) { dis.push_back(r.F.back()); fin = true; }
                if (!sin) { dis.push_back(r.S.back()); sin = true; }
            }
            if (!fin && !sin) {
                if (!r.F.empty() && r.F[0].rpos > 15 && !r.fl) part.push_back({r.F[0].chr, r.F[0].rev ? r.F[0].pos + r.F[0].mref : r.F[0].pos});
                if (!r.F.empty() && r.ft - r.F.back().rpos - r.F.back().mread > 15 && !r.fl) part.push_back({r.F.back().chr, r.F.back().rev ? r.F.back().pos : r.F.back().pos + r.F.back().mref});
                if (!r.S.empty() && r.S[0].rpos > 15 && !r.sl) part.push_back({r.S[0].chr, r.S[0].rev ? r.S[0].pos + r.S[0].mref : r.S[0].pos});
                if (!r.S.empty() && r.st - r.S.back().rpos - r.S.back().mread > 15 && !(dis.empty() ? false : blk_same(dis.back(), r.S.back())) && !r.sl)
                    part.push_back({r.S.back().chr, r.S.back().rev ? r.S.back().pos : r.S.back().pos + r.S.back().mref});
            }
        }
        std::sort(part.begin(), part.end(), [](std::pair<int, int> a, std::pair<int, int> b) { return a.first == b.first ? a.second < b.second : a.first < b.first; });
        std::sort(dis.begin(), dis.end(), blk_lt);  // :264 (same unstable sort on the same sequence)
        const size_t nD = dis.size();
        dis.push_back(Blk{0, 0, 0, 0, 0, 0, false, false});  // what *cend() reads under the harness's zeroing allocator
        size_t ds = 0, de = 0, ps = 0, pe = 0;
        std::vector<std::pair<int, std::pair<int, int>>> main_, other_;
        std::vector<Blk> rest, cc, pc;  // ConcordRest (heap), ConcordantCluster, PartialAlignCluster
        auto heap_cmp = [](const Blk &l, const Blk &r) { return !blk_lt(l, r); };  // MinHeapComp, :15-17
        size_t occ = 0, opc = 0;
        int disChr = 0, otherChr = 0, nextChr = 0, disRight = 0, otherRight = 0, nextRight = 0, markStart = -1, markChr = -1;
        Rd last;
        auto regroup = [&]() {  // :341-348 / :604-611
            disRight = nextRight; disChr = nextChr;
            nextRight = dis[ds].pos + dis[ds].mref;
            for (de = ds; de != nD && dis[de].chr == dis[ds].chr && dis[de].pos < nextRight + RL; de++) {
                nextRight = std::max(nextRight, dis[de].pos + dis[de].mref);
                nextChr = dis[de].chr;
            }
        };
        RecClass rc;
        for (uint64_t ri = 0; ri < conc.n_rec; ri++) {
            classify(conc, ri, names, last, rc);
            if (!rc.keep) continue;
            const Aln &a = rc.a;
            const Rd &rd = rc.rd;
            const std::vector<Blk> &own = rc.own();
            if (rc.has_blk()) {
                main_.push_back({own[0].chr, {own[0].pos, own[0].mref}});
                for (size_t k = 1; k < own.size(); k++) other_.push_back({own[k].chr, {own[k].pos, own[k].mref}});
            }
            if (ds == nD) break;  // :338
            if (de <= ds) regroup();
            while (ds != nD && (dis[ds].chr < a.chr || (dis[ds].chr == a.chr && nextRight < a.pos))) {  // :353
                int curEnd = 0, curStart = 0, disS = -1, disE = -1, disCnt = -1;
                bool split = false;
                if (markStart != -1 && dis[ds].chr != markChr) { markChr = -1; markStart = -1; }
                while (cc.size() != occ && cc[occ].chr < dis[ds].chr) occ++;
                while (pc.size() != opc && pc[opc].chr < dis[ds].chr) opc++;
                if (cc.size() != occ && dis[ds].pos > cc.back().pos + cc.back().mref + RL) occ = cc.size();
                if (pc.size() != opc && dis[ds].pos > pc.back().pos + pc.back().mref + RL) opc = pc.size();
                curStart = dis[ds].pos;
                Blk t{};
                if (cc.size() != occ && pc.size() != opc) t = blk_lt(cc[occ], pc[opc]) ? cc[occ] : pc[opc];
                else if (cc.size() != occ) t = cc[occ];
                else if (pc.size() != opc) t = pc[opc];
                if ((cc.size() != occ || pc.size() != opc) && (t.chr < dis[ds].chr || (t.chr == dis[ds].chr && t.pos < dis[ds].pos))) curStart = t.pos;
                curStart = std::max(curStart, markStart);
                while (!rest.empty() && (rest.front().chr < dis[ds].chr || (rest.front().chr == dis[ds].chr && rest.front().pos < dis[ds].pos - RL))) {
                    std::pop_heap(rest.begin(), rest.end(), heap_cmp); rest.pop_back();
                }
                for (; ps != part.size() && (part[ps].first < dis[ds].chr || (part[ps].first == dis[ds].chr && part[ps].second + RL < dis[ds].pos)); ps++) {}
                for (pe = ps; pe != part.size() && part[pe].first == dis[ds].chr && part[pe].second < nextRight + RL; pe++) {}
                while (ds != de) {  // :395
                    if (ds != 0 && dis[ds].chr != dis[ds - 1].chr && cc.size() == occ && pc.size() == opc) curStart = dis[ds].pos;
                    split = false;
                    std::vector<int> mp;
                    size_t dc;
                    for (dc = ds; dc != de; dc++) {
                        mp.push_back(dis[dc].pos); mp.push_back(dis[dc].pos + dis[dc].mref);
                        curEnd = std::max(curEnd, mp.back());
                        if (dc + 1 != de && dis[dc + 1].pos > dis[dc].pos + dis[dc].mref) break;
                    }
                    disS = std::max(curStart, dis[ds].pos); disE = curEnd; disCnt = (int)(dc - ds);
                    if (dc != de) for (dc++; dc != de && dis[dc].pos < curEnd + thresh; dc++) { mp.push_back(dis[dc].pos); mp.push_back(dis[dc].pos + dis[dc].mref); }
                    for (size_t q = ps; q != pe && part[q].second < curEnd + thresh; q++) mp.push_back(part[q].second);
                    for (size_t i = opc; i != pc.size(); i++) {  // :420-434
                        const Blk &b = pc[i];
                        if (b.chr == dis[ds].chr && b.rpos > 15 && b.pos > mp.front() - thresh && b.pos < curEnd + thresh) {
                            if (b.rev && b.pos + b.mref > mp.front() - thresh && b.pos + b.mref < curEnd + thresh) mp.push_back(b.pos + b.mref);
                            else if (!b.rev && b.pos > mp.front() - thresh && b.pos < curEnd + thresh) mp.push_back(b.pos);
                        } else if (b.chr == dis[ds].chr) {
                            if (b.rev && b.pos > mp.front() - thresh && b.pos < curEnd + thresh) mp.push_back(b.pos);
                            else if (!b.rev && b.pos + b.mref > mp.front() - thresh && b.pos + b.mref < curEnd + thresh) mp.push_back(b.pos + b.mref);
                        }
                    }
                    std::sort(mp.begin(), mp.end());
                    int lastCur = -1, lastSup = 0;
                    for (size_t ib = 0; ib < mp.size(); ib++) {  // :440-504
                        const int brk = mp[ib];
                        if (!nodes.empty() && nodes.back().chr == dis[ds].chr && brk - nodes.back().pos - nodes.back().len < thresh * 20) continue;
                        int sr = 0, pl = 0, pr = 0;
                        for (size_t k = 0; k < mp.size() && mp[k] < brk + thresh; k++) if (std::abs(brk - mp[k]) < thresh) sr++;
                        for (size_t k = ds; k != de; k++) {
                            if (dis[k].pos + dis[k].mref < brk && dis[k].pos + dis[k].mref > brk - RL && !dis[k].rev) pl++;
                            else if (dis[k].pos > brk && dis[k].pos < brk + RL && dis[k].rev) pr++;
                        }
                        if (sr > 3 || sr + pl > 4 || sr + pr > 4) {
                            int cov = 0;
                            auto spans = [&](const Blk &b) { return b.chr == dis[ds].chr && b.pos + b.mref >= brk + thresh && b.pos < brk - thresh; };
                            for (size_t i = occ; i < cc.size(); i++) cov += spans(cc[i]);
                            for (size_t k = ds; k != de; k++) cov += spans(dis[k]);
                            for (size_t i = opc; i != pc.size(); i++) cov += spans(pc[i]);
                            if (sr > std::max(cov - sr, 0) + 2) for (const Blk &b : rest) cov += spans(b);
                            if (sr > std::max(cov - sr, 0) + 2) {
                                if (lastCur == -1 && brk - curStart < thresh * 20) { markStart = curStart; markChr = dis[ds].chr; }
                                else if ((lastCur == -1 || brk - lastCur < thresh * 20) && std::max(sr + pl, sr + pr) > lastSup) { lastCur = brk; lastSup = std::max(sr + pl, sr + pr); }
                                else if (brk - lastCur >= thresh * 20) {
                                    split = true;
                                    if (dis[ds].pos - curStart > thresh * 20 && lastCur - dis[ds].pos > thresh * 20) { nodes.push_back(Node{dis[ds].chr, curStart, dis[ds].pos - curStart, 0, 0}); curStart = dis[ds].pos; }
                                    nodes.push_back(Node{dis[ds].chr, curStart, lastCur - curStart, 0, 0});
                                    curStart = lastCur; curEnd = lastCur; markStart = lastCur; markChr = dis[ds].chr; lastCur = brk;
                                }
                            }
                        }
                        size_t nx = ib;
                        while (nx < mp.size() && mp[nx] == brk) nx++;
                        if (nx < mp.size()) ib = nx - 1; else break;
                    }
                    if (lastCur != -1 && (!split || nodes.back().pos + nodes.back().len != lastCur)) {  // :505-516
                        split = true;
                        if (dis[ds].pos - curStart > thresh * 20 && lastCur - dis[ds].pos > thresh * 20) { nodes.push_back(Node{dis[ds].chr, curStart, dis[ds].pos - curStart, 0, 0}); curStart = dis[ds].pos; }
                        nodes.push_back(Node{dis[ds].chr, curStart, lastCur - curStart, 0, 0});
                        curStart = lastCur; curEnd = lastCur; markStart = lastCur; markChr = dis[ds].chr;
                    }
                    if (disS != -1 && !split && disCnt > std::min(5.0, 4.0 * (disE - disS) / RL)) {  // :518-527
                        if (!nodes.empty() && nodes.back().chr == dis[de - 1].chr && disE - nodes.back().pos - nodes.back().len < thresh * 20) nodes.back().len += disE - nodes.back().pos - nodes.back().len;
                        else nodes.push_back(Node{dis[de - 1].chr, disS, disE - disS, 0, 0});
                        curStart = disE; curEnd = disE; markStart = disE; markChr = dis[ds].chr;
                    }
                    while (cc.size() != occ && cc[occ].chr < dis[ds].chr) occ++;
                    while (pc.size() != opc && pc[opc].chr < dis[ds].chr) opc++;
                    for (dc = ds; dc != de && dis[dc].pos + dis[dc].mref <= curEnd; dc++) {}
                    int c0 = curStart;
                    do {  // :537-567
                        bool f1 = false, f2 = false;
                        for (int w = 0; w < 2; w++) {
                            std::vector<Blk> &v = w ? pc : cc;
                            size_t &off = w ? opc : occ;
                            if (v.size() == off) continue;
                            bool f = true;
                            const Blk &b = v[off];
                            if (b.chr > dis[ds].chr) f = false;
                            if (dc != nD && b.chr == dis[dc].chr && b.pos + b.mref + RL >= dis[dc].pos) f = false;
                            if (!nodes.empty() && (b.chr > nodes.back().chr || (b.chr == nodes.back().chr && b.pos >= nodes.back().pos + nodes.back().len))) f = false;
                            if (f) { c0 = std::max(c0, b.pos + b.mref); off++; }
                            (w ? f2 : f1) = f;
                        }
                        if (!f1 && !f2) break;
                    } while (cc.size() != occ || pc.size() != opc);
                    do {  // :570-601
                        if (markStart != -1 && (a.chr > markChr || a.pos > c0 + RL) && (cc.size() == occ || cc[occ].chr != markChr || cc[occ].pos > c0 + RL) &&
                            (pc.size() == opc || pc[opc].chr != markChr || pc[opc].pos > c0)) {
                            if (c0 > markStart && c0 < markStart + thresh * 20 && !nodes.empty() && nodes.back().chr == markChr) nodes.back().len += c0 - nodes.back().pos - nodes.back().len;
                            else if (c0 > markStart) nodes.push_back(Node{markChr, markStart, c0 - markStart, 0, 0});
                            curStart = c0; markChr = -1; markStart = -1;
                            break;
                        }
                        bool f1 = false, f2 = false;
                        for (int w = 0; w < 2; w++) {
                            std::vector<Blk> &v = w ? pc : cc;
                            size_t &off = w ? opc : occ;
                            if (v.size() == off) continue;
                            const Blk &b = v[off];
                            const bool f = dc == nD || b.chr < dis[dc].chr || (b.chr == dis[dc].chr && b.pos + b.mref + RL < dis[dc].pos);
                            if (f) { c0 = std::max(c0, b.pos + b.mref); off++; }
                            (w ? f2 : f1) = f;
                        }
                        if (!f1 && !f2) break;
                    } while (cc.size() != occ || pc.size() != opc);
                    ds = dc;
                }
                if (de <= ds) regroup();  // :604-611 (reads the zeroed sentinel once ds == nD)
            }
            // :616-646
            int curRight = (disChr > otherChr || (disChr == otherChr && disRight > otherRight)) ? disRight : otherRight;
            int curChr = disChr > otherChr ? disChr : otherChr;
            const bool zero = (a.chr != curChr || a.pos > curRight + RL) && (curChr < dis[ds].chr || (curChr == dis[ds].chr && curRight + RL < dis[ds].pos));
            if (zero && markStart != -1) {
                if (curChr == markChr && curRight > markStart && curRight - markStart < thresh * 20 && !nodes.empty() && markStart == nodes.back().pos + nodes.back().len) nodes.back().len += curRight - markStart;
                else if (curChr == markChr && curRight > markStart && curRight - markStart >= thresh * 20) nodes.push_back(Node{markChr, markStart, curRight - markStart, 0, 0});
                markStart = -1; markChr = -1;
            }
            if (zero && (curChr != dis[ds].chr || curRight + RL < dis[ds].pos)) { occ = cc.size(); opc = pc.size(); }
            else {
                for (int w = 0; w < 2; w++) {
                    std::vector<Blk> &v = w ? pc : cc;
                    size_t &off = w ? opc : occ;
                    while (v.size() > off && v[off].chr != a.chr) off++;
                    while (v.size() > off && (v[off].chr < dis[ds].chr || (!nodes.empty() && v[off].chr == nodes.back().chr && v[off].pos < nodes.back().pos + nodes.back().len))) off++;
                }
            }
            // :649-700
            if (rc.conc) {
                const std::vector<Blk> *ownp = rc.other_own();
                if (ownp) {
                    const int e = ownp->front().pos + ownp->front().mref;
                    if (otherChr == a.chr) otherRight = std::max(otherRight, e); else { otherRight = e; otherChr = a.chr; }
                }
                if (rc.part_f) pc.push_back(rd.F.front());
                if (rc.part_s) pc.push_back(rd.S.front());
                if (!rc.part_f && !rc.part_s) cc.push_back(a.first() ? rd.F.front() : rd.S.front());
                if (ownp && ownp->size() > 1)
                    for (size_t i = 1; i < ownp->size(); i++)
                        if (ds != nD && (*ownp)[i].pos >= dis[ds].pos - RL) { rest.push_back((*ownp)[i]); std::push_heap(rest.begin(), rest.end(), heap_cmp); }
            }
        }
        // NormalizeSeedNodes :19-38 and genome tiling :714-761
        std::sort(nodes.begin(), nodes.end(), [](const Node &x, const Node &y) { return x.chr != y.chr ? x.chr < y.chr : (x.pos != y.pos ? x.pos < y.pos : x.len < y.len); });
        std::vector<Node> norm;
        for (const Node &n : nodes) {
            if (norm.empty() || norm.back().chr != n.chr || norm.back().pos + norm.back().len <= n.pos) norm.push_back(n);
            else norm.back().len = std::max(norm.back().pos + norm.back().len, n.pos + n.len) - norm.back().pos;
        }
        std::vector<Node> tiles;
        for (Node n : norm) {
            if (tiles.empty() || tiles.back().chr != n.chr) {
                if (!tiles.empty() && tiles.back().pos + tiles.back().len != ref_len[tiles.back().chr])
                    tiles.push_back(Node{tiles.back().chr, tiles.back().pos + tiles.back().len, ref_len[tiles.back().chr] - tiles.back().pos - tiles.back().len, 0, 0});
                for (int c = tiles.empty() ? 0 : tiles.back().chr + 1; c != n.chr; c++) tiles.push_back(Node{c, 0, ref_len[c], 0, 0});
                if (n.pos != 0) {
                    if (n.pos > 100) tiles.push_back(Node{n.chr, 0, n.pos, 0, 0});
                    else { n.len += n.pos; n.pos = 0; tiles.push_back(n); continue; }
                }
            }
            if (!tiles.empty() && tiles.back().chr == n.chr) {
                const int gap = n.pos - tiles.back().pos - tiles.back().len;
                if (gap > 100) tiles.push_back(Node{n.chr, n.pos - gap, gap, 0, 0});
                else if (gap > 0) { n.len += gap; n.pos -= gap; }
            }
            tiles.push_back(n);
        }
        if (!tiles.empty() && tiles.back().pos + tiles.back().len != ref_len[tiles.back().chr])
            tiles.push_back(Node{tiles.back().chr, tiles.back().pos + tiles.back().len, ref_len[tiles.back().chr] - tiles.back().pos - tiles.back().len, 0, 0});
        for (int c = tiles.back().chr + 1; c < (int)ref_len.size(); c++) tiles.push_back(Node{c, 0, ref_len[c], 0, 0});
        nodes = tiles;
        // per-node read counts, :766-826
        size_t it = 0;
        for (Node &n : nodes) {
            int cnt = 0, sum = 0;
            for (; it != nD && dis[it].chr == n.chr && dis[it].pos < n.pos + n.len; it++)
                if (dis[it].pos >= n.pos && dis[it].pos + dis[it].mref <= n.pos + n.len) { cnt++; sum += dis[it].mref; }
            n.support = cnt; n.depth = sum;
        }
        std::sort(other_.begin(), other_.end(), [](const std::pair<int, std::pair<int, int>> &x, const std::pair<int, std::pair<int, int>> &y) { return x.first != y.first ? x.first < y.first : x.second.first < y.second.first; });
        for (int pass = 0; pass < 2; pass++) {
            const auto &v = pass ? other_ : main_;
            if (v.empty()) continue;
            size_t q = 0;
            for (Node &n : nodes) {
                int cnt = 0, sum = 0;
                for (; q != v.size(); q++) {
                    if (v[q].first == n.chr && v[q].second.first >= n.pos - thresh && v[q].second.first + v[q].second.second <= n.pos + n.len + thresh) { cnt++; sum += v[q].second.second; }
                    else if (v[q].second.first >= n.pos + n.len || v[q].first != n.chr) break;
                }
                n.support += cnt; n.depth += sum;
                if (pass) n.depth = 1.0 * n.depth / n.len;
            }
        }
    }

    // ---- LocateRead(int, ReadRec_t&), SegmentGraph.cpp:1207-1293 -------------------------------------------------
    std::vector<int> locate(int guess, Rd &r) const {
        const int N = (int)nodes.size(), tol = 5;
        std::vector<int> out;
        int i = guess;
        for (int m = 0; m < 2; m++)
            for (Blk &b : (m ? r.S : r.F)) {
                if (i < 0 || i >= N) i = guess;
                auto fits = [&](int j) { return nodes[j].chr == b.chr && b.pos >= nodes[j].pos - tol && b.pos + b.mref <= nodes[j].pos + nodes[j].len + tol; };
                if (!fits(i)) {
                    if (nodes[i].chr < b.chr || (nodes[i].chr == b.chr && nodes[i].pos <= b.pos)) { for (; i < N && nodes[i].chr <= b.chr; i++) if (fits(i)) break; }
                    else { for (; i > -1 && nodes[i].chr >= b.chr; i--) if (fits(i)) break; }
                }
                if (i < 0 || i >= N || nodes[i].chr != b.chr) { out.push_back(-1); continue; }
                out.push_back(i);
                if (b.pos < nodes[i].pos) {  // :1229-1239
                    const int d = nodes[i].pos - b.pos;
                    if (!b.rev) b.rpos += d;
                    b.mref -= d; b.mread -= d; b.pos = nodes[i].pos;
                }
                if (b.pos + b.mref > nodes[i].pos + nodes[i].len) {  // :1240-1248
                    const int d = b.pos + b.mref - nodes[i].pos - nodes[i].len;
                    if (b.rev) b.rpos += d;
                    b.mref -= d; b.mread -= d;
                }
            }
        return out;
    }
    int spanning(int ffi, const Blk &b) const {  // :1408-1409 / :1614-1615
        const int N = (int)nodes.size();
        int i = ffi;
        for (; i < N && (nodes[i].chr < b.chr || (nodes[i].chr == b.chr && nodes[i].pos + nodes[i].len < b.pos)); i++) {}
        for (; i > -1 && (i >= N || nodes[i].chr > b.chr || (nodes[i].chr == b.chr && nodes[i].pos > b.pos)); i--) {}
        return i;
    }
    // shared body of RawEdgesChim (:1398-1527) and RawEdgesOther (:1606-1686) for one read
    void read_edges(Rd &r, int &ffi, bool chim_mode, bool rec_first) {
        std::vector<int> nd = locate(ffi, r);
        if (!nd.empty() && nd[0] != -1) ffi = nd[0];
        const int nf = (int)r.F.size(), ns = (int)r.S.size(), N = (int)nodes.size();
        for (int k = 0; k < nf + ns; k++)
            if (nd[k] == -1) {
                const int i = spanning(ffi, k < nf ? r.F[k] : r.S[k - nf]);
                if (i >= 0 && i + 1 < N) edges.push_back(mk_edge(i, false, i + 1, true));
            }
        for (int m = 0; m < 2; m++) {
            const std::vector<Blk> &v = m ? r.S : r.F;
            const int base = m ? nf : 0;
            for (int k = 0; k + 1 < (int)v.size(); k++) {
                const int i = nd[base + k], j = nd[base + k + 1];
                if (i != j && i != -1 && j != -1) edges.push_back(mk_edge(i, v[k].rev, j, !v[k + 1].rev));
            }
        }
        if ((chim_mode || rec_first) && nf > 0 && ns > 0 && !single_anch(r) && !end_disc(r.F) && !end_disc(r.S)) {
            const int i = nd[nf - 1], j = nd.back();
            bool ov = false;
            for (int k = 0; k < nf; k++) if (j == nd[k]) ov = true;
            for (int k = 0; k < ns; k++) if (i == nd[nf + k]) ov = true;
            if (nf > 1 && std::abs(i - j) < 3) ov = true;
            if (ns > 1 && std::abs(i - j) < 3) ov = true;
            if (i != j && i != -1 && j != -1 && !ov) {
                const Edge e = mk_edge(i, r.F.back().rev, j, r.S.back().rev);
                const bool d = edge_disc(e), pd = pair_disc(r, false);
                if (chim_mode ? (!d || pd) : (pd == d)) edges.push_back(e);
            }
        }
    }
    // BuildEdges, SegmentGraph.cpp:1932-1959
    // raw: when non-null, one (record index, edge_key packing) pair per edge RawEdgesOther emits, in emission order
    void build_edges(const SqmbView &conc, std::vector<Rd> &chim, std::vector<int64_t> *raw = nullptr) {
        int ffi = 0;
        for (Rd &r : chim) { if (r.F.empty() && r.S.empty()) continue; read_edges(r, ffi, true, true); }  // RawEdgesChim (weights = counts)
        const std::vector<std::string> names = names_of(chim);
        ffi = 0;
        Rd last;
        for (uint64_t ri = 0; ri < conc.n_rec; ri++) {  // RawEdgesOther, :1577-1687
            const Aln a = fetch(conc, ri);
            if (!gate(a, names, false)) continue;
            Rd rd = decode(a, o);
            sort_rpos(rd);
            add_mate_block(a, rd);
            if (rd_equal(last, rd)) continue;
            last = rd;
            bool build = rd.F.empty() || rd.S.empty();
            if (!build) build = (rd.F.front().rpos <= 15 || (a.first() && rd.fl)) && (rd.S.front().rpos <= 15 || (!a.first() && rd.sl));
            if (!build) continue;
            const size_t e0 = edges.size();
            read_edges(rd, ffi, false, a.first());
            if (raw)
                for (size_t k = e0; k < edges.size(); k++) {
                    const Edge &e = edges[k];
                    raw->push_back((int64_t)ri);
                    raw->push_back((int64_t)(((uint64_t)(uint32_t)e.a << 33) | ((uint64_t)(uint32_t)e.b << 2) | ((uint64_t)e.ha << 1) | (uint64_t)e.hb));
                }
        }
        std::sort(edges.begin(), edges.end(), edge_lt);
        std::vector<Edge> u;
        for (const Edge &e : edges) {
            if (!u.empty() && u.back().a == e.a && u.back().b == e.b && u.back().ha == e.ha && u.back().hb == e.hb) u.back().w += e.w;
            else u.push_back(e);
        }
        edges.clear();
        for (const Edge &e : u) if (e.w > 0) edges.push_back(e);
    }
    // the BAM pass of ExactBPConcordantSupport, SegmentGraph.cpp:3124-3166
    std::vector<int> bp_coverage(const SqmbView &conc, const std::vector<Rd> &chim, const std::vector<std::pair<int, int>> &bps) const {
        const std::vector<std::string> names = names_of(chim);
        std::vector<int> cov(bps.size(), 0);
        size_t ind = 0;
        for (uint64_t ri = 0; ri < conc.n_rec; ri++) {
            const Aln a = fetch(conc, ri);
            if (!gate(a, names, true)) continue;
            if (a.mate_mapped() && a.mchr == a.chr && a.mpos > a.pos) continue;
            if (a.mate_mapped() && a.mchr == a.chr && a.mpos == a.pos && a.second()) continue;
            if (ind == bps.size()) break;
            const int start = (a.mate_mapped() && a.mchr == a.chr) ? a.mpos : a.pos, end = a.end();
            if (a.chr > bps[ind].first || (a.chr == bps[ind].first && start > bps[ind].second + o.dist_pos)) ind++;
            for (size_t k = ind; k < bps.size(); k++) {
                if (a.chr == bps[k].first && start <= bps[k].second && end > bps[k].second) cov[k]++;
                else if (a.chr < bps[k].first || (a.chr == bps[k].first && end <= bps[k].second)) break;
            }
        }
        return cov;
    }
};

static void dump(const std::string &path, const std::vector<int32_t> &v) {
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) return;
    if (!v.empty()) fwrite(v.data(), 4, v.size(), f);
    fclose(f);
}
static std::vector<int32_t> chim_rows(const std::vector<Rd> &c) {
    std::vector<int32_t> a;
    for (size_t i = 0; i < c.size(); i++)
        for (int m = 0; m < 2; m++)
            for (const Blk &b : (m ? c[i].S : c[i].F)) { a.push_back((int32_t)i); a.push_back(m); a.push_back(b.chr); a.push_back(b.pos); a.push_back(b.rpos); a.push_back(b.mref); a.push_back(b.mread); a.push_back(b.rev); }
    return a;
}
static void set_opts(Opt &o, const int *opts) {
    if (opts) { o.phred33 = opts[0]; o.max_lowphred = opts[1]; o.min_phred = opts[2]; o.min_mapq = opts[3] < 0 ? 255 : opts[3]; o.dist_pos = opts[4]; o.dist_idx = opts[5]; }
}
static void dump_edges(const std::string &path, const std::vector<Edge> &edges) {
    std::vector<int32_t> a;
    for (const Edge &e : edges) { a.push_back(e.a); a.push_back(e.b); a.push_back(e.ha); a.push_back(e.hb); a.push_back(e.w); }
    dump(path, a);
}
}  // namespace

// opts: {phred33, max_lowphred_len, min_phred, min_mapq, concord_dist_pos, concord_dist_idx}; bps_file may be NULL.
// stop_after: 0 = everything, 1 = chimeric loader only, 2 = nodes, 3 = edges, -1 = the coverage pass alone (it reads neither
// segments nor edges; a stream too short to trigger a segment group can still be covered).  Returns 0, or <0 on I/O error.
extern "C" int sqo_run(const char *conc_path, const char *chim_path, const char *outdir, const int *opts, const char *bps_file, int stop_after) {
    SqmbView conc, chim;
    if (!conc.open(conc_path) || !chim.open(chim_path)) return -1;
    Graph g;
    set_opts(g.o, opts);
    g.ref_len.assign(conc.ref_len, conc.ref_len + conc.n_ref);
    std::vector<Rd> cr = load_chim(chim, g.o);
    const std::string d = outdir;
    dump(d + "/chim_loaded.bin", chim_rows(cr));
    {
        std::vector<int32_t> t;
        for (const Rd &r : cr) { t.push_back(r.ft); t.push_back(r.st); t.push_back(r.ft ? (int)r.fl : -1); t.push_back(r.st ? (int)r.sl : -1); }
        dump(d + "/chim_loaded.bin.meta", t);
    }
    dump(d + "/readlen.bin", std::vector<int32_t>{g.o.read_len});
    if (stop_after == 1) return 0;
    if (stop_after >= 0) {
        g.build_nodes(conc, cr);
        {
            std::vector<int32_t> a;
            std::vector<double> dep;
            for (const Node &n : g.nodes) { a.push_back(n.chr); a.push_back(n.pos); a.push_back(n.len); a.push_back(n.support); dep.push_back(n.depth); }
            dump(d + "/nodes_i32.bin", a);
            FILE *f = fopen((d + "/nodes_f64.bin").c_str(), "wb");
            if (f) { if (!dep.empty()) fwrite(dep.data(), 8, dep.size(), f); fclose(f); }
        }
        if (stop_after == 2) return 0;
        g.build_edges(conc, cr);
        dump_edges(d + "/edges_i32.bin", g.edges);
        dump(d + "/chim_after_edges.bin", chim_rows(cr));
    }
    if (stop_after == 3 || !bps_file) return 0;
    std::vector<std::pair<int, int>> bps;
    FILE *f = fopen(bps_file, "rb");
    if (!f) return -2;
    int32_t xy[2];
    while (fread(xy, 4, 2, f) == 2) bps.push_back({xy[0], xy[1]});
    fclose(f);
    const std::vector<int> cov = g.bp_coverage(conc, cr, bps);
    dump(d + "/cov_i32.bin", std::vector<int32_t>(cov.begin(), cov.end()));
    return 0;
}

// The per-record preamble of BuildNode_STAR over the WHOLE concordant stream (no stop at the last discordant group: that
// truncation belongs to the seed machine, not to the filter).  Writes classify_i32.bin, one row of 9 int32 per record:
//   class bits (sq_common.cuh's CLS_* values, defined from the reference's lines: GATE :302; KEEP = GATE and not Equal
//   :315-318; HASBLK = KEEP and own blocks :320-333; DISPL = HASBLK and own[0].pos != pos; CONC :651-655; PART :668-683;
//   REST = CONC, a mate flag and more than one own block),
//   first-block length of a CONC record (else 0), ConcordantCluster end (else INT32_MIN), otherrightmost contribution (else -1),
//   (otherChr, otherRight) in front of the record, coverage-pass qualification (:3136-3142), fragment start and end.
// Also writes readlen.bin.  Returns 0, or <0 on I/O error.
extern "C" int sqo_classify(const char *conc_path, const char *chim_path, const char *outdir, const int *opts) {
    SqmbView conc, chim;
    if (!conc.open(conc_path) || !chim.open(chim_path)) return -1;
    Graph g;
    set_opts(g.o, opts);
    g.ref_len.assign(conc.ref_len, conc.ref_len + conc.n_ref);
    const std::vector<Rd> cr = load_chim(chim, g.o);
    const std::vector<std::string> names = Graph::names_of(cr);
    std::vector<int32_t> rows;
    rows.reserve((size_t)conc.n_rec * 9);
    Rd last;
    Graph::RecClass rc;
    int otherChr = 0, otherRight = 0;
    for (uint64_t ri = 0; ri < conc.n_rec; ri++) {
        g.classify(conc, ri, names, last, rc);
        const Aln &a = rc.a;
        int cls = 0, flen = 0, cc_end = INT32_MIN, other_end = -1;
        if (rc.gate) cls |= 1;
        if (rc.keep) cls |= 2;
        if (rc.keep && rc.has_blk()) { cls |= 16; if (rc.own()[0].pos != a.pos) cls |= 32; }
        if (rc.conc) {
            cls |= 4;
            if (rc.part_f || rc.part_s) cls |= 8;
            else cc_end = (a.first() ? rc.rd.F.front() : rc.rd.S.front()).pos + (a.first() ? rc.rd.F.front() : rc.rd.S.front()).mref;
            flen = rc.own()[0].mref;
            const std::vector<Blk> *ownp = rc.other_own();
            if (ownp) {
                if (ownp->size() > 1) cls |= 64;
                other_end = ownp->front().pos + ownp->front().mref;
            }
        }
        const bool same = a.mate_mapped() && a.mchr == a.chr;
        const bool q = rc.gate && !(same && a.mpos > a.pos) && !(same && a.mpos == a.pos && a.second());
        const int32_t row[9] = {cls, flen, cc_end, other_end, otherChr, otherRight, q, same ? a.mpos : a.pos, a.end()};
        rows.insert(rows.end(), row, row + 9);
        if (other_end >= 0) {
            if (otherChr == a.chr) otherRight = std::max(otherRight, other_end); else { otherRight = other_end; otherChr = a.chr; }
        }
    }
    const std::string d = outdir;
    dump(d + "/classify_i32.bin", rows);
    dump(d + "/readlen.bin", std::vector<int32_t>{g.o.read_len});
    return 0;
}

// BuildEdges on a segment table the caller supplies (the graph reload of SegmentGraph_t(string), SegmentGraph.cpp:126-157):
// loads the chimeric reads, installs the (chr, pos, len) int32 rows of nodes_path as the segments and writes edges_i32.bin and
// chim_after_edges.bin.  dump_raw != 0 also writes raw_edges.bin: int64 (record index, packed key) rows, one per edge that
// RawEdgesOther emits, the key packed as sq_locate.cuh's edge_key packs it.  Returns 0, or <0 on I/O error.
extern "C" int sqo_edges_on_nodes(const char *conc_path, const char *chim_path, const char *outdir, const int *opts, const char *nodes_path, int dump_raw) {
    SqmbView conc, chim;
    if (!conc.open(conc_path) || !chim.open(chim_path)) return -1;
    Graph g;
    set_opts(g.o, opts);
    g.ref_len.assign(conc.ref_len, conc.ref_len + conc.n_ref);
    std::vector<Rd> cr = load_chim(chim, g.o);
    FILE *f = fopen(nodes_path, "rb");
    if (!f) return -2;
    int32_t row[3];
    while (fread(row, 4, 3, f) == 3) g.nodes.push_back(Node{row[0], row[1], row[2], 0, 0});
    fclose(f);
    std::vector<int64_t> raw;
    g.build_edges(conc, cr, dump_raw ? &raw : nullptr);
    const std::string d = outdir;
    dump_edges(d + "/edges_i32.bin", g.edges);
    dump(d + "/chim_after_edges.bin", chim_rows(cr));
    if (dump_raw) {
        FILE *r = fopen((d + "/raw_edges.bin").c_str(), "wb");
        if (!r) return -3;
        if (!raw.empty()) fwrite(raw.data(), 8, raw.size(), r);
        fclose(r);
    }
    return 0;
}
