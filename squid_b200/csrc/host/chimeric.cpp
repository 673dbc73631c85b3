// Host twin of BuildChimericSBamRecord and the SoA packer.  See chimeric.h.
#include "chimeric.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <thread>

#include "sq_cigar.cuh"

namespace sqh {

Alignment alignment_at(const SqmbView &v, uint64_t r) {
    Alignment a;
    a.ref_id = v.ref_id[r]; a.pos = v.pos[r]; a.mate_ref_id = v.mate_ref_id[r]; a.mate_pos = v.mate_pos[r];
    a.flag = v.flag[r]; a.mapq = v.mapq[r];
    a.tag_xa = v.aux[r] & 1; a.tag_ih = v.aux[r] & 2; a.ih_value = v.ih[r];
    a.cigar = v.cigar + v.cigar_off[r]; a.n_cigar = v.cigar_off[r + 1] - v.cigar_off[r];
    if (v.seq_off[r] >= 0) {
        const uint8_t *b = v.blob + v.seq_off[r];
        uint32_t l;
        memcpy(&l, b, 4);
        a.l_seq = l; a.seq = (const char *)b + 4; a.qual = (const char *)b + 4 + l;
    } else {
        a.synth_lowrun = v.lowrun[r]; a.synth_polya = v.polya[r];
    }
    return a;
}

std::string name_at(const SqmbView &v, uint64_t r) {
    std::string s = "q" + std::to_string(v.name_id[r]);
    if (v.aux[r] & 4) s += (v.flag[r] & 0x80) ? "/2" : "/1";
    return s;
}

// name_at() into a buffer: 'q' + decimal name_id (+ "/1" or "/2")
static size_t name_into_at(const SqmbView &v, uint64_t r, char *buf) {
    char tmp[24];
    int k = 0;
    long long x = (long long)v.name_id[r];
    const bool neg = x < 0;
    unsigned long long u = neg ? 0ull - (unsigned long long)x : (unsigned long long)x;
    do { tmp[k++] = (char)('0' + u % 10); u /= 10; } while (u);
    size_t n = 0;
    buf[n++] = 'q';
    if (neg) buf[n++] = '-';
    while (k) buf[n++] = tmp[--k];
    if (v.aux[r] & 4) { buf[n++] = '/'; buf[n++] = (v.flag[r] & 0x80) ? '2' : '1'; }
    return n;
}
AlnSource source_of(const SqmbView &v) {
    AlnSource s;
    s.n_rec = v.n_rec;
    s.at = [&v](uint64_t r) { return alignment_at(v, r); };
    s.name = [&v](uint64_t r) { return name_at(v, r); };
    s.name_into = [&v](uint64_t r, char *buf) { return name_into_at(v, r, buf); };
    return s;
}
void load_chimeric(const SqmbView &chim, HostConfig &cfg, std::vector<Read> &out) { load_chimeric(source_of(chim), cfg, out); }
int pack_concordant(const SqmbView &conc, const HostConfig &cfg, const std::unordered_set<std::string> &chim_names, PackedBatch &out, std::string &err) {
    return pack_concordant(source_of(conc), cfg, chim_names, out, err);
}

// src/ReadRec.cpp:329-413
void load_chimeric(const AlnSource &chim, HostConfig &cfg, std::vector<Read> &out) {
    std::vector<Read> recs;
    std::vector<int> sample;  // first five totals (ReadRec.cpp:336, 347-348)
    Decoded d;
    for (uint64_t r = 0; r < chim.n_rec; r++) {
        Alignment a = chim.at(r);
        if (!a.is_mapped() || a.is_dup()) continue;  // :344
        decode_alignment(a, cfg, d);
        Read rd;
        rd.qname = chim.name(r);
        if (rd.qname.size() >= 2) {  // :12-13
            const std::string tail = rd.qname.substr(rd.qname.size() - 2);
            if (tail == "/1" || tail == "/2") rd.qname.resize(rd.qname.size() - 2);
        }
        const bool low = d.lowphred_run > cfg.max_lowphred_len;
        if (a.is_first()) { rd.first_total = d.total_len; rd.first_low = low; rd.first = d.blocks; }
        else { rd.second_total = d.total_len; rd.second_low = low; rd.second = d.blocks; }
        if (sample.size() < 5) sample.push_back(std::max(rd.first_total, rd.second_total));
        recs.push_back(std::move(rd));
    }
    // group by Qname: same unstable std::sort on the same sequence with the same ordering as the
    // reference (:354) so that equal-name records merge in the same order
    std::sort(recs.begin(), recs.end(), [](const Read &x, const Read &y) { return x.qname < y.qname; });
    std::vector<Read> merged;
    merged.reserve(recs.size());
    for (Read &r : recs) {
        if (merged.empty() || r.qname != merged.back().qname) { merged.push_back(std::move(r)); continue; }
        Read &m = merged.back();  // :359-372
        if (m.first_total == 0 && r.first_total != 0) { m.first_total = r.first_total; m.first_low = r.first_low; }
        if (m.second_total == 0 && r.second_total != 0) { m.second_total = r.second_total; m.second_low = r.second_low; }
        m.first.insert(m.first.end(), r.first.begin(), r.first.end());
        m.second.insert(m.second.end(), r.second.begin(), r.second.end());
    }
    for (Read &r : merged) r.sort_by_read_pos();
    if (!sample.empty()) {  // :378-379
        std::sort(sample.begin(), sample.end());
        cfg.read_len = sample[sample.size() / 2];
    }
    std::sort(merged.begin(), merged.end(), Read::front_smaller);  // :382
    // PCR duplicates: same first-mate front position and Equal() to an already kept read (:388-409)
    out.clear();
    for (Read &r : merged) {
        bool dup = false;
        if (!out.empty() && !r.first.empty() && !out.back().first.empty() &&
            r.first.front().ref_id == out.back().first.front().ref_id && r.first.front().ref_pos == out.back().first.front().ref_pos) {
            for (size_t k = out.size(); k-- > 0;) {
                const Read &o = out[k];
                if (o.first.empty() || o.first.front().ref_id != r.first.front().ref_id || o.first.front().ref_pos != r.first.front().ref_pos) break;
                if (Read::equal(r, o)) { dup = true; break; }
            }
        }
        if (!dup) out.push_back(std::move(r));
    }
}

sqg_batch PackedBatch::view() const {
    sqg_batch b;
    b.n_rec = (int64_t)ref_id.size(); b.n_blk = (int64_t)blk_ref_pos.size();
    b.ref_id = ref_id.data(); b.pos = pos.data(); b.mate_ref_id = mate_ref_id.data(); b.mate_pos = mate_pos.data(); b.end_pos = end_pos.data();
    b.flag = flag.data(); b.total_len = total_len.data(); b.lowphred_run = lowphred_run.data();
    b.mapq = mapq.data(); b.aux = aux.data(); b.blk_off = blk_off.data();
    b.blk_ref_pos = blk_ref_pos.data(); b.blk_match_ref = blk_match_ref.data();
    b.blk_read_pos = blk_read_pos.data(); b.blk_match_read = blk_match_read.data();
    return b;
}

std::string packer_refusal(uint64_t r, int limit, int64_t total_len) {
    if (limit == 1) return "record " + std::to_string(r) + " has more than 16 aligned blocks";
    // the batch keeps read coordinates in 16 bits (include/squid_b200.h): a longer read is refused, never wrapped
    return "record " + std::to_string(r) + " is longer than 65535 bases (TotalLen " + std::to_string(total_len) + ")";
}

int pack_concordant(const AlnSource &conc, const HostConfig &cfg, const std::unordered_set<std::string> &chim_names, PackedBatch &out, std::string &err) {
    const uint64_t n = conc.n_rec;
    const bool timing = getenv("SQH_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) { if (!timing) return; const auto t = std::chrono::steady_clock::now(); fprintf(stderr, "[sqh]   pack: %-20s %8.3f ms\n", what, 1e3 * std::chrono::duration<double>(t - t_last).count()); t_last = t; };
    out.ref_id.resize(n); out.pos.resize(n); out.mate_ref_id.resize(n); out.mate_pos.resize(n); out.flag.resize(n); out.mapq.resize(n);
    out.end_pos.resize(n); out.total_len.resize(n); out.lowphred_run.resize(n); out.aux.resize(n);
    out.blk_off.assign(n + 1, 0);
    lap("allocate");
    // ChimName probe (SegmentGraph.cpp:302, a binary search over strings in the reference): nearly every record misses, so a
    // two-probe Bloom filter over a 64-bit hash of the name answers first and only a hit goes to the exact set
    auto fnv = [](const char *p, size_t len) { uint64_t h = 1469598103934665603ull; for (size_t i = 0; i < len; i++) { h ^= (unsigned char)p[i]; h *= 1099511628211ull; } return h; };
    size_t bloom_bits = 1024;
    while (bloom_bits < 16 * chim_names.size()) bloom_bits <<= 1;
    std::vector<uint64_t> bloom(bloom_bits / 64, 0);
    for (const std::string &nm : chim_names) {
        const uint64_t h = fnv(nm.data(), nm.size());
        const uint64_t a = h & (bloom_bits - 1), b2 = (h >> 32) & (bloom_bits - 1);
        bloom[a >> 6] |= 1ull << (a & 63); bloom[b2 >> 6] |= 1ull << (b2 & 63);
    }
    const bool probe_names = !chim_names.empty();
    // pass 1 (parallel over record ranges): per-record summaries and block counts
    const unsigned nt = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    std::vector<std::vector<Block>> tblocks(nt);
    std::vector<std::string> terr(nt);
    auto work = [&](unsigned t) {
        const uint64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        Decoded d;
        std::vector<Block> &acc = tblocks[t];
        acc.reserve((size_t)((hi - lo) + (hi - lo) / 2 + 16));
        char nbuf[320];
        for (uint64_t r = lo; r < hi; r++) {
            Alignment a = conc.at(r);
            out.ref_id[r] = a.ref_id; out.pos[r] = a.pos; out.mate_ref_id[r] = a.mate_ref_id; out.mate_pos[r] = a.mate_pos;
            out.flag[r] = a.flag; out.mapq[r] = a.mapq;
            decode_alignment(a, cfg, d);
            if (const int lim = sq::packer_limit((uint32_t)d.blocks.size(), d.total_len)) { terr[t] = packer_refusal(r, lim, d.total_len); return; }
            out.end_pos[r] = d.end_pos;
            out.total_len[r] = (uint16_t)d.total_len;
            out.lowphred_run[r] = (uint16_t)std::min(d.lowphred_run, 65535);  // <= total_len
            uint8_t aux = 0;
            if (a.tag_xa) aux |= SQG_AUX_XA;
            if (a.tag_ih && a.ih_value > 1) aux |= SQG_AUX_IH_GT1;
            if (probe_names) {
                bool maybe = true;
                if (conc.name_into) {
                    const size_t len = conc.name_into(r, nbuf);
                    const uint64_t h = fnv(nbuf, len);
                    const uint64_t x = h & (bloom_bits - 1), y = (h >> 32) & (bloom_bits - 1);
                    maybe = ((bloom[x >> 6] >> (x & 63)) & 1ull) && ((bloom[y >> 6] >> (y & 63)) & 1ull);
                    if (maybe && chim_names.count(std::string(nbuf, len))) aux |= SQG_AUX_CHIMNAME;
                } else if (chim_names.count(conc.name(r))) aux |= SQG_AUX_CHIMNAME;
            }
            out.aux[r] = aux;
            out.blk_off[r + 1] = (uint32_t)d.blocks.size();
            acc.insert(acc.end(), d.blocks.begin(), d.blocks.end());
        }
    };
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++) th.emplace_back(work, t);
    for (auto &x : th) x.join();
    lap("decode (parallel)");
    for (unsigned t = 0; t < nt; t++) if (!terr[t].empty()) { err = terr[t]; return SQG_EUNSUPPORTED; }
    // block offsets: every thread's range starts where the blocks of the ranges before it end
    std::vector<uint64_t> tbase(nt + 1, 0);
    for (unsigned t = 0; t < nt; t++) tbase[t + 1] = tbase[t] + tblocks[t].size();
    if (tbase[nt] > 0xFFFFFFFFull) { err = "more than 2^32 - 1 aligned blocks in one batch: shard the stream"; return SQG_EUNSUPPORTED; }
    const size_t nb = (size_t)tbase[nt];
    out.blk_ref_pos.resize(nb); out.blk_match_ref.resize(nb); out.blk_read_pos.resize(nb); out.blk_match_read.resize(nb);
    auto tail = [&](unsigned t) {
        const uint64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        uint32_t run = (uint32_t)tbase[t];
        for (uint64_t r = lo; r < hi; r++) { const uint32_t c = out.blk_off[r + 1]; out.blk_off[r + 1] = run + c; run += c; }  // blk_off[r + 1] = blocks up to and including r
        size_t o = (size_t)tbase[t];
        for (const Block &b : tblocks[t]) {
            out.blk_ref_pos[o] = b.ref_pos; out.blk_match_ref[o] = b.match_ref;
            out.blk_read_pos[o] = (uint16_t)b.read_pos; out.blk_match_read[o] = (uint16_t)b.match_read;
            o++;
        }
    };
    th.clear();
    for (unsigned t = 0; t < nt; t++) th.emplace_back(tail, t);
    for (auto &x : th) x.join();
    lap("offsets + block copy");
    return SQG_OK;
}

sqg_chimeric PackedChimeric::view() {
    sqg_chimeric c;
    c.n_reads = (int64_t)n_first.size(); c.n_blk = (int64_t)blk_ref_id.size();
    c.read_off = read_off.data(); c.n_first = n_first.data();
    c.first_total_len = first_total.data(); c.second_total_len = second_total.data();
    c.first_lowphred = first_low.data(); c.second_lowphred = second_low.data(); c.multi_filter = multi_filter.data();
    c.blk_ref_id = blk_ref_id.data(); c.blk_ref_pos = blk_ref_pos.data(); c.blk_read_pos = blk_read_pos.data();
    c.blk_match_ref = blk_match_ref.data(); c.blk_match_read = blk_match_read.data(); c.blk_is_reverse = blk_is_reverse.data();
    return c;
}

void PackedChimeric::from_reads(const std::vector<Read> &reads) {
    *this = PackedChimeric();
    read_off.push_back(0);
    for (const Read &r : reads) {
        n_first.push_back((uint16_t)r.first.size());
        first_total.push_back(r.first_total); second_total.push_back(r.second_total);
        first_low.push_back(r.first_low); second_low.push_back(r.second_low); multi_filter.push_back(r.multi_filter);
        for (int m = 0; m < 2; m++)
            for (const Block &b : (m ? r.second : r.first)) {
                blk_ref_id.push_back(b.ref_id); blk_ref_pos.push_back(b.ref_pos); blk_read_pos.push_back(b.read_pos);
                blk_match_ref.push_back(b.match_ref); blk_match_read.push_back(b.match_read); blk_is_reverse.push_back(b.is_reverse);
            }
        read_off.push_back((uint32_t)blk_ref_id.size());
    }
}

void PackedChimeric::to_reads(std::vector<Read> &reads) const {
    for (size_t i = 0; i < reads.size(); i++) {
        size_t o = read_off[i];
        for (int m = 0; m < 2; m++)
            for (Block &b : (m ? reads[i].second : reads[i].first)) {
                b.ref_pos = blk_ref_pos[o]; b.read_pos = blk_read_pos[o]; b.match_ref = blk_match_ref[o]; b.match_read = blk_match_read[o];
                o++;
            }
    }
}

}  // namespace sqh
