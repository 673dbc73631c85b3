// Host twin of SQUID's read model: CIGAR -> aligned blocks, discordance predicates.
// Follows the behaviour of src/ReadRec.cpp (cited per function); written from scratch.
#include "readrec.h"

#include <algorithm>

#include "sq_cigar.cuh"

namespace sqh {

// src/ReadRec.cpp:10-88 through the shared CIGAR rules (sq_cigar.cuh).  Without explicit bases and qualities the record carries
// summaries instead: `synth_lowrun` times '#' then 'I' as qualities, and `synth_polya` bits for its first four blocks.
void decode_alignment(const Alignment &a, const HostConfig &cfg, Decoded &out) {
    out.blocks.clear();
    auto op = [&a](uint32_t i) { return a.cigar[i]; };
    const sq::CigarSummary s = sq::cigar_summary(op, a.n_cigar, a.pos);
    out.total_len = s.total_len;
    out.end_pos = s.end_pos;

    const int thr = sq::phred_threshold(cfg.phred33, cfg.min_phred);
    if (a.qual) out.lowphred_run = sq::low_quality_run([&a](uint32_t i) { return (int)(signed char)a.qual[i]; }, a.l_seq, thr);
    else out.lowphred_run = 'I' < thr ? s.lseq : '#' < thr ? std::min<int>(a.synth_lowrun, s.lseq) : 0;

    const bool rev = a.is_reverse(), first = a.is_first();
    auto keep = [&](int32_t ref_pos, int32_t match_ref, int32_t read_pos, int32_t match_read) {
        out.blocks.push_back(Block{a.ref_id, ref_pos, read_pos, match_ref, match_read, a.mapq, rev, first});
    };
    if (a.seq) {
        sq::cigar_blocks(op, a.n_cigar, a.pos, s.total_len, rev, [&a](uint32_t, int32_t lo, int32_t hi) {
            sq::ATCount n{0, 0};
            for (int32_t k = std::max(lo, 0); k < std::min(hi, (int32_t)a.l_seq); k++) {  // the reference asserts instead of clamping
                const char c = a.seq[k];
                if (c == 'a' || c == 'A') n.a++;
                else if (c == 't' || c == 'T') n.t++;
            }
            return n;
        }, keep);
    } else {
        sq::cigar_blocks(op, a.n_cigar, a.pos, s.total_len, rev, [&a](uint32_t k, int32_t lo, int32_t hi) {
            sq::ATCount n{0, 0};
            if (k < 4) {
                if (a.synth_polya >> (4 + k) & 1) n.t = hi - lo;  // painted last => wins
                else if (a.synth_polya >> k & 1) n.a = hi - lo;
            }
            return n;
        }, keep);
    }
}

void Read::sort_by_read_pos() {
    auto by_read_pos = [](const Block &x, const Block &y) { return x.read_pos < y.read_pos; };
    std::sort(first.begin(), first.end(), by_read_pos);
    std::sort(second.begin(), second.end(), by_read_pos);
}

bool Read::single_anchored() const { return (first.empty() || second.empty()) && !multi_filter; }

static bool mate_is_discordant(const std::vector<Block> &v) {
    for (size_t i = 0; i + 1 < v.size(); i++) {
        const Block &x = v[i], &y = v[i + 1];
        if (x.ref_id != y.ref_id || x.is_reverse != y.is_reverse) return true;
        const bool ref_fwd = x.ref_pos < y.ref_pos, read_fwd = x.read_pos < y.read_pos;
        if (!x.is_reverse && ref_fwd != read_fwd) return true;
        if (x.is_reverse && ref_fwd == read_fwd) return true;
    }
    return false;
}
bool Read::end_discordant(bool first_mate) const { return mate_is_discordant(first_mate ? first : second); }

bool Read::pair_discordant(bool check_ends) const {
    if (first.empty() || second.empty()) return false;
    if (check_ends && (end_discordant(true) || end_discordant(false))) return true;
    const Block &ff = first.front(), &fb = first.back(), &sf = second.front(), &sb = second.back();
    if (ff.ref_id != sb.ref_id || ff.is_reverse == sb.is_reverse) return true;
    if (!ff.is_reverse && ff.ref_pos - ff.read_pos > sb.ref_pos - (second_total - sb.read_pos - sb.match_read)) return true;
    if (!sf.is_reverse && sf.ref_pos - sf.read_pos > fb.ref_pos - (first_total - fb.read_pos - fb.match_read)) return true;
    return false;
}

static bool lists_match(const std::vector<Block> &x, const std::vector<Block> &y) {
    if (x.size() != y.size()) return false;
    for (size_t i = 0; i < x.size(); i++)
        if (x[i].ref_id != y[i].ref_id || x[i].ref_pos != y[i].ref_pos || x[i].match_ref != y[i].match_ref) return false;
    return true;
}
bool Read::equal(const Read &a, const Read &b) {
    return (lists_match(a.first, b.first) && lists_match(a.second, b.second)) ||
           (lists_match(a.first, b.second) && lists_match(a.second, b.first));
}

bool Read::front_smaller(const Read &a, const Read &b) {
    const Block *x = nullptr, *y = nullptr;
    if (!a.first.empty() && !b.first.empty()) { x = &a.first.front(); y = &b.first.front(); }
    else if (!a.second.empty() && !b.second.empty()) { x = &a.second.front(); y = &b.second.front(); }
    else if (!a.first.empty() && !b.second.empty()) { x = &a.first.front(); y = &b.second.front(); }
    else if (!a.second.empty() && !b.first.empty()) { x = &a.second.front(); y = &b.first.front(); }
    else return false;
    return x->ref_id != y->ref_id ? x->ref_id < y->ref_id : x->ref_pos < y->ref_pos;
}

}  // namespace sqh
