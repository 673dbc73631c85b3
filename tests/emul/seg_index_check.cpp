// Exhaustive check of the segment table's position index (sq_common.cuh: seg_at and the lookups built on it) on the CPU.
//
//   seg_index_check TABLE BIN_SHIFT FORM
//
// TABLE: int32 n_ref, ref_len[n_ref], then rows (chr, pos, len) sorted by chromosome that tile each chromosome.  The index is
// built in FORM "packed" (headers and bin entries, as sqg_nodes.cu builds it for the device) or "plain" (chr_first, bin_off,
// bin_seg, as the CPU stepping harness builds it); BIN_SHIFT 0: no bins, the binary-search fallback.  For every position of every
// chromosome and a few positions past both ends, every lookup is compared with its definition over the plain arrays
// (std::upper_bound / std::lower_bound).  Prints the number of positions checked and exits 1 on the first mismatch.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "sq_common.cuh"

using namespace sq;

int main(int argc, char **argv) {
    if (argc != 4) { fprintf(stderr, "usage: %s TABLE BIN_SHIFT packed|plain\n", argv[0]); return 2; }
    const bool packed = std::string(argv[3]) == "packed";
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    int32_t n_ref = 0;
    if (fread(&n_ref, 4, 1, f) != 1 || n_ref <= 0) { fprintf(stderr, "bad table\n"); return 2; }
    std::vector<int32_t> ref_len(n_ref), nchr, npos, nend;
    if (fread(ref_len.data(), 4, n_ref, f) != (size_t)n_ref) { fprintf(stderr, "bad table\n"); return 2; }
    int32_t row[3];
    while (fread(row, 4, 3, f) == 3) { nchr.push_back(row[0]); npos.push_back(row[1]); nend.push_back(row[1] + row[2]); }
    fclose(f);
    const int32_t N = (int32_t)nchr.size();
    std::vector<int32_t> chr_first(n_ref + 1, N);
    for (int32_t i = N - 1; i >= 0; i--) chr_first[nchr[i]] = i;
    for (int32_t c = n_ref - 1; c >= 0; c--) if (chr_first[c] == N) chr_first[c] = chr_first[c + 1];

    NodeTable nt;
    nt.n = N; nt.n_ref = n_ref; nt.chr = nchr.data(); nt.pos = npos.data(); nt.end = nend.data();
    nt.bin_shift = atoi(argv[2]);
    std::vector<int32_t> bin_off(n_ref + 1, 0);
    if (nt.bin_shift > 0)
        for (int32_t c = 0; c < n_ref; c++) bin_off[c + 1] = bin_off[c] + (ref_len[c] >> nt.bin_shift) + 1;
    std::vector<ChrHead> head(n_ref);
    std::vector<BinEnt> bins;
    std::vector<int32_t> bin_seg;
    if (packed) {
        for (int32_t c = 0; c < n_ref; c++) head[c] = chr_head_value(chr_first.data(), nend.data(), bin_off.data(), c);
        nt.head = head.data();
    } else {
        nt.chr_first = chr_first.data();
        if (nt.bin_shift > 0) nt.bin_off = bin_off.data();
    }
    if (nt.bin_shift > 0) {
        bins.resize(bin_off[n_ref]);
        bin_seg.resize(bin_off[n_ref]);
        for (int32_t c = 0; c < n_ref; c++)
            for (int32_t k = 0; k < bin_off[c + 1] - bin_off[c]; k++) {
                bins[bin_off[c] + k] = bin_ent_value(nt, c, k, bin_off[c + 1] - bin_off[c]);
                bin_seg[bin_off[c] + k] = bin_seg_value(nt, c, k);
            }
        if (packed) nt.bins = bins.data();
        else nt.bin_seg = bin_seg.data();
    }

    long long checked = 0;
    const auto fail = [&](const char *what, int32_t c, int32_t x, int32_t got, int32_t want) {
        fprintf(stderr, "mismatch: %s chr %d x %d: got %d, want %d\n", what, c, x, got, want);
        return 1;
    };
    for (int32_t c = 0; c < n_ref; c++) {
        const int32_t c0 = chr_first[c], c1 = chr_first[c + 1];
        const ChrHead h = chr_head(nt, c);
        if (h.c0 != c0 || h.c1 != c1) return fail("header", c, 0, h.c0, c0);
        const int32_t lim = c1 > c0 ? nend[c1 - 1] : ref_len[c];
        for (int32_t x = -3; x <= lim + 3; x++, checked++) {
            const int32_t gt = (int32_t)(std::upper_bound(nend.begin() + c0, nend.begin() + c1, x) - nend.begin());
            const int32_t ge = (int32_t)(std::lower_bound(nend.begin() + c0, nend.begin() + c1, x) - nend.begin());
            const int32_t le = (int32_t)(std::upper_bound(npos.begin() + c0, npos.begin() + c1, x) - npos.begin()) - 1;
            const SegHit g = seg_first_end_gt(nt, h, x);
            if (g.s != gt) return fail("seg_first_end_gt", c, x, g.s, gt);
            if (g.s < c1 && (g.pos != npos[g.s] || g.end != nend[g.s])) return fail("seg_first_end_gt Position/End", c, x, g.pos, npos[g.s]);
            if (seg_first_end_ge(nt, h, x) != ge) return fail("seg_first_end_ge", c, x, seg_first_end_ge(nt, h, x), ge);
            if (seg_last_pos_le(nt, h, x) != le) return fail("seg_last_pos_le", c, x, seg_last_pos_le(nt, h, x), le);
            if (c1 > c0) {
                const int32_t want = gt < c1 ? gt : c1 - 1;
                const SegHit s = seg_at(nt, h, x);
                if (s.s != want) return fail("seg_at", c, x, s.s, want);
                if (s.pos != npos[want] || s.end != nend[want]) return fail("seg_at Position/End", c, x, s.pos, npos[want]);
            }
        }
    }
    printf("%lld\n", checked);
    return 0;
}
