// The CIGAR rules of SQUID's read model (src/ReadRec.cpp:10-88, BamTools GetEndPosition), as `SQ_HD` code: the one definition the
// host packer (host/readrec.cpp decode_alignment) and the device decoder (sq_bam.cuh) both run.  A CIGAR is read through an
// accessor `op(i)` that returns element i in the BAM encoding len << 4 | op.
#ifndef SQ_CIGAR_CUH
#define SQ_CIGAR_CUH
#include <stdint.h>

#include "sq_common.cuh"

namespace sq {

enum : uint32_t { CIG_M = 0, CIG_I, CIG_D, CIG_N, CIG_S, CIG_H, CIG_P, CIG_EQ, CIG_X };
constexpr uint32_t kCigTotal = 1u << CIG_M | 1u << CIG_S | 1u << CIG_H | 1u << CIG_I | 1u << CIG_EQ | 1u << CIG_X;  // TotalLen (ReadRec.cpp:16-18)
constexpr uint32_t kCigRef = 1u << CIG_M | 1u << CIG_D | 1u << CIG_N | 1u << CIG_EQ | 1u << CIG_X;                  // GetEndPosition
constexpr uint32_t kCigSeq = 1u << CIG_M | 1u << CIG_I | 1u << CIG_S | 1u << CIG_EQ | 1u << CIG_X;                  // the bases a record holds

struct CigarSummary {
    int32_t total_len;  // TotalLen: sum of M, S, H, I, =, X
    int32_t end_pos;    // pos + sum of M, D, N, =, X, in unsigned arithmetic
    int32_t lseq;       // sum of M, I, S, =, X: the read length of synthesised qualities
};
template <class Op>
SQ_HD CigarSummary cigar_summary(Op op, uint32_t n, int32_t pos) {
    int32_t total = 0, lseq = 0;
    uint32_t end = (uint32_t)pos;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t c = op(i), bit = 1u << (c & 15);
        const int32_t l = (int32_t)(c >> 4);
        if (bit & kCigTotal) total += l;
        if (bit & kCigRef) end += (uint32_t)l;
        if (bit & kCigSeq) lseq += l;
    }
    return CigarSummary{total, (int32_t)end, lseq};
}

struct ATCount { int32_t a, t; };
// The aligned blocks of a CIGAR (ReadRec.cpp:46-87); returns how many were kept.  Quirks kept on purpose (SURVEY.md App. A-15, E3,
// E4, E7):
//  * a block opens at M or = and swallows every op up to the next S, H or N (D adds to the reference span only, I to the read
//    span only, P and X to both);
//  * I, D, X, P met outside a block are skipped without advancing anything;
//  * count(k, lo, hi) gives the A and T bases of block k at read offsets [lo, hi) (lo = read position - hard clips, hi - lo = the
//    block's read span; the range may leave the bases), and a block with >= 75 % of either is dropped;
//  * a kept block goes to sink(ref_pos, match_ref, read_pos, match_read), with read_pos = total_len - read_pos - span on the
//    reverse strand.
template <class Op, class Count, class Sink>
SQ_HD uint32_t cigar_blocks(Op op, uint32_t n, int32_t pos, int32_t total_len, bool rev, Count &&count, Sink &&sink) {
    int32_t read_pos = 0, ref_pos = pos, hard = 0;
    uint32_t kept = 0, k = 0;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t c = op(i), o = c & 15;
        const int32_t l = (int32_t)(c >> 4);
        if (o == CIG_S || o == CIG_H) {
            read_pos += l;
            if (o == CIG_H) hard += l;
        } else if (o == CIG_M || o == CIG_EQ) {
            int32_t span_read = 0, span_ref = 0;
            uint32_t j = i;
            for (; j < n; j++) {
                const uint32_t cj = op(j), oj = cj & 15;
                if (oj == CIG_S || oj == CIG_H || oj == CIG_N) break;
                if (oj != CIG_D) span_read += (int32_t)(cj >> 4);
                if (oj != CIG_I) span_ref += (int32_t)(cj >> 4);
            }
            const ATCount at = count(k, read_pos - hard, read_pos - hard + span_read);
            // 1.0 * n / span < 0.75  <=>  4n < 3 span for the integer ranges that occur
            if (4 * at.a < 3 * span_read && 4 * at.t < 3 * span_read) {
                sink(ref_pos, span_ref, rev ? total_len - read_pos - span_read : read_pos, span_read);
                kept++;
            }
            read_pos += span_read;
            ref_pos += span_ref;
            k++;
            i = j - 1;
        } else if (o == CIG_N) {
            ref_pos += l;
        }
    }
    return kept;
}

// What a packed batch holds of one record (read coordinates in 16 bits, include/squid_b200.h; a mate's blocks in kMaxBlocks
// slots): 0 = the record fits, 1 = more than kMaxBlocks blocks (tested first), 2 = TotalLen above 65535.
SQ_HD int packer_limit(uint32_t n_blk, int32_t total_len) { return n_blk > (uint32_t)kMaxBlocks ? 1 : total_len > 65535 ? 2 : 0; }

// The quality threshold of -pt / -pm as ReadRec.cpp:19-38 compares it: (signed char)(phred offset + min_phred).
SQ_HD int32_t phred_threshold(bool phred33, int32_t min_phred) { return (int32_t)(signed char)((phred33 ? 33 : 64) + min_phred); }
// Longest run of qualities below thr; q(i) is quality character i as a signed char.
template <class Q>
SQ_HD int32_t low_quality_run(Q q, uint32_t n, int32_t thr) {
    int32_t best = 0, run = 0;
    for (uint32_t i = 0; i < n; i++) {
        run = q(i) < thr ? run + 1 : 0;
        if (run > best) best = run;
    }
    return best;
}

}  // namespace sq
#endif
