// BAM records in an inflated window, as `SQ_HD` rules (device: sqg_load_concordant_bam in sqg_api.cu; CPU: tests/emul/emul_bam.cpp).
//   * Record boundaries, whatever the writer.  A window is cut into segments at its BGZF member starts.  Per segment a
//     speculative first record start is searched (the first offset from which a chain of plausible records reaches the
//     segment's end or kSpecDepth records), and the segment is walked from it to its exit (the first record start at or past
//     its end).  Segment k is proven when the exit of segment k-1 equals its start: by induction from segment 0, which starts at
//     a true boundary (end of the header or of the previous window's last whole record), every proven start is a true one.
//     Segments that are not proven are walked again from their true entry, in rounds, until nothing changes; correctness never
//     depends on the search, only the number of rounds does.  The walk itself checks exactly what host/bam.cpp checks.
//   * The per-record decode of host/bam.cpp + pack_concordant + decode_alignment (host/readrec.cpp): fields, TotalLen,
//     GetEndPosition, the low-quality run, XA / IH with BamTools' GetTag<int> semantics, the ChimName probe, and the aligned
//     blocks (poly-A/T test on the 4-bit bases, strand flip).
#ifndef SQ_BAM_CUH
#define SQ_BAM_CUH
#include <stdint.h>

#include "sq_common.cuh"
#include "squid_b200.h"

namespace sq {

constexpr int kSpecDepth = 4;  // plausible records a speculative start needs (or the segment's end)
constexpr int kBamMaxRounds = 8;  // repair rounds before one sequential walk of the window

// one BGZF member of a window: deflate payload at comp[cdata, cdata + clen) -> win[out, out + isize)
struct BamMember { uint64_t cdata, out; uint32_t clen, isize, crc, pad; };

SQ_HD uint32_t bam_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
SQ_HD uint32_t bam_u32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

// The record whose block_size sits at b[p]: 1 = well formed as host/bam.cpp requires (*next = the following record), 0 = it
// does not end before L but could end before the stream does (Lstream: end of the stream in the same coordinates), -1 = malformed.
SQ_HD int bam_rec_check(const uint8_t *b, int64_t p, int64_t L, int64_t Lstream, int64_t *next) {
    if (p + 4 > L) return p + 4 > Lstream ? -1 : 0;
    const int32_t bs = (int32_t)bam_u32(b + p);
    if (bs < 32) return -1;
    if (p + 4 + bs > L) return p + 4 + bs > Lstream ? -1 : 0;
    const uint8_t *q = b + p + 4;
    const uint32_t l_name = q[8], n_cig = bam_u16(q + 12), l_seq = bam_u32(q + 16);
    if (32ull + l_name + 4ull * n_cig + ((uint64_t)l_seq + 1) / 2 + l_seq > (uint64_t)bs) return -1;
    *next = p + 4 + bs;
    return 1;
}
// Stricter, for the speculative search only: refID and next refID in [-1, n_ref), a NUL-terminated name.
SQ_HD int bam_rec_plausible(const uint8_t *b, int64_t p, int64_t L, int64_t Lstream, int32_t n_ref, int64_t *next) {
    const int r = bam_rec_check(b, p, L, Lstream, next);
    if (r != 1) return r;
    const uint8_t *q = b + p + 4;
    const int32_t rid = (int32_t)bam_u32(q), mrid = (int32_t)bam_u32(q + 20);
    const uint32_t l_name = q[8];
    if (rid < -1 || rid >= n_ref || mrid < -1 || mrid >= n_ref || l_name < 1 || q[32 + l_name - 1] != 0) return -1;
    return 1;
}

struct SegWalk { int64_t exit; uint32_t n; uint8_t bad; };
// Walk from a record start a through the segment ending at e: records whose start is < e.
SQ_HD SegWalk bam_walk(const uint8_t *b, int64_t a, int64_t e, int64_t L, int64_t Lstream, int64_t *rec_out) {
    SegWalk w{a, 0, 0};
    int64_t p = a;
    while (p < e) {
        int64_t nx = 0;
        const int r = bam_rec_check(b, p, L, Lstream, &nx);
        if (r == 0) break;            // the record goes on in the next window
        if (r < 0) { w.bad = 1; break; }
        if (rec_out) rec_out[w.n] = p;
        w.n++;
        p = nx;
    }
    w.exit = p;
    return w;
}
// Speculative first record start of the segment [s, e): e when no offset qualifies.
SQ_HD int64_t bam_spec_start(const uint8_t *b, int64_t s, int64_t e, int64_t L, int64_t Lstream, int32_t n_ref) {
    const int64_t hi = e < L ? e : L;
    for (int64_t o = s; o < hi; o++) {
        int64_t p = o;
        bool ok = true;
        for (int d = 0; d < kSpecDepth && p < e; d++) {
            int64_t nx = 0;
            const int r = bam_rec_plausible(b, p, L, Lstream, n_ref, &nx);
            if (r == 0) break;
            if (r < 0) { ok = false; break; }
            p = nx;
        }
        if (ok) return o;
    }
    return e;
}

// size of one aux value of type t at p (behind the type byte), 0 when malformed (host/bam.cpp aux_size)
SQ_HD uint64_t bam_aux_size(char t, const uint8_t *p, const uint8_t *end) {
    switch (t) {
        case 'A': case 'c': case 'C': return 1;
        case 's': case 'S': return 2;
        case 'i': case 'I': case 'f': return 4;
        case 'Z': case 'H': { const uint8_t *q = p; while (q < end && *q) q++; return q < end ? (uint64_t)(q - p) + 1 : 0; }
        case 'B': {
            if (p + 5 > end) return 0;
            const char st = (char)p[0];
            const uint64_t cnt = bam_u32(p + 1);
            const uint64_t es = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : (st == 'i' || st == 'I' || st == 'f') ? 4 : 0;
            return es ? 5 + cnt * es : 0;
        }
        default: return 0;
    }
}

// ChimName as an open-addressing set of 64-bit FNV-1a hashes (the packer's hash), each with its name for the exact compare.
struct NameSet {
    const uint64_t *hash;      // cap slots; a slot is empty when len == -1
    const int32_t *len;
    const int64_t *off;        // into blob
    const uint8_t *blob;
    uint64_t mask;             // cap - 1 (cap a power of two); cap == 0: no names, nothing is probed
    bool active;
};
SQ_HD uint64_t name_hash(const uint8_t *p, uint32_t n) { uint64_t h = 1469598103934665603ull; for (uint32_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ull; } return h; }
SQ_HD bool nameset_has(const NameSet &s, const uint8_t *p, uint32_t n) {
    const uint64_t h = name_hash(p, n);
    for (uint64_t k = h & s.mask;; k = (k + 1) & s.mask) {
        if (s.len[k] < 0) return false;
        if (s.hash[k] == h && (uint32_t)s.len[k] == n) {
            const uint8_t *q = s.blob + s.off[k];
            uint32_t i = 0;
            while (i < n && q[i] == p[i]) i++;
            if (i == n) return true;
        }
    }
}

struct BamDecodeParams { int32_t thr; };  // (signed char)(phred offset + min_phred), as decode_alignment compares

// The aligned blocks of a record (decode_alignment): block k goes to sink(k, ref_pos, match_ref, read_pos, match_read); returns
// their number.  rec: the record's block_size field.
template <class Sink>
SQ_HD uint32_t bam_blocks(const uint8_t *rec, Sink &&sink) {
    const uint8_t *p = rec + 4;
    const int32_t pos = (int32_t)bam_u32(p + 4);
    const uint32_t l_name = p[8], n_cig = bam_u16(p + 12), l_seq = bam_u32(p + 16);
    const uint16_t flag = (uint16_t)bam_u16(p + 14);
    const uint8_t *cig = p + 32 + l_name, *seq = cig + 4 * n_cig;
    int total = 0;
    for (uint32_t i = 0; i < n_cig; i++) {
        const uint32_t op = bam_u32(cig + 4 * i) & 15;
        if (op == 0 || op == 4 || op == 5 || op == 1 || op == 7 || op == 8) total += (int)(bam_u32(cig + 4 * i) >> 4);
    }
    const bool rev = (flag & 0x10) != 0;
    int read_pos = 0, ref_pos = pos, hard = 0;
    uint32_t nb = 0;
    for (uint32_t i = 0; i < n_cig; i++) {
        const uint32_t c = bam_u32(cig + 4 * i), op = c & 15;
        const int l = (int)(c >> 4);
        if (op == 4 || op == 5) {
            read_pos += l;
            if (op == 5) hard += l;
        } else if (op == 0 || op == 7) {  // a block opens at M or = and runs up to the next S, H or N
            int span_read = 0, span_ref = 0;
            uint32_t j = i;
            for (; j < n_cig; j++) {
                const uint32_t cj = bam_u32(cig + 4 * j), oj = cj & 15;
                if (oj == 4 || oj == 5 || oj == 3) break;
                if (oj != 2) span_read += (int)(cj >> 4);
                if (oj != 1) span_ref += (int)(cj >> 4);
            }
            int n_a = 0, n_t = 0;
            int k0 = read_pos - hard, k1 = read_pos + span_read - hard;
            if (k0 < 0) k0 = 0;
            if (k1 > (int)l_seq) k1 = (int)l_seq;
            for (int k = k0; k < k1; k++) {  // 4-bit codes: 1 = A, 8 = T
                const uint32_t v = (seq[k >> 1] >> ((k & 1) ? 0 : 4)) & 15;
                n_a += v == 1; n_t += v == 8;
            }
            if (4 * n_a < 3 * span_read && 4 * n_t < 3 * span_read) {  // poly-A/T blocks (>= 75 %) are dropped
                sink(nb, ref_pos, span_ref, rev ? total - read_pos - span_read : read_pos, span_read);
                nb++;
            }
            read_pos += span_read;
            ref_pos += span_ref;
            i = j - 1;
        } else if (op == 3) {
            ref_pos += l;
        }
    }
    return nb;
}

// One decoded record: the per-record fields of sqg_batch and the block count.
struct BamRec {
    int32_t ref_id, pos, mate_ref_id, mate_pos, end_pos;
    uint16_t flag; uint8_t mapq, aux;
    int32_t total_len, lowphred, lseq_cigar;
    uint32_t n_blk, l_seq;
    bool aux_bad;
};
// rec: the record's block_size field (the walk has checked that its fixed and variable-length fields fit).
SQ_HD void bam_decode(const uint8_t *rec, const BamDecodeParams &prm, const NameSet &names, BamRec &o) {
    const uint8_t *p = rec + 4;
    const uint8_t *end = p + (uint32_t)bam_u32(rec);
    o.ref_id = (int32_t)bam_u32(p); o.pos = (int32_t)bam_u32(p + 4);
    const uint32_t l_name = p[8];
    o.mapq = p[9];
    const uint32_t n_cig = bam_u16(p + 12);
    o.flag = (uint16_t)bam_u16(p + 14);
    const uint32_t l_seq = bam_u32(p + 16);
    o.l_seq = l_seq;
    o.mate_ref_id = (int32_t)bam_u32(p + 20); o.mate_pos = (int32_t)bam_u32(p + 24);
    const uint8_t *name = p + 32, *cig = name + l_name, *seq = cig + 4 * n_cig, *qual = seq + (l_seq + 1) / 2;
    // TotalLen, GetEndPosition and the read length the synthesised qualities would have (decode_alignment)
    int total = 0, lseq = 0;
    uint32_t endp = (uint32_t)o.pos;
    for (uint32_t i = 0; i < n_cig; i++) {
        const uint32_t c = bam_u32(cig + 4 * i), op = c & 15;
        const int l = (int)(c >> 4);
        if (op == 0 || op == 4 || op == 5 || op == 1 || op == 7 || op == 8) total += l;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) endp += (uint32_t)l;
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) lseq += l;
    }
    o.total_len = total; o.end_pos = (int32_t)endp; o.lseq_cigar = lseq;
    // longest run of qualities below the threshold, compared as the host compares (signed char)(q + 33)
    int best = 0, run = 0;
    for (uint32_t i = 0; i < l_seq; i++) {
        run = ((int)(signed char)(uint8_t)(qual[i] + 33) < prm.thr) ? run + 1 : 0;
        if (run > best) best = run;
    }
    o.lowphred = best;
    // aux: XA present, IH as GetTag<int> reads it (the last IH tag wins; non-integer types leave the value as it was)
    bool xa = false, ih = false;
    int32_t ihv = 0;
    o.aux_bad = false;
    const uint8_t *q = qual + l_seq;
    while (q + 3 <= end) {
        const char t0 = (char)q[0], t1 = (char)q[1], ty = (char)q[2];
        const uint64_t sz = bam_aux_size(ty, q + 3, end);
        if (sz == 0 || sz > (uint64_t)(end - (q + 3))) { o.aux_bad = true; break; }
        if (t0 == 'X' && t1 == 'A') xa = true;
        else if (t0 == 'I' && t1 == 'H') {
            ih = true;
            const uint8_t *v = q + 3;
            switch (ty) {
                case 'A': case 'c': case 'C': ihv = v[0]; break;
                case 's': case 'S': ihv = (int32_t)bam_u16(v); break;
                case 'i': case 'I': ihv = (int32_t)bam_u32(v); break;
                default: break;
            }
        }
        q += 3 + sz;
    }
    uint8_t aux = 0;
    if (xa) aux |= SQG_AUX_XA;
    if (ih && ihv > 1) aux |= SQG_AUX_IH_GT1;
    if (names.active && nameset_has(names, name, l_name ? l_name - 1 : 0)) aux |= SQG_AUX_CHIMNAME;
    o.aux = aux;
    o.n_blk = bam_blocks(rec, [](uint32_t, int32_t, int32_t, int32_t, int32_t) {});
}

}  // namespace sq
#endif
