// The BAM record rules, as `SQ_HD` code: the one definition the host BAM front end (host/bam.cpp), the device decoder
// (sqg_load_concordant_bam in sqg_api.cu) and its CPU stepping (tests/emul/emul_bam.cpp) all run.
//   * Record well-formedness (bam_rec_check), aux value sizes and the XA / IH scan with BamTools' GetTag<int> semantics.
//   * Record boundaries, whatever the writer.  A window is cut into segments at its BGZF member starts.  Per segment a
//     speculative first record start is searched (the first offset from which a chain of plausible records reaches the
//     segment's end or kSpecDepth records), and the segment is walked from it to its exit (the first record start at or past
//     its end).  Segment k is proven when the exit of segment k-1 equals its start: by induction from segment 0, which starts at
//     a true boundary (end of the header or of the previous window's last whole record), every proven start is a true one.
//     Segments that are not proven are walked again from their true entry, in rounds, until nothing changes; correctness never
//     depends on the search, only the number of rounds does.
//   * The per-record decode of the device: fields, the CIGAR rules of sq_cigar.cuh (TotalLen, GetEndPosition, the low-quality
//     run, the aligned blocks with the poly-A/T test on the 4-bit bases), XA / IH and the ChimName probe.
#ifndef SQ_BAM_CUH
#define SQ_BAM_CUH
#include <stdint.h>

#include "sq_cigar.cuh"
#include "sq_common.cuh"
#include "squid_b200.h"

namespace sq {

constexpr int kSpecDepth = 4;  // plausible records a speculative start needs (or the segment's end)
constexpr int kBamMaxRounds = 8;  // repair rounds before one sequential walk of the window

// one BGZF member of a window: deflate payload at comp[cdata, cdata + clen) -> win[out, out + isize)
struct BamMember { uint64_t cdata, out; uint32_t clen, isize, crc, pad; };

SQ_HD uint32_t bam_u16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
SQ_HD uint32_t bam_u32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

// The record whose block_size sits at b[p]: 1 = well formed (block_size >= 32 and the variable-length fields fit inside it; *next =
// the following record), 0 = it does not end before L but could end before the stream does (Lstream: end of the stream in the
// same coordinates), -1 = malformed.
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

// size of one aux value of type t at p (behind the type byte), 0 when malformed
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

// The aux fields [q, end) of a record: XA present, IH present and its value as BamTools' GetTag<int> reads it (the destination is
// zeroed and the 1, 2 or 4 value bytes are copied over its low end: no sign extension of the narrow signed types; 'A' converts as
// well; any other type leaves the value as it was; the last IH wins).  false when a field is malformed.
struct BamAux { bool xa, ih; int32_t ih_value; };
SQ_HD bool bam_aux_scan(const uint8_t *q, const uint8_t *end, BamAux &a) {
    a = BamAux{false, false, 0};
    while (q + 3 <= end) {
        const char t0 = (char)q[0], t1 = (char)q[1], ty = (char)q[2];
        const uint64_t sz = bam_aux_size(ty, q + 3, end);
        if (sz == 0 || sz > (uint64_t)(end - (q + 3))) return false;
        if (t0 == 'X' && t1 == 'A') a.xa = true;
        else if (t0 == 'I' && t1 == 'H') {
            a.ih = true;
            const uint8_t *v = q + 3;
            switch (ty) {
                case 'A': case 'c': case 'C': a.ih_value = v[0]; break;
                case 's': case 'S': a.ih_value = (int32_t)bam_u16(v); break;
                case 'i': case 'I': a.ih_value = (int32_t)bam_u32(v); break;
                default: break;
            }
        }
        q += 3 + sz;
    }
    return true;
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

struct BamDecodeParams { int32_t thr; };  // phred_threshold(-pt, -pm)

// CIGAR element i of a record whose CIGAR starts at cig (unaligned little-endian bytes)
struct BamCigar {
    const uint8_t *cig;
    SQ_HD uint32_t operator()(uint32_t i) const { return bam_u32(cig + 4 * i); }
};

// The aligned blocks of a record (cigar_blocks, the poly-A/T test on the 4-bit bases): block k goes to sink(k, ref_pos, match_ref,
// read_pos, match_read); returns their number.  rec: the record's block_size field.
template <class Sink>
SQ_HD uint32_t bam_blocks(const uint8_t *rec, Sink &&sink) {
    const uint8_t *p = rec + 4;
    const int32_t pos = (int32_t)bam_u32(p + 4);
    const uint32_t l_name = p[8], n_cig = bam_u16(p + 12), l_seq = bam_u32(p + 16);
    const uint16_t flag = (uint16_t)bam_u16(p + 14);
    const BamCigar op{p + 32 + l_name};
    const uint8_t *seq = op.cig + 4 * n_cig;
    uint32_t k = 0;
    return cigar_blocks(op, n_cig, pos, cigar_summary(op, n_cig, pos).total_len, flag_rev(flag), [&](uint32_t, int32_t lo, int32_t hi) {
        ATCount n{0, 0};
        if (lo < 0) lo = 0;
        if (hi > (int32_t)l_seq) hi = (int32_t)l_seq;
        for (int32_t i = lo; i < hi; i++) {  // 4-bit codes: 1 = A, 8 = T
            const uint32_t v = (seq[i >> 1] >> ((i & 1) ? 0 : 4)) & 15;
            n.a += v == 1; n.t += v == 8;
        }
        return n;
    }, [&](int32_t ref_pos, int32_t match_ref, int32_t read_pos, int32_t match_read) { sink(k++, ref_pos, match_ref, read_pos, match_read); });
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
    const uint8_t *name = p + 32;
    const BamCigar op{name + l_name};
    const uint8_t *qual = op.cig + 4 * n_cig + (l_seq + 1) / 2;
    const CigarSummary s = cigar_summary(op, n_cig, o.pos);
    o.total_len = s.total_len; o.end_pos = s.end_pos; o.lseq_cigar = s.lseq;
    // qualities compared as the host front end spells them: (signed char)(q + 33)
    o.lowphred = low_quality_run([qual](uint32_t i) { return (int32_t)(signed char)(uint8_t)(qual[i] + 33); }, l_seq, prm.thr);
    BamAux a;
    o.aux_bad = !bam_aux_scan(qual + l_seq, end, a);
    uint8_t aux = 0;
    if (a.xa) aux |= SQG_AUX_XA;
    if (a.ih && a.ih_value > 1) aux |= SQG_AUX_IH_GT1;
    if (names.active && nameset_has(names, name, l_name ? l_name - 1 : 0)) aux |= SQG_AUX_CHIMNAME;
    o.aux = aux;
    o.n_blk = bam_blocks(rec, [](uint32_t, int32_t, int32_t, int32_t, int32_t) {});
}

}  // namespace sq
#endif
