// RFC 1951 inflate of one BGZF member and its CRC32, as `SQ_HD` rules: the device runs them one member per warp
// (k_bam_inflate in sqg_api.cu: lane 0 decodes, the warp copies long matches), tests/emul/emul_bam.cpp steps them on the CPU
// against zlib.  What counts as a corrupt stream is what zlib's raw inflate refuses (inflate.c / inftrees.c), because the host
// front end (host/bam.cpp) is the yardstick: over-subscribed codes, incomplete codes except a lone 1-bit code for literals or
// distances, a missing end-of-block code, HLIT > 286 or HDIST > 30, a repeat with no previous length or past the end, literal /
// length symbols 286-287 and distance symbols 30-31, a distance before the member's start, stored-length complement mismatch,
// block type 3, more input needed than the member has, and output beyond ISIZE.  Input after the final block is ignored, as
// zlib does.
#ifndef SQ_INFLATE_CUH
#define SQ_INFLATE_CUH
#include <stdint.h>

#include "sq_common.cuh"

namespace sq {

constexpr int kInflLitBits = 10;   // primary lookup of the literal / length code (longer codes take the canonical walk)
constexpr int kInflDistBits = 8;
constexpr uint32_t kInflWarpCopyMin = 16;  // matches at least this long are returned to the caller (the warp copies them)

struct HuffCode {  // canonical Huffman code: count of codes per length, symbols sorted by (length, symbol)
    uint16_t count[16];
    uint16_t sym[288];
};
// Decoder tables of one member (shared memory on the device: 3.9 KB).
struct InflateTables {
    uint16_t lfast[1 << kInflLitBits];   // (symbol << 4) | length for codes of <= kInflLitBits bits; 0: longer (or no) code
    uint16_t dfast[1 << kInflDistBits];
    HuffCode lit;
    HuffCode dist;                       // also the code-length code while a dynamic header is read
    uint8_t lens[320];
};

SQ_HD uint32_t inflate_rev(uint32_t c, int n) { uint32_t r = 0; for (int i = 0; i < n; i++) { r = (r << 1) | (c & 1); c >>= 1; } return r; }

// Builds a canonical code from n lengths.  Returns 0 when zlib accepts the code, -1 when it refuses it (kind 0: code lengths,
// which must be complete; 1: literals / lengths and 2: distances, which may be incomplete only as one code of one bit, and may
// be empty: every decode then fails).
SQ_HD int inflate_build(HuffCode &h, const uint8_t *len, int n, uint16_t *fast, int fast_bits, int kind) {
    for (int l = 0; l < 16; l++) h.count[l] = 0;
    for (int s = 0; s < n; s++) h.count[len[s]]++;
    if (fast) for (int i = 0; i < (1 << fast_bits); i++) fast[i] = 0;
    int max = 15;
    while (max >= 1 && h.count[max] == 0) max--;
    if (max == 0) return kind == 0 ? -1 : 0;  // no codes (a code-length code without codes decodes no valid header either)
    int left = 1;
    for (int l = 1; l < 16; l++) { left <<= 1; left -= h.count[l]; if (left < 0) return -1; }
    if (left > 0 && (kind == 0 || max != 1)) return -1;
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; l++) offs[l + 1] = (uint16_t)(offs[l] + h.count[l]);
    for (int s = 0; s < n; s++) if (len[s]) h.sym[offs[len[s]]++] = (uint16_t)s;
    if (fast) {  // canonical codes in (length, symbol) order; stream bits are LSB-first, so the table index is the reversed code
        uint32_t code = 0;
        int k = 0;
        for (int l = 1; l <= fast_bits; l++) {
            for (int c = 0; c < h.count[l]; c++, k++) {
                const uint32_t r = inflate_rev(code + (uint32_t)c, l);
                for (uint32_t f = r; f < (1u << fast_bits); f += 1u << l) fast[f] = (uint16_t)((h.sym[k] << 4) | l);
            }
            code = (code + h.count[l]) << 1;
        }
    }
    return 0;
}

struct InflateState {
    const uint8_t *in; uint32_t clen, inpos;
    uint8_t *out; uint32_t isize, outpos;
    uint64_t bits; int nbits;
    int mode;        // 0: next block header, 1: inside a Huffman block, 2: stream complete
    bool last;
};

SQ_HD void inflate_init(InflateState &s, const uint8_t *in, uint32_t clen, uint8_t *out, uint32_t isize) {
    s.in = in; s.clen = clen; s.inpos = 0; s.out = out; s.isize = isize; s.outpos = 0; s.bits = 0; s.nbits = 0; s.mode = 0; s.last = false;
}
SQ_HD void inflate_fill(InflateState &s) {  // past the payload the stream reads as zero bits; inflate_overrun() tells
    while (s.nbits <= 56) { s.bits |= (uint64_t)(s.inpos < s.clen ? s.in[s.inpos] : 0) << s.nbits; s.inpos++; s.nbits += 8; }
}
SQ_HD bool inflate_overrun(const InflateState &s) { return (uint64_t)s.inpos * 8 - (uint64_t)s.nbits > (uint64_t)s.clen * 8; }
SQ_HD uint32_t inflate_take(InflateState &s, int n) { inflate_fill(s); const uint32_t v = (uint32_t)(s.bits & ((1ull << n) - 1)); s.bits >>= n; s.nbits -= n; return v; }

// one symbol of `h`; -1 when the bits are no code of it
SQ_HD int inflate_decode(InflateState &s, const HuffCode &h, const uint16_t *fast, int fast_bits) {
    inflate_fill(s);
    if (fast) {
        const uint16_t e = fast[s.bits & ((1u << fast_bits) - 1)];
        if (e) { const int l = e & 15; s.bits >>= l; s.nbits -= l; return e >> 4; }
    }
    int code = 0, first = 0, index = 0;
    for (int l = 1; l < 16; l++) {
        code |= (int)(s.bits & 1); s.bits >>= 1; s.nbits--;
        const int count = h.count[l];
        if (code - count < first) return h.sym[index + (code - first)];
        index += count; first += count; first <<= 1; code <<= 1;
    }
    return -1;
}

SQ_HD int inflate_header(InflateState &s, InflateTables &t) {  // a dynamic block's code lengths -> tables; 0 or -1
    const int nlen = (int)inflate_take(s, 5) + 257, ndist = (int)inflate_take(s, 5) + 1, ncode = (int)inflate_take(s, 4) + 4;
    if (nlen > 286 || ndist > 30) return -1;
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint8_t cl[19];
    for (int i = 0; i < 19; i++) cl[i] = 0;
    for (int i = 0; i < ncode; i++) cl[order[i]] = (uint8_t)inflate_take(s, 3);
    if (inflate_build(t.dist, cl, 19, nullptr, 0, 0)) return -1;
    int have = 0;
    while (have < nlen + ndist) {
        const int sym = inflate_decode(s, t.dist, nullptr, 0);
        if (sym < 0) return -1;
        if (sym < 16) { t.lens[have++] = (uint8_t)sym; continue; }
        int rep; uint8_t v = 0;
        if (sym == 16) { if (have == 0) return -1; v = t.lens[have - 1]; rep = 3 + (int)inflate_take(s, 2); }
        else if (sym == 17) rep = 3 + (int)inflate_take(s, 3);
        else rep = 11 + (int)inflate_take(s, 7);
        if (have + rep > nlen + ndist) return -1;
        while (rep--) t.lens[have++] = v;
    }
    if (t.lens[256] == 0) return -1;
    if (inflate_build(t.lit, t.lens, nlen, t.lfast, kInflLitBits, 1)) return -1;
    if (inflate_build(t.dist, t.lens + nlen, ndist, t.dfast, kInflDistBits, 2)) return -1;
    return 0;
}

SQ_HD void inflate_fixed(InflateTables &t) {
    for (int i = 0; i < 144; i++) t.lens[i] = 8;
    for (int i = 144; i < 256; i++) t.lens[i] = 9;
    for (int i = 256; i < 280; i++) t.lens[i] = 7;
    for (int i = 280; i < 288; i++) t.lens[i] = 8;
    inflate_build(t.lit, t.lens, 288, t.lfast, kInflLitBits, 1);
    for (int i = 0; i < 32; i++) t.lens[i] = 5;
    inflate_build(t.dist, t.lens, 32, t.dfast, kInflDistBits, 2);
}

// Runs the member until it ends with exactly ISIZE bytes (returns 0), fails (-1) or meets a match of >= warp_min bytes (returns 1: the caller copies
// out[*dst + i] = out[*dst - *dist + i % *dist] for i < *len; outpos is already past it).  Literals and shorter matches are
// written here.
SQ_HD int inflate_step(InflateState &s, InflateTables &t, uint32_t warp_min, uint32_t *dst, uint32_t *len_out, uint32_t *dist_out) {
    for (;;) {
        if (inflate_overrun(s)) return -1;
        if (s.mode == 2) return s.outpos == s.isize ? 0 : -1;  // the member must fill exactly ISIZE bytes
        if (s.mode == 0) {
            if (s.last) { s.mode = 2; continue; }
            s.last = inflate_take(s, 1) != 0;
            const uint32_t type = inflate_take(s, 2);
            if (type == 0) {
                const int drop = s.nbits & 7;  // to the byte boundary
                s.bits >>= drop; s.nbits -= drop;
                const uint32_t ln = inflate_take(s, 16), nl = inflate_take(s, 16);
                if (ln != (~nl & 0xFFFFu)) return -1;
                if (inflate_overrun(s)) return -1;
                for (uint32_t i = 0; i < ln; i++) {  // the bit buffer holds whole bytes here
                    const uint32_t c = inflate_take(s, 8);
                    if (s.outpos >= s.isize) return -1;
                    s.out[s.outpos++] = (uint8_t)c;
                }
                continue;
            }
            if (type == 1) inflate_fixed(t);
            else if (type == 2) { if (inflate_header(s, t)) return -1; }
            else return -1;
            s.mode = 1;
        }
        const int sym = inflate_decode(s, t.lit, t.lfast, kInflLitBits);
        if (sym < 0 || sym > 285) return -1;
        if (sym < 256) {
            if (s.outpos >= s.isize) return -1;
            s.out[s.outpos++] = (uint8_t)sym;
            continue;
        }
        if (sym == 256) { s.mode = 0; continue; }
        // RFC 1951 3.2.5: length symbols 257-264 and distance symbols 0-3 carry no extra bits, then every four (two) symbols one more
        const int ls = sym - 257;
        const int le = ls < 8 || ls == 28 ? 0 : (ls - 4) >> 2;
        const uint32_t len = (ls < 8 ? 3u + ls : ls == 28 ? 258u : ((4u + (ls & 3)) << le) + 3u) + inflate_take(s, le);
        const int ds = inflate_decode(s, t.dist, t.dfast, kInflDistBits);
        if (ds < 0 || ds > 29) return -1;
        const int de = ds < 4 ? 0 : (ds - 2) >> 1;
        const uint32_t dist = (ds < 4 ? 1u + ds : ((2u + (ds & 1)) << de) + 1u) + inflate_take(s, de);
        if (dist > s.outpos || len > s.isize - s.outpos) return -1;
        if (inflate_overrun(s)) return -1;
        if (len >= warp_min) { *dst = s.outpos; *len_out = len; *dist_out = dist; s.outpos += len; return 1; }
        for (uint32_t i = 0; i < len; i++) s.out[s.outpos + i] = s.out[s.outpos - dist + i];
        s.outpos += len;
    }
}

// CRC32 (the gzip polynomial) and zlib's crc32_combine, so that 32 lanes can each sum a slice of a member.
SQ_HD uint32_t crc32_multmodp(uint32_t a, uint32_t b) {  // a * b modulo the CRC polynomial (reflected)
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
SQ_HD uint32_t crc32_entry(uint32_t n) {  // entry n of the byte-wise CRC table
    uint32_t c = n;
    for (int k = 0; k < 8; k++) c = c & 1 ? 0xEDB88320u ^ (c >> 1) : c >> 1;
    return c;
}
SQ_HD void crc32_x2n(uint32_t *x2n32) {  // x2n32[k] = x^(2^k) modulo the polynomial
    uint32_t p = 1u << 30;  // x^1
    x2n32[0] = p;
    for (int n = 1; n < 32; n++) x2n32[n] = p = crc32_multmodp(p, p);
}
SQ_HD uint32_t crc32_update(const uint32_t *table256, uint32_t crc, const uint8_t *p, uint32_t n) {
    crc = ~crc;
    for (uint32_t i = 0; i < n; i++) crc = table256[(crc ^ p[i]) & 0xFF] ^ (crc >> 8);
    return ~crc;
}
// crc of A||B from crc(A), crc(B) and |B|
SQ_HD uint32_t crc32_combine(const uint32_t *x2n32, uint32_t crc1, uint32_t crc2, uint32_t len2) {
    uint32_t p = 1u << 31;  // x^0
    int k = 3;
    for (uint32_t n = len2; n; n >>= 1, k++) if (n & 1) p = crc32_multmodp(x2n32[k & 31], p);
    return crc32_multmodp(p, crc1) ^ crc2;
}

}  // namespace sq
#endif
