// BGZF / BAM front end of the host packer (SURVEY.md 8f row 1): replaces BamTools' BamReader::Open / GetHeader /
// GetNextAlignment on the path (reference call sites: src/ReadRec.cpp:271-279, 340-343; src/SegmentGraph.cpp:293-296,
// 1570-1577, 3126-3129).  The whole file is inflated once, on all cores (BGZF blocks are independent deflate streams),
// and decoded into a struct-of-arrays table that feeds load_chimeric / pack_concordant through AlnSource -- one decode for
// all three phases instead of the reference's three passes.
// Follows the SAM/BAM specification (BGZF: gzip members with a "BC" extra subfield; BAM: little-endian records).  BamTools
// behaviour kept: Qualities = phred + 33 as characters, QueryBases from the 4-bit codes "=ACMGRSVTWYHKDBN", HasTag /
// GetTag("IH") accept any integer-typed tag (SURVEY.md 8c).
#ifndef SQUID_B200_HOST_BAM_H
#define SQUID_B200_HOST_BAM_H
#include <cstdint>
#include <cstdlib>
#include <string>
#include <vector>
#include "chimeric.h"

namespace sqh {

// uninitialised storage (std::vector would zero-fill hundreds of megabytes that are overwritten right away)
template <class T> struct RawBuf {
    T *p = nullptr; size_t n = 0;
    RawBuf() = default;
    RawBuf(const RawBuf &) = delete;
    RawBuf &operator=(const RawBuf &) = delete;
    RawBuf(RawBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    RawBuf &operator=(RawBuf &&o) noexcept { if (this != &o) { free(p); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
    ~RawBuf() { free(p); }
    bool resize(size_t m) { free(p); p = m ? (T *)malloc(m * sizeof(T)) : nullptr; n = p ? m : 0; return m == 0 || p != nullptr; }
    T *data() { return p; }
    const T *data() const { return p; }
    size_t size() const { return n; }
};

struct BamTable {
    std::vector<std::string> ref_name;
    std::vector<int32_t> ref_len;
    // one entry per alignment record, file order
    std::vector<int32_t> ref_id, pos, mate_ref_id, mate_pos, ih;
    std::vector<uint16_t> flag;
    std::vector<uint8_t> mapq, tags;            // tags: bit0 XA present, bit1 IH present
    std::vector<uint64_t> name_off, cigar_off, seq_off;   // n + 1 entries each
    RawBuf<char> names, seq, qual;              // seq / qual as BamTools strings
    RawBuf<uint32_t> cigar;
    bool walked_per_member = false;             // the record boundaries were found member by member (proven, see bam.cpp)
    uint64_t n_rec() const { return ref_id.size(); }
    // Reads a BGZF-compressed BAM (or an uncompressed BAM stream).  threads <= 0: all cores.
    bool open(const std::string &path, std::string &err, int threads = 0);
    AlnSource source() const;
};

// One BGZF member: deflate payload [cdata, cdata + clen) of the file inflates to `isize` bytes at offset `off` of the stream.
struct BgzfMember { size_t cdata, clen, off; uint32_t isize, crc; };
// Locates every member of a BGZF file by its BC subfield (shared by the host inflater and the device loader, sqg_load_concordant_bam).
bool bgzf_parse_members(const uint8_t *data, size_t len, std::vector<BgzfMember> &mem, std::string &err);
// BAM header of an inflated stream prefix: 1 = parsed (`end` = offset of the first record), 0 = the prefix is too short, -1 = malformed.
int bam_parse_header(const uint8_t *b, size_t n, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len, size_t &end, std::string &err);
// The header of a mapped file: members inflated with zlib one by one until it is complete (mem = nullptr: an uncompressed stream).
bool bam_read_header(const uint8_t *f, size_t flen, const std::vector<BgzfMember> *mem, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len,
                     size_t &end, std::string &err);
// bam_read_header() of a file on disk (BGZF or uncompressed)
bool bam_read_header_file(const std::string &path, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len, std::string &err);

// The plan of the device loader (sqg_load_concordant_bam), which its CPU stepping (tests/emul/emul_bam.cpp) runs as well.
constexpr uint32_t kRawMember = 0xFFFFFFFFu;  // crc of a pseudo-member of an uncompressed stream: copied, not inflated
// The members a mapped file is uploaded in: its BGZF members with data (EOF markers dropped), or for an uncompressed stream (raw)
// 64 KiB pieces that stand in for members (segment starts of the record walk).
bool bam_loader_members(const uint8_t *f, size_t len, bool raw, std::vector<BgzfMember> &mem, std::string &err);
// Windows of whole members, about win_bytes inflated bytes each, the first one holding the whole header: window w is the members
// [cut[w], cut[w + 1]).
std::vector<size_t> bam_window_cuts(const std::vector<BgzfMember> &mem, int64_t win_bytes, size_t hdr_end);
// Walk segments of window w in its buffer, behind the `carry` bytes of the previous window's tail: the first record start (the
// end of the header in window 0) and every member start past it.
std::vector<int64_t> bam_window_segments(const std::vector<BgzfMember> &mem, const std::vector<size_t> &cut, size_t w, int64_t carry, size_t hdr_end);
// ChimName as the loader probes it (sq_bam.cuh NameSet): open addressing over the names' hashes, duplicates dropped, each slot with
// its name's length (-1: empty) and offset into the blob for the exact compare.
struct NameTable { std::vector<uint64_t> hash; std::vector<int32_t> len; std::vector<int64_t> off; };
NameTable bam_name_table(const char *blob, const int64_t *name_off, int64_t n);

// inflate a whole BGZF file (concatenated gzip members with BSIZE) on `threads` threads
// (`member_off`, optional: offset of every member's data in `out`, plus the total as the last entry)
bool bgzf_inflate_all(const uint8_t *data, size_t len, RawBuf<uint8_t> &out, std::string &err, int threads, std::vector<size_t> *member_off = nullptr);

}  // namespace sqh
#endif
