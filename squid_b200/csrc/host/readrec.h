// Host twin of SQUID's read model (reference: src/SingleBamRec.h, src/ReadRec.{h,cpp}).
// Same vocabulary (aligned block = SingleBamRec, read pair = ReadRec, Chimrecord), our own code.
// Everything here is host-side string/CIGAR work that north_star keeps on the CPU: the only place
// that touches names, bases, qualities and CIGARs.  Its products are the SoA batches of
// include/squid_b200.h.
#ifndef SQUID_B200_HOST_READREC_H
#define SQUID_B200_HOST_READREC_H
#include <cstdint>
#include <string>
#include <vector>

namespace sqh {

struct HostConfig {              // src/Config.cpp:14-37
    bool using_star = true;
    bool phred33 = true;         // Phred_Type: true => offset 33 (Config.cpp:19, ReadRec.cpp:19-21)
    int max_lowphred_len = 10;   // -pl
    int min_phred = 4;           // -pm
    int min_mapq = 255;          // -mq (STAR default, Config.cpp:221-222)
    int concord_dist_pos = 50000;
    int concord_dist_idx = 20;
    int min_edge_weight = 5;
    double discordant_ratio = 8;
    int max_allowed_degree = 5;
    int read_len = 0;            // ReadLen, inferred by load_chimeric()
};

// One alignment line as the path sees it (the BamAlignment members listed in SURVEY.md §8c).
struct Alignment {
    int32_t ref_id = -1, pos = -1, mate_ref_id = -1, mate_pos = -1;
    uint16_t flag = 0;
    uint8_t mapq = 0;
    bool tag_xa = false, tag_ih = false;
    int ih_value = 0;
    const uint32_t *cigar = nullptr;  // BAM encoding len<<4|op
    uint32_t n_cigar = 0;
    // explicit bases/qualities (may be null => synthesised from the two summaries below)
    const char *seq = nullptr, *qual = nullptr;
    uint32_t l_seq = 0;
    uint16_t synth_lowrun = 0;  // qualities: `synth_lowrun` chars below any threshold, then high
    uint8_t synth_polya = 0;    // bit k: k-th aligned block all 'A'; bit 4+k: all 'T'
    bool is_mapped() const { return !(flag & 0x4); }
    bool is_mate_mapped() const { return !(flag & 0x8); }
    bool is_reverse() const { return flag & 0x10; }
    bool is_mate_reverse() const { return flag & 0x20; }
    bool is_first() const { return flag & 0x40; }
    bool is_second() const { return flag & 0x80; }
    bool is_dup() const { return flag & 0x400; }
    bool is_proper() const { return flag & 0x2; }
};

struct Block {  // SingleBamRec_t (src/SingleBamRec.h:25-61)
    int32_t ref_id, ref_pos, read_pos, match_ref, match_read;
    uint8_t mapq;
    bool is_reverse, is_first;
    bool before(const Block &o) const { return ref_id != o.ref_id ? ref_id < o.ref_id : ref_pos < o.ref_pos; }  // operator<
    bool after(const Block &o) const { return ref_id != o.ref_id ? ref_id > o.ref_id : ref_pos > o.ref_pos; }   // operator>
    bool same(const Block &o) const {
        return ref_id == o.ref_id && ref_pos == o.ref_pos && read_pos == o.read_pos && match_read == o.match_read &&
               match_ref == o.match_ref && is_reverse == o.is_reverse && is_first == o.is_first;
    }
};

// What ReadRec_t::ReadRec_t derives from one alignment (src/ReadRec.cpp:10-88).
struct Decoded {
    int total_len = 0;        // ReadRec.cpp:16-18
    int32_t end_pos = 0;      // BamTools GetEndPosition()
    int lowphred_run = 0;     // ReadRec.cpp:19-38 (longest run below threshold)
    std::vector<Block> blocks;  // CIGAR order, poly-A/T blocks removed, read_pos strand-flipped
};
void decode_alignment(const Alignment &a, const HostConfig &cfg, Decoded &out);

struct Read {  // ReadRec_t
    std::string qname;
    std::vector<Block> first, second;
    int first_total = 0, second_total = 0;
    bool first_low = false, second_low = false;
    bool multi_filter = false;

    void sort_by_read_pos();                       // ReadRec.cpp:143-146
    bool single_anchored() const;                  // :171-176
    bool end_discordant(bool first_mate) const;    // :178-209
    bool pair_discordant(bool check_ends = true) const;  // :211-228
    static bool equal(const Read &a, const Read &b);     // :119-141
    static bool front_smaller(const Read &a, const Read &b);  // :90-117
};

}  // namespace sqh
#endif
