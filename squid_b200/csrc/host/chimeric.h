// Host twin of BuildChimericSBamRecord (src/ReadRec.cpp:329-413) and of the SoA packing step that
// north_star places on the host.  Inputs are SQMB tables (include/sqmb_format.h).
#ifndef SQUID_B200_HOST_CHIMERIC_H
#define SQUID_B200_HOST_CHIMERIC_H
#include <cstdint>
#include <functional>
#include <string>
#include <unordered_set>
#include <vector>
#include "readrec.h"
#include "sqmb_format.h"
#include "squid_b200.h"

namespace sqh {

Alignment alignment_at(const SqmbView &v, uint64_t r);
std::string name_at(const SqmbView &v, uint64_t r);

// An alignment-level input (what BamReader::GetNextAlignment yields, in file order): SQMB tables and decoded BAM files
// (host/bam.h) both present themselves through this.
struct AlnSource {
    uint64_t n_rec = 0;
    std::function<Alignment(uint64_t)> at;
    std::function<std::string(uint64_t)> name;   // BamAlignment::Name, raw
    std::function<size_t(uint64_t, char *)> name_into;  // the same into a caller buffer of >= 256 bytes (no allocation); returns the length
};
AlnSource source_of(const SqmbView &v);
void load_chimeric(const AlnSource &chim, HostConfig &cfg, std::vector<Read> &out);

// Chimrecord: reads grouped by Qname, mates merged, blocks sorted by read position, sorted by front
// block, PCR duplicates removed; sets cfg.read_len (median of the first five totals).
void load_chimeric(const SqmbView &chim, HostConfig &cfg, std::vector<Read> &out);

// Owning storage behind a sqg_batch.
struct PackedBatch {
    std::vector<int32_t> ref_id, pos, mate_ref_id, mate_pos, end_pos;
    std::vector<uint16_t> flag, total_len, lowphred_run;
    std::vector<uint8_t> mapq, aux;
    std::vector<uint32_t> blk_off;
    std::vector<int32_t> blk_ref_pos, blk_match_ref;
    std::vector<uint16_t> blk_read_pos, blk_match_read;
    sqg_batch view() const;
};
// Twin of the per-record decode the reference repeats in each of its three BAM passes
// (ReadRec_t ctor + tag/ChimName probes, SegmentGraph.cpp:297-304).  `chim_names` holds the
// suffix-stripped Qnames of Chimrecord; the gate compares the RAW record name against them
// (SURVEY.md App. A-3), so a "/1" or "/2" suffixed name never matches.
// Why the packer refuses record r (sq::packer_limit `limit`, 1 or 2), in the words every front end reports.
std::string packer_refusal(uint64_t r, int limit, int64_t total_len);
int pack_concordant(const SqmbView &conc, const HostConfig &cfg, const std::unordered_set<std::string> &chim_names, PackedBatch &out, std::string &err);
int pack_concordant(const AlnSource &conc, const HostConfig &cfg, const std::unordered_set<std::string> &chim_names, PackedBatch &out, std::string &err);

// Owning storage behind a sqg_chimeric.
struct PackedChimeric {
    std::vector<uint32_t> read_off;
    std::vector<uint16_t> n_first;
    std::vector<int32_t> first_total, second_total;
    std::vector<uint8_t> first_low, second_low, multi_filter;
    std::vector<int32_t> blk_ref_id, blk_ref_pos, blk_read_pos, blk_match_ref, blk_match_read;
    std::vector<uint8_t> blk_is_reverse;
    sqg_chimeric view();
    void from_reads(const std::vector<Read> &reads);
    void to_reads(std::vector<Read> &reads) const;  // copies (trimmed) blocks back
};

}  // namespace sqh
#endif
