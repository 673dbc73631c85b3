// Host-side chimeric pre-pass of BuildNode_STAR (SegmentGraph.cpp:196-264, 341-348): which blocks
// of Chimrecord are "discordant", the soft-clip positions of the rest (PartAlignPos), the sort of
// both, and the chaining of discordant blocks into groups.  Tie-order sensitive (the reference's
// unstable std::sort on (RefID,RefPos) is reproduced by running the same std::sort on the same
// sequence, SURVEY.md App. A-11).  The context runs the device twin (sq_prepass.cuh); this one
// serves the shard planner and the CPU stepping harness.
#ifndef SQUID_B200_HOST_PREPASS_H
#define SQUID_B200_HOST_PREPASS_H
#include <cstdint>
#include <vector>
#include "squid_b200.h"
#include "../sq_seed.cuh"

namespace sqh {
struct ChimPrepass {
    std::vector<sq::DiscBlock> disc;   // sorted bamdiscordant + one zeroed sentinel (size = n + 1)
    std::vector<int32_t> part_chr, part_pos;  // sorted PartAlignPos (incl. the n_ref leading (0,0) entries)
    std::vector<sq::Group> groups;
};
// element of the discordant-block sort: key = (RefID << 32 | RefPos), k = block index into the sqg_chimeric arrays
struct SortKey { uint64_t key; uint32_t k; };
// std::sort's permutation (libstdc++ introsort + final insertion sort, comparison on `key` only) on `threads` threads
void sort_keys_like_std(SortKey *first, SortKey *last, int threads);
// `c` = chimeric reads as passed over the C ABI.
void chimeric_prepass(const sqg_chimeric &c, int32_t n_ref, int32_t read_len, ChimPrepass &out);
}  // namespace sqh
#endif
