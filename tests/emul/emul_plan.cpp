// TEST TOOLING — the shard planner of the resident batch (squid_b200/csrc/sq_plan.cuh) stepped on the CPU.
//
//     emul_plan <dir> <max_shards>
//
// <dir> holds the arrays of an sqg_batch (batch_<field>.bin) and of an sqg_chimeric (chim_<field>.bin) as raw little-endian
// files, and config.bin = int32 {min_mapq, max_lowphred_len, concord_dist_pos, concord_dist_idx, read_len, n_ref}.  The class
// bytes come from classify_record over the whole stream, the groups from the host pre-pass, the three exclusive scans from
// plain loops; then the SAME plan_candidate / plan_greedy the library runs.  Prints the cuts for 1..max_shards shards, one
// line each.  Not a product path: the library runs these rules in k_plan_cands and never links this file.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "host/prepass.h"
#include "sq_plan.cuh"

using namespace sq;

static std::string dir;
template <class T> static std::vector<T> load(const std::string &name) {
    std::vector<T> v;
    FILE *f = fopen((dir + "/" + name + ".bin").c_str(), "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", name.c_str()); exit(2); }
    T x;
    while (fread(&x, sizeof(T), 1, f) == 1) v.push_back(x);
    fclose(f);
    if (v.empty()) v.push_back(T());  // (an empty array still needs a valid pointer)
    return v;
}

int main(int argc, char **argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s dir max_shards\n", argv[0]); return 2; }
    dir = argv[1];
    const int32_t max_shards = atoi(argv[2]);
    const std::vector<int32_t> cfg = load<int32_t>("config");
    auto ref_id = load<int32_t>("batch_ref_id"), pos = load<int32_t>("batch_pos"), mate_ref_id = load<int32_t>("batch_mate_ref_id"),
         mate_pos = load<int32_t>("batch_mate_pos"), end_pos = load<int32_t>("batch_end_pos"), blk_ref_pos = load<int32_t>("batch_blk_ref_pos"),
         blk_match_ref = load<int32_t>("batch_blk_match_ref");
    auto flag = load<uint16_t>("batch_flag"), total_len = load<uint16_t>("batch_total_len"), lowphred_run = load<uint16_t>("batch_lowphred_run"),
         blk_read_pos = load<uint16_t>("batch_blk_read_pos"), blk_match_read = load<uint16_t>("batch_blk_match_read");
    auto mapq = load<uint8_t>("batch_mapq"), aux = load<uint8_t>("batch_aux");
    auto blk_off = load<uint32_t>("batch_blk_off");
    DevBatch b;
    b.n_rec = (int64_t)blk_off.size() - 1; b.n_blk = blk_off.back();
    b.ref_id = ref_id.data(); b.pos = pos.data(); b.mate_ref_id = mate_ref_id.data(); b.mate_pos = mate_pos.data(); b.end_pos = end_pos.data();
    b.flag = flag.data(); b.total_len = total_len.data(); b.lowphred_run = lowphred_run.data(); b.mapq = mapq.data(); b.aux = aux.data();
    b.blk_off = blk_off.data(); b.blk_ref_pos = blk_ref_pos.data(); b.blk_match_ref = blk_match_ref.data();
    b.blk_read_pos = blk_read_pos.data(); b.blk_match_read = blk_match_read.data();
    Params p;
    p.min_mapq = cfg[0]; p.max_lowphred_len = cfg[1]; p.concord_dist_pos = cfg[2]; p.concord_dist_idx = cfg[3]; p.read_len = cfg[4]; p.n_ref = cfg[5];

    auto read_off = load<uint32_t>("chim_read_off");
    auto n_first = load<uint16_t>("chim_n_first");
    auto first_total = load<int32_t>("chim_first_total_len"), second_total = load<int32_t>("chim_second_total_len");
    auto first_low = load<uint8_t>("chim_first_lowphred"), second_low = load<uint8_t>("chim_second_lowphred"), multi = load<uint8_t>("chim_multi_filter");
    auto c_ref_id = load<int32_t>("chim_blk_ref_id"), c_ref_pos = load<int32_t>("chim_blk_ref_pos"), c_read_pos = load<int32_t>("chim_blk_read_pos"),
         c_match_ref = load<int32_t>("chim_blk_match_ref"), c_match_read = load<int32_t>("chim_blk_match_read");
    auto c_rev = load<uint8_t>("chim_blk_is_reverse");
    sqg_chimeric chim;
    chim.n_reads = (int64_t)read_off.size() - 1; chim.n_blk = chim.n_reads > 0 ? read_off.back() : 0;
    chim.read_off = read_off.data(); chim.n_first = n_first.data(); chim.first_total_len = first_total.data(); chim.second_total_len = second_total.data();
    chim.first_lowphred = first_low.data(); chim.second_lowphred = second_low.data(); chim.multi_filter = multi.data();
    chim.blk_ref_id = c_ref_id.data(); chim.blk_ref_pos = c_ref_pos.data(); chim.blk_read_pos = c_read_pos.data();
    chim.blk_match_ref = c_match_ref.data(); chim.blk_match_read = c_match_read.data(); chim.blk_is_reverse = c_rev.data();
    sqh::ChimPrepass pre;
    sqh::chimeric_prepass(chim, p.n_ref, p.read_len, pre);

    const int64_t n = b.n_rec;
    std::vector<uint8_t> cls((size_t)n);
    for (int64_t r = 0, prev = -1; r < n; r++) {  // the classification pass: the previous gate-passing record of the whole stream
        cls[(size_t)r] = classify_record(b, p, r, prev).cls;
        if (cls[(size_t)r] & CLS_GATE) prev = r;
    }
    std::vector<int32_t> keep_excl((size_t)n), upd_excl((size_t)n);
    std::vector<uint64_t> before((size_t)n);
    uint64_t run = 0;
    int32_t last_keep = -1, last_upd = -1;
    for (int64_t r = 0; r < n; r++) {
        before[(size_t)r] = run; keep_excl[(size_t)r] = last_keep; upd_excl[(size_t)r] = last_upd;
        run = std::max(run, plan_reach_key(b.ref_id[r], plan_reach(b, r)));
        if (cls[(size_t)r] & CLS_KEEP) last_keep = (int32_t)r;
        if (plan_updates_other(cls[(size_t)r], b.flag[r])) last_upd = (int32_t)r;
    }
    // SQ_EMUL_PLAN_NO_GROUPS=1: plan as if there were no discordant group (shows a test that condition C decides its cuts)
    const int32_t nG = getenv("SQ_EMUL_PLAN_NO_GROUPS") ? 0 : (int32_t)pre.groups.size();
    std::vector<uint64_t> cand;
    for (int64_t c = 0; c < n; c++) {
        const int64_t m = plan_candidate(b, p, cls[(size_t)c], before[(size_t)c], keep_excl.data(), upd_excl.data(), pre.groups.data(), pre.disc.data(), nG, c);
        if (m >= 0) cand.push_back(plan_pack(c, m));
    }
    fprintf(stderr, "emul_plan: %lld records, %d groups, %zu candidates\n", (long long)n, nG, cand.size());
    std::vector<int64_t> cuts((size_t)max_shards + 1);
    for (int32_t ns = 1; ns <= max_shards; ns++) {
        const int32_t k = plan_greedy(cand.data(), (int64_t)cand.size(), n, ns, cuts.data());
        for (int32_t i = 0; i <= k; i++) printf(i ? " %lld" : "%lld", (long long)cuts[(size_t)i]);
        printf("\n");
    }
    return 0;
}
