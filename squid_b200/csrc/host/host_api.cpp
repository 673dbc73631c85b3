// C entry points of the host twin (include/squid_b200_host.h).
#include <cstdio>
#include <cstring>
#include <new>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <unordered_set>

#include "bam.h"
#include "chimeric.h"
#include "squid_b200_host.h"

struct sqh_case {
    sqh::HostConfig cfg;
    SqmbView conc, chim;
    sqh::BamTable bconc, bchim;
    std::vector<sqh::Read> reads;
    sqh::PackedBatch batch;
    sqh::PackedChimeric pchim;
    sqg_batch bview;
    sqg_chimeric cview;
    sqg_config gcfg;
    std::vector<int32_t> ref_len;
    std::string chim_blob;               // the ChimName list the packer probes, as a blob with offsets (sqh_case_chim_names)
    std::vector<int64_t> chim_off;
    void set_chim_names(const std::unordered_set<std::string> &names) {
        chim_blob.clear(); chim_off.assign(1, 0);
        for (const std::string &s : names) { chim_blob += s; chim_off.push_back((int64_t)chim_blob.size()); }
    }
};

extern "C" {
void sqh_default_options(sqh_options *o) {
    if (!o) return;
    o->phred33 = 1; o->max_lowphred_len = 10; o->min_phred = 4; o->min_mapq = -1; o->concord_dist_pos = 50000; o->concord_dist_idx = 20;
}

namespace {
struct HostLaps {  // SQH_TIMING=1: wall-clock laps of the host front end, to stderr
    bool on; std::chrono::steady_clock::time_point t0;
    HostLaps() : on(getenv("SQH_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void operator()(const char *what) {
        if (!on) return;
        const auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[sqh] %-28s %8.3f ms\n", what, 1e3 * std::chrono::duration<double>(t - t0).count());
        t0 = t;
    }
};
}  // namespace
static int open_case(bool bam, bool conc_header_only, const char *conc_path, const char *chim_path, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen) {
    auto fail = [&](int code, const std::string &m) { if (errbuf && errlen > 0) snprintf(errbuf, errlen, "%s", m.c_str()); return code; };
    if (!conc_path || !chim_path || !out) return fail(SQG_EINVAL, "null argument");
    *out = nullptr;
    sqh_case *c = new (std::nothrow) sqh_case();
    if (!c) return fail(SQG_ENOMEM, "out of memory");
    sqh_options o;
    if (opt) o = *opt; else sqh_default_options(&o);
    c->cfg.phred33 = o.phred33 != 0; c->cfg.max_lowphred_len = o.max_lowphred_len; c->cfg.min_phred = o.min_phred;
    c->cfg.min_mapq = o.min_mapq < 0 ? 255 : o.min_mapq; c->cfg.concord_dist_pos = o.concord_dist_pos; c->cfg.concord_dist_idx = o.concord_dist_idx;
    sqh::AlnSource sconc, schim;
    if (bam) {  // BGZF/BAM front end (host/bam.h): BamReader::Open + GetHeader + GetNextAlignment of the reference
        std::string e;
        if (conc_header_only) {  // the records are decoded on the device (sqg_load_concordant_bam): an empty concordant source
            std::vector<std::string> names;
            if (!sqh::bam_read_header_file(conc_path, names, c->ref_len, e)) { delete c; return fail(SQG_EINVAL, e); }
        } else if (!c->bconc.open(conc_path, e)) { delete c; return fail(SQG_EINVAL, e); }
        if (!c->bchim.open(chim_path, e)) { delete c; return fail(SQG_EINVAL, e); }
        if (!conc_header_only) { c->ref_len = c->bconc.ref_len; sconc = c->bconc.source(); }  // BuildRefName reads the header of the concordant BAM (ReadRec.cpp:267-283)
        schim = c->bchim.source();
    } else {
        if (!c->conc.open(conc_path)) { delete c; return fail(SQG_EINVAL, std::string("cannot open ") + conc_path); }
        if (!c->chim.open(chim_path)) { delete c; return fail(SQG_EINVAL, std::string("cannot open ") + chim_path); }
        c->ref_len.assign(c->conc.ref_len, c->conc.ref_len + c->conc.n_ref);
        sconc = sqh::source_of(c->conc); schim = sqh::source_of(c->chim);
    }
    HostLaps lap;
    lap("open files");
    sqh::load_chimeric(schim, c->cfg, c->reads);
    lap("chimeric loader");
    std::unordered_set<std::string> names;
    names.insert("");  // ChimName is pre-sized with empty strings before the names are appended (SegmentGraph.cpp:196-198)
    for (const sqh::Read &r : c->reads) names.insert(r.qname);
    c->set_chim_names(names);
    lap("ChimName set");
    std::string err;
    int rc = sqh::pack_concordant(sconc, c->cfg, names, c->batch, err);
    if (rc) { delete c; return fail(rc, err); }
    lap("decode + pack concordant");
    c->pchim.from_reads(c->reads);
    lap("pack chimeric");
    c->bview = c->batch.view();
    c->cview = c->pchim.view();
    c->gcfg.using_star = 1; c->gcfg.max_lowphred_len = c->cfg.max_lowphred_len; c->gcfg.min_mapq = c->cfg.min_mapq;
    c->gcfg.concord_dist_pos = c->cfg.concord_dist_pos; c->gcfg.concord_dist_idx = c->cfg.concord_dist_idx; c->gcfg.read_len = c->cfg.read_len;
    *out = c;
    return SQG_OK;
}
int sqh_open_case(const char *conc_path, const char *chim_path, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen) {
    return open_case(false, false, conc_path, chim_path, opt, out, errbuf, errlen);
}
int sqh_open_bam_case(const char *conc_bam, const char *chim_bam, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen) {
    return open_case(true, false, conc_bam, chim_bam, opt, out, errbuf, errlen);
}
int sqh_open_bam_chimeric(const char *conc_bam, const char *chim_bam, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen) {
    return open_case(true, true, conc_bam, chim_bam, opt, out, errbuf, errlen);
}
// The concordant BAM alone, for a caller that already holds Chimrecord (the binding of INTEGRATION.md): ChimName is built from
// the Qnames it passes (SegmentGraph.cpp:196-201), the chimeric side of the case stays empty.
int sqh_open_concordant(const char *conc_path, const char *const *chim_qnames, int64_t n_names, const sqh_options *opt, sqh_case **out, char *errbuf, int errlen) {
    auto fail = [&](int code, const std::string &m) { if (errbuf && errlen > 0) snprintf(errbuf, errlen, "%s", m.c_str()); return code; };
    if (!conc_path || !out || n_names < 0 || (n_names > 0 && !chim_qnames)) return fail(SQG_EINVAL, "null argument");
    *out = nullptr;
    sqh_case *c = new (std::nothrow) sqh_case();
    if (!c) return fail(SQG_ENOMEM, "out of memory");
    sqh_options o;
    if (opt) o = *opt; else sqh_default_options(&o);
    c->cfg.phred33 = o.phred33 != 0; c->cfg.max_lowphred_len = o.max_lowphred_len; c->cfg.min_phred = o.min_phred;
    c->cfg.min_mapq = o.min_mapq < 0 ? 255 : o.min_mapq; c->cfg.concord_dist_pos = o.concord_dist_pos; c->cfg.concord_dist_idx = o.concord_dist_idx;
    if (!c->conc.open(conc_path)) { delete c; return fail(SQG_EINVAL, std::string("cannot open ") + conc_path); }
    c->ref_len.assign(c->conc.ref_len, c->conc.ref_len + c->conc.n_ref);
    std::unordered_set<std::string> names;
    names.insert("");  // ChimName is pre-sized with empty strings before the names are appended (SegmentGraph.cpp:196-198)
    for (int64_t i = 0; i < n_names; i++) names.insert(chim_qnames[i] ? chim_qnames[i] : "");
    c->set_chim_names(names);
    std::string err;
    const int rc = sqh::pack_concordant(sqh::source_of(c->conc), c->cfg, names, c->batch, err);
    if (rc) { delete c; return fail(rc, err); }
    c->pchim.from_reads(c->reads);
    c->bview = c->batch.view();
    c->cview = c->pchim.view();
    c->gcfg.using_star = 1; c->gcfg.max_lowphred_len = c->cfg.max_lowphred_len; c->gcfg.min_mapq = c->cfg.min_mapq;
    c->gcfg.concord_dist_pos = c->cfg.concord_dist_pos; c->gcfg.concord_dist_idx = c->cfg.concord_dist_idx; c->gcfg.read_len = 0;
    *out = c;
    return SQG_OK;
}
void sqh_close_case(sqh_case *c) { delete c; }
const sqg_batch *sqh_case_batch(const sqh_case *c) { return c ? &c->bview : nullptr; }
sqg_chimeric *sqh_case_chimeric(sqh_case *c) { return c ? &c->cview : nullptr; }
const sqg_config *sqh_case_config(const sqh_case *c) { return c ? &c->gcfg : nullptr; }
int sqh_case_chim_names(const sqh_case *c, const char **blob, const int64_t **off, int64_t *n) {
    if (!c || !blob || !off || !n) return SQG_EINVAL;
    *blob = c->chim_blob.data(); *off = c->chim_off.data(); *n = (int64_t)c->chim_off.size() - 1;
    return SQG_OK;
}
int32_t sqh_case_n_ref(const sqh_case *c) { return c ? (int32_t)c->ref_len.size() : 0; }
const int32_t *sqh_case_ref_len(const sqh_case *c) { return c ? c->ref_len.data() : nullptr; }
int32_t sqh_case_blocks(const sqh_case *c, int64_t r, int32_t *out4, int32_t max_blocks, int32_t *total_len, int32_t *lowphred_run) {
    if (!c || r < 0 || (size_t)r + 1 >= c->batch.blk_off.size()) return -1;
    const uint32_t o = c->batch.blk_off[r], n = c->batch.blk_off[r + 1] - o;
    for (uint32_t k = 0; k < n && (int32_t)k < max_blocks; k++) {
        out4[4 * k] = c->batch.blk_ref_pos[o + k]; out4[4 * k + 1] = c->batch.blk_match_ref[o + k];
        out4[4 * k + 2] = c->batch.blk_read_pos[o + k]; out4[4 * k + 3] = c->batch.blk_match_read[o + k];
    }
    if (total_len) *total_len = c->batch.total_len[r];
    if (lowphred_run) *lowphred_run = c->batch.lowphred_run[r];
    return (int32_t)n;
}
}
