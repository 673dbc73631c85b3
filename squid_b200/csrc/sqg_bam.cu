// The concordant batch decoded from a BAM file on the device (sqg_load_concordant_bam).
#include <cub/cub.cuh>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cstring>

#include "sq_inflate.cuh"
#include "sq_bam.cuh"
#include "sqg_ctx.cuh"
#include "host/bam.h"

using namespace sq;

// ------------------------------------------------------------------------------------------------
// Concordant BAM decoded on the device (sq_inflate.cuh, sq_bam.cuh): the host maps the file, indexes the BGZF members and
// streams the compressed bytes through pinned staging; per window of whole members the device inflates (one member per warp),
// finds the record boundaries (speculative segment starts proven in parallel, repaired in rounds) and decodes the records into
// the resident batch.  Only the header is read on the host.
// ------------------------------------------------------------------------------------------------
constexpr int kInflWarps = 8;
constexpr size_t kBamStage = 32u << 20;  // bytes per pinned staging buffer
enum { BS_CHANGED = 0, BS_BAD, BS_AUXBAD, BS_ERRKEY, BS_SEQ, BS_INFL, BS_N };

__global__ void __launch_bounds__(kInflWarps * 32) k_bam_inflate(const BamMember *mem, int64_t n, const uint8_t *comp, uint8_t *win, int64_t *small) {
    __shared__ InflateTables tabs[kInflWarps];
    __shared__ uint32_t crc_tab[256], x2n[32];
    crc_tab[threadIdx.x] = crc32_entry(threadIdx.x);
    if (threadIdx.x == 0) crc32_x2n(x2n);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * kInflWarps + warp;
    if (k >= n) return;
    const BamMember m = mem[k];
    uint8_t *out = win + m.out;
    InflateState s;
    int rc = 0;
    if (lane == 0) inflate_init(s, comp + m.cdata, m.clen, out, m.isize);
    for (;;) {  // lane 0 decodes; a long match comes back to the warp, which copies it
        uint32_t dst = 0, len = 0, dist = 1;
        if (lane == 0) rc = inflate_step(s, tabs[warp], kInflWarpCopyMin, &dst, &len, &dist);
        __syncwarp();
        rc = __shfl_sync(0xFFFFFFFFu, rc, 0);
        if (rc != 1) break;
        dst = __shfl_sync(0xFFFFFFFFu, dst, 0); len = __shfl_sync(0xFFFFFFFFu, len, 0); dist = __shfl_sync(0xFFFFFFFFu, dist, 0);
        for (uint32_t i = lane; i < len; i += 32) out[dst + i] = out[dst - dist + i % dist];  // sources all lie before dst
        __syncwarp();
    }
    if (rc < 0) { if (lane == 0) atomicOr((unsigned long long *)&small[BS_INFL], 1ull); return; }
    __syncwarp();
    const uint32_t a = (uint32_t)((uint64_t)m.isize * lane / 32), b = (uint32_t)((uint64_t)m.isize * (lane + 1) / 32);
    uint32_t crc = crc32_update(crc_tab, 0, out + a, b - a), len = b - a;
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t c2 = __shfl_down_sync(0xFFFFFFFFu, crc, off), l2 = __shfl_down_sync(0xFFFFFFFFu, len, off);
        if ((lane & (2 * off - 1)) == 0) { crc = crc32_combine(x2n, crc, c2, l2); len += l2; }
    }
    if (lane == 0 && crc != m.crc) atomicOr((unsigned long long *)&small[BS_INFL], 2ull);
}

struct BamWin { const uint8_t *b; int64_t L, Lstream; int32_t n_ref; int64_t S; const int64_t *seg; };
SQ_HD int64_t bam_seg_end(const BamWin &w, int64_t k) { return k + 1 < w.S ? w.seg[k + 1] : w.L; }

__global__ void k_bam_spec(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    const int64_t e = bam_seg_end(w, k);
    const int64_t a = k == 0 ? w.seg[0] : bam_spec_start(w.b, w.seg[k], e, w.L, w.Lstream, w.n_ref);
    const SegWalk r = bam_walk(w.b, a, e, w.L, w.Lstream, nullptr);
    start[k] = a; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
}
__global__ void k_bam_mark(BamWin w, const int64_t *start, const int64_t *exit, int64_t *newstart, uint8_t *redo, int64_t *small) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    const bool r = k > 0 && exit[k - 1] != start[k];
    redo[k] = r;
    if (r) { newstart[k] = exit[k - 1]; atomicAdd((unsigned long long *)&small[BS_CHANGED], 1ull); }
}
__global__ void k_bam_rewalk(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad, const int64_t *newstart, const uint8_t *redo) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S || !redo[k]) return;
    const SegWalk r = bam_walk(w.b, newstart[k], bam_seg_end(w, k), w.L, w.Lstream, nullptr);
    start[k] = newstart[k]; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
}
__global__ void k_bam_sequential(BamWin w, int64_t *start, int64_t *exit, uint32_t *cnt, uint8_t *bad) {
    int64_t a = w.seg[0];
    for (int64_t k = 0; k < w.S; k++) {
        const SegWalk r = bam_walk(w.b, a, bam_seg_end(w, k), w.L, w.Lstream, nullptr);
        start[k] = a; exit[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
        a = r.exit;
    }
}
__global__ void k_bam_offsets(BamWin w, const int64_t *start, const uint8_t *bad, const uint32_t *base, int64_t *rec_off, int64_t *small) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w.S) return;
    if (bad[k]) { atomicOr((unsigned long long *)&small[BS_BAD], 1ull); return; }
    bam_walk(w.b, start[k], bam_seg_end(w, k), w.L, w.Lstream, rec_off + base[k]);
}

struct BamOut {
    int32_t *ref_id, *pos, *mate_ref_id, *mate_pos, *end_pos;
    uint16_t *flag, *total_len, *lowphred_run;
    uint8_t *mapq, *aux;
    uint32_t *blk_off;
    int32_t *blk_ref_pos, *blk_match_ref;
    uint16_t *blk_read_pos, *blk_match_read;
    uint16_t *lseq;  // non-null only under the synthesised-quality rule
};
__global__ void k_bam_decode(const uint8_t *b, const int64_t *rec_off, int64_t n, int64_t r0, BamDecodeParams prm, NameSet ns, BamOut o, uint32_t *nblk, int64_t *small) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    BamRec x;
    bam_decode(b + rec_off[i], prm, ns, x);
    const int64_t r = r0 + i;
    o.ref_id[r] = x.ref_id; o.pos[r] = x.pos; o.mate_ref_id[r] = x.mate_ref_id; o.mate_pos[r] = x.mate_pos; o.end_pos[r] = x.end_pos;
    o.flag[r] = x.flag; o.mapq[r] = x.mapq; o.aux[r] = x.aux;
    o.total_len[r] = (uint16_t)x.total_len;
    o.lowphred_run[r] = (uint16_t)(x.lowphred < 65535 ? x.lowphred : 65535);
    if (o.lseq) o.lseq[r] = (uint16_t)((uint32_t)x.lseq_cigar < 65535u ? (uint32_t)x.lseq_cigar : 65535u);
    nblk[i] = x.n_blk;
    if (x.aux_bad) atomicOr((unsigned long long *)&small[BS_AUXBAD], 1ull);
    if (x.l_seq) small[BS_SEQ] = 1;
    // pack_concordant's refusals, the first record in file order wins: key = record << 33 | (limit - 1) << 32 | TotalLen
    if (const int lim = packer_limit(x.n_blk, x.total_len))
        atomicMin((unsigned long long *)&small[BS_ERRKEY], ((unsigned long long)r << 33) | ((unsigned long long)(lim - 1) << 32) | (uint32_t)x.total_len);
}
__global__ void k_bam_blocks(const uint8_t *b, const int64_t *rec_off, int64_t n, int64_t r0, uint64_t b0, const uint64_t *incl, const uint32_t *nblk, BamOut o) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t first = b0 + incl[i] - nblk[i];
    o.blk_off[r0 + i + 1] = (uint32_t)(b0 + incl[i]);
    bam_blocks(b + rec_off[i], [&](uint32_t k, int32_t ref_pos, int32_t match_ref, int32_t read_pos, int32_t match_read) {
        o.blk_ref_pos[first + k] = ref_pos; o.blk_match_ref[first + k] = match_ref;
        o.blk_read_pos[first + k] = (uint16_t)read_pos; o.blk_match_read[first + k] = (uint16_t)match_read;
    });
}
__global__ void k_bam_null_qual(uint16_t *lowphred_run, const uint16_t *lseq, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) lowphred_run[i] = lseq[i];
}

namespace {
struct MappedFile {
    const uint8_t *p = nullptr; size_t n = 0;
    ~MappedFile() { if (p) munmap((void *)p, n); }
};
}  // namespace

static int bam_load(sqg_ctx *ctx, const char *path, const sqg_bam_decode *opt, int64_t first_record_index) {
    HostLap lap;
    MappedFile mf;
    {  // the host front end's wording for a missing / empty file
        int fd = ::open(path, O_RDONLY);
        if (fd < 0) FAIL(SQG_EINVAL, std::string("cannot open ") + path);
        struct stat st;
        if (fstat(fd, &st) != 0 || st.st_size < 4) { ::close(fd); FAIL(SQG_EINVAL, std::string(path) + " is empty"); }
        void *m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        ::close(fd);
        if (m == MAP_FAILED) FAIL(SQG_EINVAL, std::string("cannot map ") + path);
        mf.p = (const uint8_t *)m; mf.n = (size_t)st.st_size;
    }
    const uint8_t *f = mf.p;
    const bool raw = memcmp(f, "BAM\1", 4) == 0;
    std::vector<sqh::BgzfMember> mem;
    std::string e;
    if (!sqh::bam_loader_members(f, mf.n, raw, mem, e)) FAIL(SQG_EINVAL, e);
    std::vector<std::string> ref_names;
    std::vector<int32_t> ref_lens;
    size_t hdr_end = 0;
    std::string hdr_err;
    const bool hdr_ok = sqh::bam_read_header(f, mf.n, raw ? nullptr : &mem, ref_names, ref_lens, hdr_end, hdr_err);
    if (raw && !hdr_ok) FAIL(SQG_EINVAL, hdr_err);
    lap("bam: index + header");
    const int64_t T = mem.empty() ? 0 : (int64_t)(mem.back().off + mem.back().isize);
    // windows of whole members, about SQG_BAM_WINDOW_MB of inflated bytes
    const int64_t win_bytes = (int64_t)std::max(1, getenv("SQG_BAM_WINDOW_MB") ? atoi(getenv("SQG_BAM_WINDOW_MB")) : 1024) << 20;
    const std::vector<size_t> wcut = sqh::bam_window_cuts(mem, win_bytes, hdr_end);
    const size_t W = wcut.size() - 1;
    if (W == 0) FAIL(SQG_EINVAL, hdr_err);  // no data at all
    ctx->bam_members = (int64_t)mem.size(); ctx->bam_windows = (int64_t)W; ctx->bam_repair_rounds = 0;
    const int64_t nn = opt->n_names;
    const sqh::NameTable nt = sqh::bam_name_table(opt->names, opt->name_off, nn);
    const size_t cap = nt.hash.size();
    const int64_t blob_len = nn > 0 ? opt->name_off[nn] : 0;
    cudaStream_t st = ctx->stream;
    if (!ctx->stream_up) CK(cudaStreamCreateWithFlags(&ctx->stream_up, cudaStreamNonBlocking));
    cudaStream_t up = ctx->stream_up;
    while (ctx->bam_ev.size() < 3) { cudaEvent_t ev; CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)); ctx->bam_ev.push_back(ev); }
    CK(ctx->bam_nhash.ensure(cap)); CK(ctx->bam_nlen.ensure(cap)); CK(ctx->bam_noff.ensure(cap)); CK(ctx->bam_nblob.ensure((size_t)blob_len + 1));
    CK(cudaMemcpyAsync(ctx->bam_nhash.p, nt.hash.data(), cap * 8, cudaMemcpyHostToDevice, st)); CK(cudaMemcpyAsync(ctx->bam_nlen.p, nt.len.data(), cap * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->bam_noff.p, nt.off.data(), cap * 8, cudaMemcpyHostToDevice, st));
    if (blob_len) CK(cudaMemcpyAsync(ctx->bam_nblob.p, opt->names, (size_t)blob_len, cudaMemcpyHostToDevice, st));
    NameSet ns{ctx->bam_nhash.p, ctx->bam_nlen.p, ctx->bam_noff.p, ctx->bam_nblob.p, cap - 1, nn > 0};
    const int thr = phred_threshold(opt->phred33, opt->min_phred);
    const BamDecodeParams prm{thr};
    // with no qualities anywhere in the file the host decoder synthesises them ('I' everywhere, decode_alignment), which only
    // matters when the threshold lies above 'I': then the run is the read length of the CIGAR
    const bool keep_lseq = thr > 'I';
    CK(ctx->bam_small.ensure(BS_N)); CK(ctx->bam_hsmall.ensure(BS_N)); CK(ctx->cnt.ensure());  // (sqg_stat: as after a wire load)
    for (int i = 0; i < 2; i++) CK(ctx->bam_stage[i].ensure(kBamStage));
    for (const char *nm : {"bam_h2d", "bam_inflate", "bam_records", "bam_decode"}) { ctx->acc_ms[nm] = 0.f; PhaseTimer &t = ctx->timers[nm]; if (!t.a) { CK(cudaEventCreate(&t.a)); CK(cudaEventCreate(&t.b)); } t.done = false; }
    const int64_t zero_small[BS_N] = {0, 0, 0, -1, 0, 0};  // BS_ERRKEY: ~0 as unsigned, the neutral element of atomicMin
    CK(cudaMemcpyAsync(ctx->bam_small.p, zero_small, sizeof(zero_small), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    int64_t R = 0;        // records so far
    uint64_t B = 0;       // blocks so far
    int64_t carry = 0;    // unconsumed tail of the previous window, at the front of this one's buffer
    int cur = 0;
    int fatal = 0;        // walk / header / capacity refusal: later windows are only inflated (an inflate error outranks it, as on the host)
    std::string fatal_msg;
    bool aux_bad = false;
    int64_t infl_bits = 0;
    auto elapsed = [&](const char *nm) { PhaseTimer &t = ctx->timers[nm]; float ms = 0.f; if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) ctx->acc_ms[nm] += ms; };
    for (size_t w = 0; w < W; w++) {
        const sqh::BgzfMember &m0 = mem[wcut[w]], &m1 = mem[wcut[w + 1] - 1];
        const int64_t wstream = (int64_t)m0.off, wisize = (int64_t)(m1.off + m1.isize) - wstream;
        const int64_t L = carry + wisize, Lstream = carry + (T - wstream);
        // -- upload: the file range of the window's members, through two pinned staging buffers; raw streams go straight to the window
        const size_t f0 = m0.cdata, f1 = m1.cdata + m1.clen;
        CK(ctx->bam_win[cur].grow((size_t)L + 8, 0, st));
        uint8_t *dwin = ctx->bam_win[cur].p;
        if (carry) CK(cudaMemcpyAsync(dwin, ctx->bam_win[cur ^ 1].p + (ctx->bam_win_len - carry), (size_t)carry, cudaMemcpyDeviceToDevice, st));
        uint8_t *dst = raw ? dwin + carry : nullptr;
        if (!raw) { CK(ctx->bam_comp.ensure(f1 - f0)); dst = ctx->bam_comp.p; }
        CK(cudaEventRecord(ctx->bam_ev[2], st)); CK(cudaStreamWaitEvent(up, ctx->bam_ev[2], 0));  // buffers free of the previous window
        CK(cudaEventRecord(ctx->timers["bam_h2d"].a, up));
        for (size_t o = f0, c = 0; o < f1; o += kBamStage, c++) {
            const size_t len = std::min(kBamStage, f1 - o), sb = c & 1;
            if (c >= 2) CK(cudaEventSynchronize(ctx->bam_ev[sb]));
            memcpy(ctx->bam_stage[sb].p, f + o, len);
            CK(cudaMemcpyAsync(dst + (o - f0), ctx->bam_stage[sb].p, len, cudaMemcpyHostToDevice, up));
            CK(cudaEventRecord(ctx->bam_ev[sb], up));
        }
        CK(cudaEventRecord(ctx->timers["bam_h2d"].b, up));
        CK(cudaStreamWaitEvent(st, ctx->timers["bam_h2d"].b, 0));
        // -- inflate
        CK(cudaEventRecord(ctx->timers["bam_inflate"].a, st));
        if (!raw) {
            const int64_t nm = (int64_t)(wcut[w + 1] - wcut[w]);
            std::vector<BamMember> hm((size_t)nm);
            for (int64_t i = 0; i < nm; i++) {
                const sqh::BgzfMember &m = mem[wcut[w] + (size_t)i];
                hm[(size_t)i] = BamMember{m.cdata - f0, (uint64_t)(carry + ((int64_t)m.off - wstream)), (uint32_t)m.clen, m.isize, m.crc, 0};
            }
            CK(ctx->bam_mem.ensure((size_t)nm));
            CK(cudaMemcpyAsync(ctx->bam_mem.p, hm.data(), hm.size() * sizeof(BamMember), cudaMemcpyHostToDevice, st));
            LAUNCH_ON(st, k_bam_inflate, (unsigned)((nm + kInflWarps - 1) / kInflWarps), kInflWarps * 32, ctx->bam_mem.p, nm, ctx->bam_comp.p, dwin, ctx->bam_small.p);
            CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));  // (pageable member table: the copy above must finish before hm goes)
            infl_bits |= ctx->bam_hsmall.p[BS_INFL];
        }
        CK(cudaEventRecord(ctx->timers["bam_inflate"].b, st));
        if (w == 0 && !hdr_ok && !fatal) { fatal = SQG_EINVAL; fatal_msg = hdr_err; }
        if (infl_bits || fatal) { CK(cudaStreamSynchronize(st)); elapsed("bam_h2d"); elapsed("bam_inflate"); carry = 0; continue; }
        // -- record boundaries
        CK(cudaEventRecord(ctx->timers["bam_records"].a, st));
        const std::vector<int64_t> seg = sqh::bam_window_segments(mem, wcut, w, carry, hdr_end);
        const int64_t S = (int64_t)seg.size();
        CK(ctx->bam_seg.ensure((size_t)S)); CK(ctx->bam_start.ensure((size_t)S)); CK(ctx->bam_exit.ensure((size_t)S)); CK(ctx->bam_newstart.ensure((size_t)S));
        CK(ctx->bam_cnt.ensure((size_t)S + 1)); CK(ctx->bam_base.ensure((size_t)S + 1)); CK(ctx->bam_bad.ensure((size_t)S)); CK(ctx->bam_redo.ensure((size_t)S));
        CK(cudaMemcpyAsync(ctx->bam_seg.p, seg.data(), (size_t)S * 8, cudaMemcpyHostToDevice, st));
        const BamWin bw{dwin, L, Lstream, (int32_t)ref_lens.size(), S, ctx->bam_seg.p};
        LAUNCH_ON(st, k_bam_spec, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p);
        for (int round = 0;; round++) {
            CK(cudaMemsetAsync(ctx->bam_small.p + BS_CHANGED, 0, 8, st));
            LAUNCH_ON(st, k_bam_mark, blocks_for(S), kThreads, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_newstart.p, ctx->bam_redo.p, ctx->bam_small.p);
            CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (ctx->bam_hsmall.p[BS_CHANGED] == 0) break;
            ctx->bam_repair_rounds++;
            if (round == kBamMaxRounds) {
                LAUNCH_ON(st, k_bam_sequential, 1, 1, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p);
                break;
            }
            LAUNCH_ON(st, k_bam_rewalk, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_exit.p, ctx->bam_cnt.p, ctx->bam_bad.p, ctx->bam_newstart.p, ctx->bam_redo.p);
        }
        CK(cudaMemsetAsync(ctx->bam_cnt.p + S, 0, 4, st));
        CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::ExclusiveSum(t, tb, ctx->bam_cnt.p, ctx->bam_base.p, (int)(S + 1), st); }));
        int64_t nrec_w = 0, tail = 0;
        uint32_t nrec32 = 0;
        CK(cudaMemcpyAsync(&nrec32, ctx->bam_base.p + S, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&tail, ctx->bam_exit.p + (S - 1), 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nrec_w = nrec32;
        CK(ctx->bam_recoff.ensure((size_t)nrec_w + 1));
        LAUNCH_ON(st, k_bam_offsets, blocks_for(S, 128), 128, bw, ctx->bam_start.p, ctx->bam_bad.p, ctx->bam_base.p, ctx->bam_recoff.p, ctx->bam_small.p);
        CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaEventRecord(ctx->timers["bam_records"].b, st));
        if (ctx->bam_hsmall.p[BS_BAD] || (w + 1 == W && tail != L)) { fatal = SQG_EINVAL; fatal_msg = "truncated or malformed BAM alignment record"; }
        else if (R + nrec_w >= 0x7fffff00ll) { fatal = SQG_EUNSUPPORTED; fatal_msg = "more than 2^31 records per context: shard the stream"; }
        if (fatal) { CK(cudaStreamSynchronize(st)); elapsed("bam_h2d"); elapsed("bam_inflate"); elapsed("bam_records"); carry = 0; continue; }
        // -- decode into the resident batch (capacity grows geometrically and keeps what earlier windows wrote)
        CK(cudaEventRecord(ctx->timers["bam_decode"].a, st));
        const size_t need = (size_t)(R + nrec_w) + 1, used = (size_t)R;
#define X(T, name, ext) if (ext != BX_BLK) CK(ctx->o_##name.grow(need + (ext == BX_OFF), used + (ext == BX_OFF), st));
        SQ_BATCH_ARRAYS(X)
#undef X
        if (keep_lseq) CK(ctx->bam_lseq.grow(need, used, st));
        if (R == 0) CK(cudaMemsetAsync(ctx->o_blk_off.p, 0, 4, st));
        CK(ctx->bam_nblk.ensure((size_t)nrec_w + 1)); CK(ctx->bam_incl.ensure((size_t)nrec_w + 1));
        BamOut bo{ctx->o_ref_id.p, ctx->o_pos.p, ctx->o_mate_ref_id.p, ctx->o_mate_pos.p, ctx->o_end_pos.p, ctx->o_flag.p, ctx->o_total_len.p, ctx->o_lowphred_run.p,
                  ctx->o_mapq.p, ctx->o_aux.p, ctx->o_blk_off.p, nullptr, nullptr, nullptr, nullptr, keep_lseq ? ctx->bam_lseq.p : nullptr};
        uint64_t nblk_w = 0;
        if (nrec_w > 0) {
            LAUNCH_ON(st, k_bam_decode, blocks_for(nrec_w), kThreads, dwin, ctx->bam_recoff.p, nrec_w, R, prm, ns, bo, ctx->bam_nblk.p, ctx->bam_small.p);
            CK(cub_call(ctx->d_temp, [&](void *t, size_t &tb) { return cub::DeviceScan::InclusiveSum(t, tb, ctx->bam_nblk.p, ctx->bam_incl.p, (int)nrec_w, st); }));
            CK(cudaMemcpyAsync(&nblk_w, ctx->bam_incl.p + (nrec_w - 1), 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        if (B + nblk_w > 0xFFFFFFFFull) { fatal = SQG_EUNSUPPORTED; fatal_msg = "more than 2^32 - 1 aligned blocks in one batch: shard the stream"; }
        else if (nrec_w > 0) {
            const size_t bneed = (size_t)(B + nblk_w) + 1;
#define X(T, name, ext) if (ext == BX_BLK) CK(ctx->o_##name.grow(bneed, (size_t)B, st));
            SQ_BATCH_ARRAYS(X)
#undef X
            bo.blk_ref_pos = ctx->o_blk_ref_pos.p; bo.blk_match_ref = ctx->o_blk_match_ref.p; bo.blk_read_pos = ctx->o_blk_read_pos.p; bo.blk_match_read = ctx->o_blk_match_read.p;
            LAUNCH_ON(st, k_bam_blocks, blocks_for(nrec_w), kThreads, dwin, ctx->bam_recoff.p, nrec_w, R, B, ctx->bam_incl.p, ctx->bam_nblk.p, bo);
        }
        CK(cudaEventRecord(ctx->timers["bam_decode"].b, st));
        CK(cudaStreamSynchronize(st));
        elapsed("bam_h2d"); elapsed("bam_inflate"); elapsed("bam_records"); elapsed("bam_decode");
        R += nrec_w; B += nblk_w;
        carry = L - tail;
        ctx->bam_win_len = L;
        cur ^= 1;
    }
    CK(cudaMemcpyAsync(ctx->bam_hsmall.p, ctx->bam_small.p, BS_N * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    aux_bad = ctx->bam_hsmall.p[BS_AUXBAD] != 0;
    for (const char *nm : {"bam_h2d", "bam_inflate", "bam_records", "bam_decode"}) ctx->timers[nm].done = false;
    lap("bam: windows");
    // the host front end's order: inflate, header, record boundaries, aux fields, then the packer's own refusals
    if (infl_bits) FAIL(SQG_EINVAL, (infl_bits & 1) ? "corrupt deflate stream in a BGZF block" : "BGZF block fails its CRC32");
    if (fatal == SQG_EINVAL) FAIL(fatal, fatal_msg);
    if (aux_bad) FAIL(SQG_EINVAL, "malformed BAM alignment record");
    const uint64_t key = (uint64_t)ctx->bam_hsmall.p[BS_ERRKEY];
    if (key != ~0ull) {
        FAIL(SQG_EUNSUPPORTED, sqh::packer_refusal(key >> 33, (int)(key >> 32 & 1) + 1, (uint32_t)key));
    }
    if (fatal) FAIL(fatal, fatal_msg);
    if (keep_lseq && R > 0 && ctx->bam_hsmall.p[BS_SEQ] == 0) LAUNCH_ON(st, k_bam_null_qual, blocks_for(R), kThreads, ctx->o_lowphred_run.p, ctx->bam_lseq.p, R);
#define X(T, name, ext) CK(ctx->o_##name.grow(1, 0, st));
    SQ_BATCH_ARRAYS(X)  // (every array exists, also for an empty batch)
#undef X
    if (R == 0) CK(cudaMemsetAsync(ctx->o_blk_off.p, 0, 4, st));  // an empty batch still has its blk_off[0]
    point_batch_at_own_arrays(ctx, R, (int64_t)B);
    reset_batch_state(ctx, true, first_record_index, false);
    return SQG_OK;
}

extern "C" int sqg_load_concordant_bam(sqg_ctx *ctx, const char *path, const sqg_bam_decode *opt, int64_t first_record_index) {
    if (!ctx || !path || !opt || opt->n_names < 0 || (opt->n_names > 0 && (!opt->names || !opt->name_off))) return SQG_EINVAL;
    CK(cudaSetDevice(ctx->device));
    { const int rcj = cov_join(ctx); if (rcj) return rcj; }
    ctx->have_batch = false;  // the resident arrays are rewritten from here on: a refused load leaves no batch
    ctx->acc_ms.clear();
    const int rc = bam_load(ctx, path, opt, first_record_index);
    if (rc == SQG_ECUDA) cudaGetLastError();
    return rc;
}
