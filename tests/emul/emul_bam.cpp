// CPU stepping of the device BAM decode (squid_b200/csrc/sq_inflate.cuh, sq_bam.cuh): the loader's own plan (host/bam.h) and the
// same SQ_HD rules, run serially in the order the kernels of sqg_load_concordant_bam run them, so that tests/test_cpu_bam_device.py
// can compare them with zlib and with the host front end without a GPU.
//   emul_bam inflate <bgzf file> <out>
//       every member inflated as k_bam_inflate does it (matches of kInflWarpCopyMin bytes or more copied by the "warp", the CRC
//       summed over 32 slices and combined); writes the stream to <out>, prints "status <bits>" (1: a corrupt member, 2: a CRC mismatch)
//   emul_bam decode <bam> <names blob> <names int64 offsets> <phred33> <min_phred> <window bytes> <outdir>
//       the windowed record boundaries and the decode; writes the 15 sqg_batch arrays as <outdir>/<field>.bin and prints
//       "records <n> blocks <n> windows <n> rounds <n>", or "error <code> <message>" (exit 3)
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "host/bam.h"
#include "sq_bam.cuh"
#include "sq_inflate.cuh"

using namespace sq;

static std::vector<uint8_t> slurp(const char *path) {
    std::vector<uint8_t> v;
    FILE *f = fopen(path, "rb");
    if (!f) return v;
    fseek(f, 0, SEEK_END);
    v.resize((size_t)ftell(f));
    fseek(f, 0, SEEK_SET);
    if (!v.empty() && fread(v.data(), 1, v.size(), f) != v.size()) v.clear();
    fclose(f);
    return v;
}

static uint32_t crc_tab[256], x2n[32];

// one member as the warp runs it; 0 ok, 1 corrupt, 2 CRC mismatch
static int inflate_member(const uint8_t *in, uint32_t clen, uint8_t *out, uint32_t isize, uint32_t crc_want) {
    static InflateTables t;
    InflateState s;
    inflate_init(s, in, clen, out, isize);
    int rc;
    for (;;) {
        uint32_t dst = 0, len = 0, dist = 1;
        rc = inflate_step(s, t, kInflWarpCopyMin, &dst, &len, &dist);
        if (rc != 1) break;
        for (uint32_t lane = 0; lane < 32; lane++)
            for (uint32_t i = lane; i < len; i += 32) out[dst + i] = out[dst - dist + i % dist];
    }
    if (rc < 0) return 1;
    uint32_t crc[32], len[32];
    for (uint32_t lane = 0; lane < 32; lane++) {
        const uint32_t a = (uint32_t)((uint64_t)isize * lane / 32), b = (uint32_t)((uint64_t)isize * (lane + 1) / 32);
        crc[lane] = crc32_update(crc_tab, 0, out + a, b - a); len[lane] = b - a;
    }
    for (int off = 1; off < 32; off <<= 1)
        for (int lane = 0; lane + off < 32; lane++)
            if ((lane & (2 * off - 1)) == 0) { crc[lane] = crc32_combine(x2n, crc[lane], crc[lane + off], len[lane + off]); len[lane] += len[lane + off]; }
    return crc[0] == crc_want ? 0 : 2;
}

static int fail(int code, const std::string &m) { printf("error %d %s\n", code, m.c_str()); return 3; }

template <class T> static void dump(const std::string &dir, const char *name, const std::vector<T> &v) {
    FILE *f = fopen((dir + "/" + name + ".bin").c_str(), "wb");
    if (!v.empty()) fwrite(v.data(), sizeof(T), v.size(), f);
    fclose(f);
}

int main(int argc, char **argv) {
    for (uint32_t n = 0; n < 256; n++) crc_tab[n] = crc32_entry(n);
    crc32_x2n(x2n);
    if (argc == 4 && !strcmp(argv[1], "inflate")) {
        const std::vector<uint8_t> f = slurp(argv[2]);
        std::vector<sqh::BgzfMember> mem;
        std::string e;
        if (!sqh::bgzf_parse_members(f.data(), f.size(), mem, e)) { printf("parse %s\n", e.c_str()); return 3; }
        std::vector<uint8_t> out(mem.empty() ? 0 : mem.back().off + mem.back().isize);
        int bits = 0;
        for (const sqh::BgzfMember &m : mem) if (m.isize) { const int r = inflate_member(f.data() + m.cdata, (uint32_t)m.clen, out.data() + m.off, m.isize, m.crc); if (r) bits |= r; }
        FILE *o = fopen(argv[3], "wb");
        if (!out.empty()) fwrite(out.data(), 1, out.size(), o);
        fclose(o);
        printf("status %d\n", bits);
        return 0;
    }
    if (argc != 9 || strcmp(argv[1], "decode")) { fprintf(stderr, "usage: see the head of emul_bam.cpp\n"); return 2; }
    const std::vector<uint8_t> f = slurp(argv[2]);
    if (f.size() < 4) return fail(-1, std::string(argv[2]) + " is empty");
    const std::vector<uint8_t> blob = slurp(argv[3]), offb = slurp(argv[4]);
    std::vector<int64_t> name_off(offb.size() / 8);
    if (!offb.empty()) memcpy(name_off.data(), offb.data(), offb.size());
    const int64_t nn = name_off.empty() ? 0 : (int64_t)name_off.size() - 1;
    const int thr = phred_threshold(atoi(argv[5]) != 0, atoi(argv[6]));
    const int64_t win_bytes = atoll(argv[7]);
    const std::string outdir = argv[8];
    const bool raw = memcmp(f.data(), "BAM\1", 4) == 0;
    std::vector<sqh::BgzfMember> mem;
    std::string e;
    if (!sqh::bam_loader_members(f.data(), f.size(), raw, mem, e)) return fail(-1, e);
    std::vector<std::string> rn; std::vector<int32_t> rl;
    size_t hdr_end = 0;
    std::string herr;
    const bool hdr_ok = sqh::bam_read_header(f.data(), f.size(), raw ? nullptr : &mem, rn, rl, hdr_end, herr);
    if (raw && !hdr_ok) return fail(-1, herr);
    const int64_t T = mem.empty() ? 0 : (int64_t)(mem.back().off + mem.back().isize);
    const std::vector<size_t> wcut = sqh::bam_window_cuts(mem, win_bytes, hdr_end);
    const size_t W = wcut.size() - 1;
    if (W == 0) return fail(-1, herr);
    const sqh::NameTable nt = sqh::bam_name_table((const char *)blob.data(), name_off.data(), nn);
    const NameSet ns{nt.hash.data(), nt.len.data(), nt.off.data(), blob.data(), nt.hash.size() - 1, nn > 0};
    const BamDecodeParams prm{thr};
    std::vector<int32_t> ref_id, pos, mref, mpos, endp, bref, bmref; std::vector<uint16_t> flag, tlen, low, brpos, bmread, lseq; std::vector<uint8_t> mapq, aux;
    std::vector<uint32_t> blk_off{0};
    std::vector<uint8_t> prev, cur;
    int64_t carry = 0, rounds = 0;
    int infl = 0, fatal = 0;
    std::string fmsg, refusal;
    bool aux_bad = false, any_seq = false;
    for (size_t w = 0; w < W; w++) {
        const sqh::BgzfMember &m0 = mem[wcut[w]], &m1 = mem[wcut[w + 1] - 1];
        const int64_t wstream = (int64_t)m0.off, wis = (int64_t)(m1.off + m1.isize) - wstream, L = carry + wis, Ls = carry + (T - wstream);
        cur.assign((size_t)L + 8, 0);
        if (carry) memcpy(cur.data(), prev.data() + (prev.size() - 8 - carry), (size_t)carry);
        for (size_t i = wcut[w]; i < wcut[w + 1]; i++) {
            const sqh::BgzfMember &m = mem[i];
            uint8_t *o = cur.data() + carry + ((int64_t)m.off - wstream);
            if (raw) memcpy(o, f.data() + m.cdata, m.clen);
            else infl |= inflate_member(f.data() + m.cdata, (uint32_t)m.clen, o, m.isize, m.crc);
        }
        if (w == 0 && !hdr_ok && !fatal) { fatal = -1; fmsg = herr; }
        if (infl || fatal) { carry = 0; continue; }
        const std::vector<int64_t> seg = sqh::bam_window_segments(mem, wcut, w, carry, hdr_end);
        const int64_t S = (int64_t)seg.size();
        auto send = [&](int64_t k) { return k + 1 < S ? seg[k + 1] : L; };
        std::vector<int64_t> start(S), ex(S), ns2(S); std::vector<uint32_t> cnt(S); std::vector<uint8_t> bad(S), redo(S);
        const uint8_t *b = cur.data();
        for (int64_t k = 0; k < S; k++) {  // k_bam_spec
            const int64_t a = k == 0 ? seg[0] : bam_spec_start(b, seg[k], send(k), L, Ls, (int32_t)rl.size());
            const SegWalk r = bam_walk(b, a, send(k), L, Ls, nullptr);
            start[k] = a; ex[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad;
        }
        for (int round = 0;; round++) {
            int64_t changed = 0;
            for (int64_t k = 0; k < S; k++) { redo[k] = k > 0 && ex[k - 1] != start[k]; if (redo[k]) { ns2[k] = ex[k - 1]; changed++; } }  // k_bam_mark
            if (!changed) break;
            rounds++;
            if (round == kBamMaxRounds) {  // k_bam_sequential
                int64_t a = seg[0];
                for (int64_t k = 0; k < S; k++) { const SegWalk r = bam_walk(b, a, send(k), L, Ls, nullptr); start[k] = a; ex[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad; a = r.exit; }
                break;
            }
            for (int64_t k = 0; k < S; k++) if (redo[k]) { const SegWalk r = bam_walk(b, ns2[k], send(k), L, Ls, nullptr); start[k] = ns2[k]; ex[k] = r.exit; cnt[k] = r.n; bad[k] = r.bad; }
        }
        std::vector<int64_t> rec;
        bool anybad = false;
        for (int64_t k = 0; k < S; k++) {  // k_bam_offsets
            if (bad[k]) { anybad = true; continue; }
            std::vector<int64_t> r(cnt[k]);
            bam_walk(b, start[k], send(k), L, Ls, r.data());
            rec.insert(rec.end(), r.begin(), r.end());
        }
        if (anybad || (w + 1 == W && ex[S - 1] != L)) { fatal = -1; fmsg = "truncated or malformed BAM alignment record"; carry = 0; continue; }
        for (size_t i = 0; i < rec.size(); i++) {  // k_bam_decode, k_bam_blocks
            BamRec x;
            bam_decode(b + rec[i], prm, ns, x);
            const uint64_t r = ref_id.size();
            ref_id.push_back(x.ref_id); pos.push_back(x.pos); mref.push_back(x.mate_ref_id); mpos.push_back(x.mate_pos); endp.push_back(x.end_pos);
            flag.push_back(x.flag); mapq.push_back(x.mapq); aux.push_back(x.aux); tlen.push_back((uint16_t)x.total_len);
            low.push_back((uint16_t)std::min(x.lowphred, 65535)); lseq.push_back((uint16_t)std::min<uint32_t>((uint32_t)x.lseq_cigar, 65535u));
            aux_bad |= x.aux_bad; any_seq |= x.l_seq > 0;
            const int lim = packer_limit(x.n_blk, x.total_len);
            if (lim && refusal.empty()) refusal = sqh::packer_refusal(r, lim, x.total_len);
            bam_blocks(b + rec[i], [&](uint32_t, int32_t rp, int32_t mr, int32_t qp, int32_t mq) {
                bref.push_back(rp); bmref.push_back(mr); brpos.push_back((uint16_t)qp); bmread.push_back((uint16_t)mq);
            });
            blk_off.push_back((uint32_t)bref.size());
        }
        carry = L - ex[S - 1];
        prev.swap(cur);
    }
    if (infl) return fail(-1, (infl & 1) ? "corrupt deflate stream in a BGZF block" : "BGZF block fails its CRC32");
    if (fatal) return fail(fatal, fmsg);
    if (aux_bad) return fail(-1, "malformed BAM alignment record");
    if (!refusal.empty()) return fail(-5, refusal);
    if (thr > 'I' && !any_seq) low = lseq;
    dump(outdir, "ref_id", ref_id); dump(outdir, "pos", pos); dump(outdir, "mate_ref_id", mref); dump(outdir, "mate_pos", mpos); dump(outdir, "end_pos", endp);
    dump(outdir, "flag", flag); dump(outdir, "total_len", tlen); dump(outdir, "lowphred_run", low); dump(outdir, "mapq", mapq); dump(outdir, "aux", aux);
    dump(outdir, "blk_off", blk_off); dump(outdir, "blk_ref_pos", bref); dump(outdir, "blk_match_ref", bmref); dump(outdir, "blk_read_pos", brpos); dump(outdir, "blk_match_read", bmread);
    printf("records %zu blocks %zu windows %zu rounds %lld\n", ref_id.size(), bref.size(), W, (long long)rounds);
    return 0;
}
