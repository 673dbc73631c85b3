#include "bam.h"

#include <fcntl.h>
#include <omp.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "sq_bam.cuh"

namespace sqh {
namespace {
inline uint16_t rd16(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }
inline uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline int32_t rdi32(const uint8_t *p) { int32_t v; memcpy(&v, p, 4); return v; }

}  // namespace

bool bgzf_parse_members(const uint8_t *d, size_t len, std::vector<BgzfMember> &mem, std::string &err) {
    mem.clear();
    size_t o = 0, total = 0;
    while (o < len) {
        if (o + 18 > len || d[o] != 0x1f || d[o + 1] != 0x8b || d[o + 2] != 8 || !(d[o + 3] & 4)) { err = "not a BGZF member at offset " + std::to_string(o); return false; }
        const uint16_t xlen = rd16(d + o + 10);
        size_t x = o + 12, xe = x + xlen;
        if (xe > len) { err = "truncated BGZF header"; return false; }
        int64_t bsize = -1;
        while (x + 4 <= xe) {  // extra subfields: SI1 SI2 SLEN data
            const uint16_t slen = rd16(d + x + 2);
            if (d[x] == 'B' && d[x + 1] == 'C' && slen == 2 && x + 6 <= xe) bsize = rd16(d + x + 4);
            x += 4 + slen;
        }
        if (bsize < 0) { err = "gzip member without a BC subfield (plain gzip is not BGZF)"; return false; }
        const size_t msize = (size_t)bsize + 1;
        if (o + msize > len || msize < (size_t)xlen + 20) { err = "truncated BGZF block"; return false; }
        BgzfMember m;
        m.cdata = o + 12 + xlen; m.clen = msize - xlen - 20; m.isize = rd32(d + o + msize - 4); m.crc = rd32(d + o + msize - 8); m.off = total;
        if (m.isize > 65536) { err = "BGZF block larger than 64 KiB"; return false; }
        total += m.isize;
        mem.push_back(m);
        o += msize;
    }
    return true;
}

bool bgzf_inflate_all(const uint8_t *d, size_t len, RawBuf<uint8_t> &out, std::string &err, int threads, std::vector<size_t> *member_off) {
    std::vector<BgzfMember> mem;
    if (!bgzf_parse_members(d, len, mem, err)) return false;
    const size_t total = mem.empty() ? 0 : mem.back().off + mem.back().isize;
    if (!out.resize(total)) { err = "out of memory"; return false; }
    if (member_off) {
        member_off->clear();
        for (const BgzfMember &m : mem) if (m.isize) member_off->push_back(m.off);
        member_off->push_back(total);
    }
    const int T = threads > 0 ? threads : omp_get_num_procs();
    int bad = 0;  // bit 0: corrupt deflate stream, bit 1: CRC mismatch
#pragma omp parallel for num_threads(T) schedule(dynamic, 16) reduction(| : bad)
    for (long long i = 0; i < (long long)mem.size(); i++) {
        const BgzfMember &m = mem[(size_t)i];
        if (m.isize == 0) continue;  // the EOF marker
        z_stream z;
        memset(&z, 0, sizeof(z));
        if (inflateInit2(&z, -15) != Z_OK) { bad |= 1; continue; }
        z.next_in = const_cast<Bytef *>(d + m.cdata); z.avail_in = (uInt)m.clen;
        z.next_out = out.data() + m.off; z.avail_out = m.isize;
        const int rc = inflate(&z, Z_FINISH);
        if (rc != Z_STREAM_END || z.avail_out != 0) bad |= 1;
        else if (crc32(crc32(0L, Z_NULL, 0), out.data() + m.off, m.isize) != m.crc) bad |= 2;
        inflateEnd(&z);
    }
    if (bad) { err = !(bad & 1) ? "BGZF block fails its CRC32" : "corrupt deflate stream in a BGZF block"; return false; }
    return true;
}

int bam_parse_header(const uint8_t *b, size_t n, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len, size_t &end, std::string &err) {
    ref_name.clear(); ref_len.clear();
    if (n < 12 || memcmp(b, "BAM\1", 4) != 0) { err = "not a BAM file (magic)"; return n < 12 && (n < 4 || memcmp(b, "BAM\1", 4) == 0) ? 0 : -1; }
    size_t o = 4;
    const int32_t l_text = rdi32(b + o); o += 4;
    if (l_text < 0) { err = "truncated BAM header"; return -1; }
    if (o + (size_t)l_text + 4 > n) { err = "truncated BAM header"; return 0; }
    o += (size_t)l_text;
    const int32_t n_ref = rdi32(b + o); o += 4;
    if (n_ref < 0) { err = "truncated BAM reference list"; return -1; }
    for (int32_t i = 0; i < n_ref; i++) {
        if (o + 4 > n) { err = "truncated BAM reference list"; return 0; }
        const int32_t l_name = rdi32(b + o); o += 4;
        if (l_name < 1) { err = "truncated BAM reference list"; return -1; }
        if (o + (size_t)l_name + 4 > n) { err = "truncated BAM reference list"; return 0; }
        ref_name.emplace_back((const char *)b + o, (size_t)l_name - 1); o += (size_t)l_name;
        ref_len.push_back(rdi32(b + o)); o += 4;
    }
    end = o;
    return 1;
}

bool bam_read_header(const uint8_t *f, size_t flen, const std::vector<BgzfMember> *mem, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len,
                     size_t &end, std::string &err) {
    if (!mem) return bam_parse_header(f, flen, ref_name, ref_len, end, err) == 1;
    std::vector<uint8_t> buf;
    int rc = 0;
    for (const BgzfMember &m : *mem) {
        if (m.isize == 0) continue;
        const size_t at = buf.size();
        buf.resize(at + m.isize);
        z_stream z;
        memset(&z, 0, sizeof(z));
        if (inflateInit2(&z, -15) != Z_OK) { err = "corrupt deflate stream in a BGZF block"; return false; }
        z.next_in = const_cast<Bytef *>(f + m.cdata); z.avail_in = (uInt)m.clen;
        z.next_out = buf.data() + at; z.avail_out = m.isize;
        const int zr = inflate(&z, Z_FINISH);
        const bool ok = zr == Z_STREAM_END && z.avail_out == 0;
        inflateEnd(&z);
        if (!ok) { err = "corrupt deflate stream in a BGZF block"; return false; }
        if (crc32(crc32(0L, Z_NULL, 0), buf.data() + at, m.isize) != m.crc) { err = "BGZF block fails its CRC32"; return false; }
        rc = bam_parse_header(buf.data(), buf.size(), ref_name, ref_len, end, err);
        if (rc != 0) break;
    }
    if (rc == 0 && err.empty()) err = "not a BAM file (magic)";
    return rc == 1;
}

bool bam_read_header_file(const std::string &path, std::vector<std::string> &ref_name, std::vector<int32_t> &ref_len, std::string &err) {
    int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) { err = "cannot open " + path; return false; }
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 4) { ::close(fd); err = path + " is empty"; return false; }
    const size_t flen = (size_t)st.st_size;
    void *map = mmap(nullptr, flen, PROT_READ, MAP_PRIVATE, fd, 0);
    ::close(fd);
    if (map == MAP_FAILED) { err = "cannot map " + path; return false; }
    const uint8_t *f = (const uint8_t *)map;
    size_t end = 0;
    bool ok;
    if (memcmp(f, "BAM\1", 4) == 0) ok = bam_read_header(f, flen, nullptr, ref_name, ref_len, end, err);
    else {
        std::vector<BgzfMember> mem;
        ok = bgzf_parse_members(f, flen, mem, err) && bam_read_header(f, flen, &mem, ref_name, ref_len, end, err);
    }
    munmap(map, flen);
    return ok;
}

bool BamTable::open(const std::string &path, std::string &err, int threads) {
    *this = BamTable();
    const bool timing = getenv("SQH_TIMING") != nullptr;
    auto T0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *w) { if (timing) { auto t = std::chrono::steady_clock::now(); fprintf(stderr, "[bam] %s %.1f ms\n", w, 1e3 * std::chrono::duration<double>(t - T0).count()); T0 = t; } };
    int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) { err = "cannot open " + path; return false; }
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 4) { ::close(fd); err = path + " is empty"; return false; }
    const size_t flen = (size_t)st.st_size;
    void *map = mmap(nullptr, flen, PROT_READ, MAP_PRIVATE, fd, 0);
    ::close(fd);
    if (map == MAP_FAILED) { err = "cannot map " + path; return false; }
    const uint8_t *f = (const uint8_t *)map;
    RawBuf<uint8_t> raw;
    std::vector<size_t> blocks;  // starts of the BGZF members in the inflated stream (+ its length)
    const uint8_t *b; size_t n;
    if (memcmp(f, "BAM\1", 4) == 0) { b = f; n = flen; }  // uncompressed BAM stream
    else {
        if (!bgzf_inflate_all(f, flen, raw, err, threads, &blocks)) { munmap(map, flen); return false; }
        b = raw.data(); n = raw.size();
    }
    lap("inflate");
    bool ok = false;
    do {
        size_t o = 0;
        if (bam_parse_header(b, n, ref_name, ref_len, o, err) != 1) break;
        // Record boundaries.  htslib never lets a record straddle two BGZF members (bgzf_flush_try before every record), so in
        // the files aligners and samtools write every member starts at a record boundary and the members can be walked
        // independently.  That is an assumption about the writer, so it is PROVEN before it is used: the walk of member k
        // (started at a true boundary) must end exactly where member k+1 starts -- by induction from the end of the header,
        // which is a true boundary, every start is then a true boundary.  Any member that does not end there (records
        // straddling members: other writers, tests/test_cpu_bam.py) sends the whole file down the sequential walk.
        const int T = threads > 0 ? threads : omp_get_num_procs();
        std::vector<size_t> seg;  // walk segments: [seg[k], seg[k+1])
        seg.push_back(o);
        for (size_t x : blocks) if (x > o && x < n) seg.push_back(x);
        seg.push_back(n);
        size_t S = seg.size() - 1;
        struct Tot { size_t rec, name, cig, seq; };
        std::vector<Tot> tot(S + 1, Tot{0, 0, 0, 0});
        auto walk = [&](size_t a, size_t e, Tot &t, size_t *rec_out, uint64_t *no, uint64_t *co, uint64_t *so) -> bool {
            size_t p = a;
            while (p < e) {
                // the variable-length fields have to fit the record before their sizes enter the totals that size the allocations
                int64_t next = 0;
                if (sq::bam_rec_check(b, (int64_t)p, (int64_t)e, (int64_t)e, &next) != 1) return false;
                const uint8_t *q = b + p + 4;
                const uint32_t l_name = q[8], n_cig = rd16(q + 12), l_seq = rd32(q + 16);
                if (rec_out) { rec_out[t.rec] = p + 4; no[t.rec] = t.name; co[t.rec] = t.cig; so[t.rec] = t.seq; }
                t.rec++; t.name += l_name ? l_name - 1 : 0; t.cig += n_cig; t.seq += l_seq;
                p = (size_t)next;
            }
            return true;
        };
        bool members_ok = S > 1;
        if (members_ok) {
            int fail = 0;
#pragma omp parallel for num_threads(T) schedule(dynamic, 8) reduction(| : fail)
            for (long long k = 0; k < (long long)S; k++) { Tot t{0, 0, 0, 0}; if (!walk(seg[(size_t)k], seg[(size_t)k + 1], t, nullptr, nullptr, nullptr, nullptr)) fail |= 1; tot[(size_t)k + 1] = t; }
            members_ok = !fail;
        }
        if (!members_ok) {  // one sequential walk over the whole stream
            seg.assign({o, n}); S = 1;
            tot.assign(2, Tot{0, 0, 0, 0});
            Tot t{0, 0, 0, 0};
            if (!walk(o, n, t, nullptr, nullptr, nullptr, nullptr)) { err = "truncated or malformed BAM alignment record"; break; }
            tot[1] = t;
        }
        for (size_t k = 1; k <= S; k++) { tot[k].rec += tot[k - 1].rec; tot[k].name += tot[k - 1].name; tot[k].cig += tot[k - 1].cig; tot[k].seq += tot[k - 1].seq; }
        walked_per_member = members_ok;
        lap(members_ok ? "record boundaries (per BGZF member)" : "record boundaries (sequential)");
        const size_t R = tot[S].rec;
        std::vector<size_t> rec(R);
        ref_id.resize(R); pos.resize(R); mate_ref_id.resize(R); mate_pos.resize(R); ih.assign(R, 0); flag.resize(R); mapq.resize(R); tags.assign(R, 0);
        name_off.resize(R + 1); cigar_off.resize(R + 1); seq_off.resize(R + 1);
        name_off[R] = tot[S].name; cigar_off[R] = tot[S].cig; seq_off[R] = tot[S].seq;
#pragma omp parallel for num_threads(T) schedule(dynamic, 8)
        for (long long k = 0; k < (long long)S; k++) {
            Tot t = tot[(size_t)k];
            const size_t r0 = t.rec;
            Tot local{0, t.name, t.cig, t.seq};
            walk(seg[(size_t)k], seg[(size_t)k + 1], local, rec.data() + r0, name_off.data() + r0, cigar_off.data() + r0, seq_off.data() + r0);
        }
        if (!names.resize(name_off[R]) || !cigar.resize(cigar_off[R]) || !seq.resize(seq_off[R]) || !qual.resize(seq_off[R])) { err = "out of memory"; break; }
        int bad = 0;
        lap("offsets + allocation");
#pragma omp parallel for num_threads(T) schedule(static) reduction(| : bad)
        for (long long rr = 0; rr < (long long)R; rr++) {
            const size_t r = (size_t)rr;
            const uint8_t *p = b + rec[r];
            const size_t bs = (size_t)rdi32(p - 4);
            const uint8_t *end = p + bs;
            ref_id[r] = rdi32(p); pos[r] = rdi32(p + 4);
            const uint32_t l_name = p[8];
            mapq[r] = p[9];
            const uint32_t n_cig = rd16(p + 12);
            flag[r] = rd16(p + 14);
            const uint32_t l_seq = rd32(p + 16);
            mate_ref_id[r] = rdi32(p + 20); mate_pos[r] = rdi32(p + 24);
            const uint8_t *q = p + 32;
            if (l_name) memcpy(names.data() + name_off[r], q, l_name - 1);
            q += l_name;
            memcpy(cigar.data() + cigar_off[r], q, 4ull * n_cig);
            q += 4ull * n_cig;
            static const char code[] = "=ACMGRSVTWYHKDBN";
            static const std::array<uint16_t, 256> pair = [] {  // two bases per packed byte, as one little-endian store
                std::array<uint16_t, 256> t{};
                for (int v = 0; v < 256; v++) t[(size_t)v] = (uint16_t)((uint8_t)code[v >> 4] | ((uint16_t)(uint8_t)code[v & 15] << 8));
                return t;
            }();
            char *sb = seq.data() + seq_off[r], *ql = qual.data() + seq_off[r];
            for (uint32_t k = 0; k + 1 < l_seq; k += 2) { const uint16_t w = pair[q[k >> 1]]; memcpy(sb + k, &w, 2); }
            if (l_seq & 1) sb[l_seq - 1] = code[q[l_seq >> 1] >> 4];
            q += (l_seq + 1) / 2;
            for (uint32_t k = 0; k < l_seq; k++) ql[k] = (char)(uint8_t)(q[k] + 33);
            q += l_seq;
            sq::BamAux a;
            if (!sq::bam_aux_scan(q, end, a)) bad |= 1;
            tags[r] = (uint8_t)(a.xa | a.ih << 1);
            ih[r] = a.ih_value;
        }
        if (bad) { err = "malformed BAM alignment record"; break; }
        lap("fields");
        ok = true;
    } while (false);
    munmap(map, flen);
    if (!ok) *this = BamTable();
    return ok;
}

bool bam_loader_members(const uint8_t *f, size_t len, bool raw, std::vector<BgzfMember> &mem, std::string &err) {
    mem.clear();
    if (raw) {
        for (size_t o = 0; o < len; o += 65536) mem.push_back(BgzfMember{o, std::min<size_t>(65536, len - o), o, (uint32_t)std::min<size_t>(65536, len - o), kRawMember});
        return true;
    }
    if (!bgzf_parse_members(f, len, mem, err)) return false;
    mem.erase(std::remove_if(mem.begin(), mem.end(), [](const BgzfMember &m) { return m.isize == 0; }), mem.end());
    return true;
}

std::vector<size_t> bam_window_cuts(const std::vector<BgzfMember> &mem, int64_t win_bytes, size_t hdr_end) {
    std::vector<size_t> cut{0};
    for (size_t i = 0; i < mem.size();) {
        size_t j = i;
        int64_t bytes = 0;
        while (j < mem.size() && (j == i || bytes + mem[j].isize <= win_bytes || (cut.size() == 1 && mem[j].off <= hdr_end))) { bytes += mem[j].isize; j++; }
        cut.push_back(j);
        i = j;
    }
    return cut;
}

std::vector<int64_t> bam_window_segments(const std::vector<BgzfMember> &mem, const std::vector<size_t> &cut, size_t w, int64_t carry, size_t hdr_end) {
    std::vector<int64_t> seg{w == 0 ? (int64_t)hdr_end : 0};
    const int64_t wstream = (int64_t)mem[cut[w]].off;
    for (size_t i = cut[w]; i < cut[w + 1]; i++) { const int64_t s = carry + ((int64_t)mem[i].off - wstream); if (s > seg[0]) seg.push_back(s); }
    return seg;
}

NameTable bam_name_table(const char *blob, const int64_t *name_off, int64_t n) {
    size_t cap = 2;
    while (cap < 2 * (size_t)n) cap <<= 1;
    NameTable t{std::vector<uint64_t>(cap, 0), std::vector<int32_t>(cap, -1), std::vector<int64_t>(cap, 0)};
    for (int64_t i = 0; i < n; i++) {
        const uint8_t *p = (const uint8_t *)blob + name_off[i];
        const uint32_t len = (uint32_t)(name_off[i + 1] - name_off[i]);
        const uint64_t h = sq::name_hash(p, len);
        size_t k = h & (cap - 1);
        for (; t.len[k] >= 0; k = (k + 1) & (cap - 1))
            if (t.hash[k] == h && (uint32_t)t.len[k] == len && memcmp(blob + t.off[k], p, len) == 0) break;
        t.hash[k] = h; t.len[k] = (int32_t)len; t.off[k] = name_off[i];
    }
    return t;
}

}  // namespace sqh
// test hook: opens a BAM file with the front end; *n_rec = records, *per_member = 1 when the member-by-member walk was proven
extern "C" int sqh_probe_bam(const char *path, int64_t *n_rec, int32_t *per_member) {
    sqh::BamTable t;
    std::string err;
    if (!path || !t.open(path, err)) return -1;
    if (n_rec) *n_rec = (int64_t)t.n_rec();
    if (per_member) *per_member = t.walked_per_member ? 1 : 0;
    return 0;
}
namespace sqh {
AlnSource BamTable::source() const {
    AlnSource s;
    s.n_rec = n_rec();
    const BamTable *t = this;
    s.at = [t](uint64_t r) {
        Alignment a;
        a.ref_id = t->ref_id[r]; a.pos = t->pos[r]; a.mate_ref_id = t->mate_ref_id[r]; a.mate_pos = t->mate_pos[r];
        a.flag = t->flag[r]; a.mapq = t->mapq[r];
        a.tag_xa = t->tags[r] & 1; a.tag_ih = t->tags[r] & 2; a.ih_value = t->ih[r];
        a.cigar = t->cigar.data() + t->cigar_off[r]; a.n_cigar = (uint32_t)(t->cigar_off[r + 1] - t->cigar_off[r]);
        a.l_seq = (uint32_t)(t->seq_off[r + 1] - t->seq_off[r]);
        a.seq = t->seq.data() + t->seq_off[r]; a.qual = t->qual.data() + t->seq_off[r];
        return a;
    };
    s.name = [t](uint64_t r) { return std::string(t->names.data() + t->name_off[r], (size_t)(t->name_off[r + 1] - t->name_off[r])); };
    s.name_into = [t](uint64_t r, char *buf) { const size_t len = (size_t)(t->name_off[r + 1] - t->name_off[r]); memcpy(buf, t->names.data() + t->name_off[r], len); return len; };
    return s;
}

}  // namespace sqh
