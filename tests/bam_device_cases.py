"""BAM files for the device decode (sqg_load_concordant_bam) and its CPU stepping: the layouts, compressors and adversarial
member cuts that tests/test_cpu_bam_device.py and tests/test_gpu_bam_device.py both run."""
import os
import struct
import subprocess
import zlib

import numpy as np

from squid_b200 import bamio, sqmb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman": zlib.Z_HUFFMAN_ONLY, "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}


def member(chunk: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    cd = c.compress(chunk) + c.flush()
    return b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(cd) + 25) + cd + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk))


def bgzf_cut(data: bytes, cuts, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY) -> bytes:
    """BGZF members cut at the given stream offsets (plus the EOF marker)."""
    edges = [0] + sorted(c for c in set(cuts) if 0 < c < len(data)) + [len(data)]
    out = bytearray()
    for a, b in zip(edges[:-1], edges[1:]):
        for o in range(a, b, 0xFF00):  # no member holds more than 64 KiB
            out += member(data[o:min(b, o + 0xFF00)], level, strategy)
    return bytes(out) + bamio._BGZF_EOF


def layouts(t: sqmb.AlnTable, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY) -> dict:
    """The same table as BAM bytes in every layout the decode has to handle."""
    parts = bamio.bam_parts(t)
    raw = b"".join(parts)
    return {"htslib": bamio.bgzf_compress_records(parts, 0xFF00, level) if strategy == zlib.Z_DEFAULT_STRATEGY else None,
            "straddle_997": bgzf_cut(raw, range(997, len(raw), 997), level, strategy),
            "straddle_1500": bgzf_cut(raw, range(1500, len(raw), 1500), level, strategy),
            "straddle_ff00": bgzf_cut(raw, range(0xFF00, len(raw), 0xFF00), level, strategy),
            "uncompressed": raw}


def adversarial(t: sqmb.AlnTable, level: int = 6) -> bytes:
    """Record 20 carries a B-array tag whose bytes are copies of ten real records (block sizes included): a chain of records that
    look valid in every field.  Members are cut every 997 bytes, and one cut falls exactly on the third record inside the array,
    so that member's speculative start is a false one and only the proof against its predecessor's exit can reject it."""
    parts = bamio.bam_parts(t)
    fake = b"".join(parts[30:40])
    body = parts[20][4:] + b"ZBBC" + struct.pack("<I", len(fake)) + fake
    parts[20] = struct.pack("<i", len(body)) + body
    raw = b"".join(parts)
    array_at = sum(len(p) for p in parts[:20]) + len(parts[20]) - len(fake)
    cut = array_at + len(parts[30]) + len(parts[31])
    cuts = [c for c in range(997, len(raw), 997) if abs(c - cut) > 40] + [cut]
    return bgzf_cut(raw, cuts, level)


def known_answer_tables():
    """The hand-written records of tests/test_cpu_bam.py::test_bam_known_answers, plus every IH type and a ChimName-shaped name."""
    F = sqmb
    recs = [
        dict(ref_id=0, pos=100, cigar="5H10S40M5I20M2D10M1000N15M", flag=F.FLAG_PAIRED | F.FLAG_FIRST | F.FLAG_MATE_REVERSE, mate_ref_id=0, mate_pos=1300,
             seq="C" * 10 + "G" * 75 + "A" * 15, qual="!" * 13 + "I" * 87, name_id=7, ih=1),
        dict(ref_id=0, pos=1300, cigar="30=5X30M35S", flag=F.FLAG_PAIRED | F.FLAG_SECOND | F.FLAG_REVERSE, mate_ref_id=0, mate_pos=100,
             seq="ACGT" * 25, qual="I" * 100, name_id=7, xa=True, ih=3, name_suffix=True),
        dict(ref_id=1, pos=5, cigar="100M", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=400, lowrun=12, polya=1, name_id=9, mapq=3),
        dict(ref_id=1, pos=900, cigar="95M", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=1400, seq="A" * 71 + "C" * 23 + "A", qual="I" * 95, name_id=11),
        dict(ref_id=1, pos=950, cigar="95M", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=1400, seq="A" * 71 + "C" * 23 + "G", qual="I" * 95, name_id=12),
        dict(ref_id=1, pos=960, cigar="50M", flag=F.FLAG_PAIRED | F.FLAG_SECOND, mate_ref_id=1, mate_pos=10, name_id=1, ih=2),
        dict(ref_id=1, pos=970, cigar="50M", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=10, name_id=1, ih=255, name_suffix=True),
        dict(ref_id=1, pos=980, cigar="20M10D20M", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=10, name_id=13, ih=5),
        dict(ref_id=1, pos=990, cigar="10S30M10S", flag=F.FLAG_PAIRED | F.FLAG_FIRST | F.FLAG_REVERSE, mate_ref_id=1, mate_pos=10, name_id=14, ih=200),
    ]
    t = F.from_records([5000, 3000], recs)
    ch = F.from_records([5000, 3000], [dict(ref_id=0, pos=10, cigar="60M40S", flag=F.FLAG_PAIRED | F.FLAG_FIRST, mate_ref_id=1, mate_pos=50, name_id=1),
                                       dict(ref_id=1, pos=700, cigar="60S40M", flag=F.FLAG_PAIRED | F.FLAG_FIRST | F.FLAG_REVERSE, mate_ref_id=1, mate_pos=50, name_id=1),
                                       dict(ref_id=1, pos=50, cigar="100M", flag=F.FLAG_PAIRED | F.FLAG_SECOND | F.FLAG_REVERSE, mate_ref_id=0, mate_pos=10, name_id=1)])
    return t, ch


def random_cigar_table(seed: int, n_reads: int = 1500):
    """Records with random CIGARs over all nine ops: leading / trailing I, D, X, P and clips, H and S between blocks, blocks opened
    by M or =, N runs, A/T fractions of blocks at and around 3/4, both strands and mates, explicit bases and qualities (runs of
    qualities in narrow random bands, so that every threshold cuts them somewhere) and synthesised ones.  Within the packer's
    limits: at most 16 blocks and TotalLen <= 65535.  Read i sits alone in its own 200 kb stretch, so no two reads share a front
    position."""
    import random
    F = sqmb
    rng = random.Random(seed)
    ln = lambda lo, hi: rng.randint(lo, hi)

    def cigar(p):  # p: P may follow the first M / =, where it can fall inside a block
        ops = []
        for _ in range(rng.choice([0, 0, 1, 2])):  # leading clips and ops outside any block
            ops.append((rng.choice("HSIDXP"), ln(1, 12)))
        for b in range(ln(1, rng.choice([3, 8, 16]))):
            if b:
                for _ in range(ln(1, 3)):  # separators, with strays that fall outside the blocks
                    o = rng.choice("SHNNNIDX" + p)
                    ops.append((o, ln(1, 400) if o == "N" else ln(1, 15)))
            ops.append((rng.choice("MM="), ln(1, 60)))
            for _ in range(rng.choice([0, 0, 1, 2, 3])):
                ops.append((rng.choice("MID=X" + p), ln(1, 20)))
        for _ in range(rng.choice([0, 0, 1, 2])):
            ops.append((rng.choice("HSIDX" + p), ln(1, 12)))
        return "".join("%d%s" % (l, o) for o, l in ops), ops

    def windows(ops):  # the read windows the poly-A/T test reads, as decode_alignment walks the CIGAR
        out, rp, hard, i = [], 0, 0, 0
        while i < len(ops):
            o, l = ops[i]
            if o in "SH":
                rp += l
                hard += l if o == "H" else 0
            elif o in "M=":
                j, span = i, 0
                while j < len(ops) and ops[j][0] not in "SHN":
                    span += ops[j][1] if ops[j][0] != "D" else 0
                    j += 1
                out.append((rp - hard, span))
                rp += span
                i = j - 1
            i += 1
        return out

    recs = []
    for i in range(n_reads):
        mates = [F.FLAG_FIRST, F.FLAG_SECOND] if rng.random() < 0.8 else [rng.choice([F.FLAG_FIRST, F.FLAG_SECOND])]
        for m, mate in enumerate(mates):
            # the first block of a read's first record always stays: a read left without blocks has no place in the loader's sort
            synth = rng.random() < 0.3
            # A P inside a block widens its read span past the bases the block covers, so a synthesised poly-A/T block would
            # be all A/T for the packer but not for a reader of the materialised bases: synthesised records keep P outside blocks.
            cig, ops = cigar("" if synth else "P")
            lseq = sum(l for o, l in ops if o in "MIS=X")
            flag = F.FLAG_PAIRED | mate | (F.FLAG_REVERSE if rng.random() < 0.5 else 0) | (F.FLAG_MATE_REVERSE if rng.random() < 0.5 else 0)
            r = dict(ref_id=i % 2, pos=1000 + (i // 2) * 200000 + (0 if mate == F.FLAG_FIRST else 20000) + ln(0, 999), cigar=cig, flag=flag,
                     mate_ref_id=i % 2, mate_pos=1000 + (i // 2) * 200000, mapq=rng.choice([0, 3, 60, 255]), name_id=i,
                     name_suffix=rng.random() < 0.2, xa=rng.random() < 0.1)
            if rng.random() < 0.3:
                r["ih"] = rng.choice([0, 1, 2, 200])
            if synth:
                r["lowrun"] = rng.choice([0, ln(0, lseq), lseq, lseq + 5])
                r["polya"] = rng.getrandbits(8) & (0xEE if m == 0 else 0xFF)
            else:
                seq = [rng.choice("CGNCGT") for _ in range(lseq)]
                for b, (a, span) in enumerate(windows(ops)):
                    if m == 0 and b == 0:
                        seq[a:a + span] = [rng.choice("CG") for _ in seq[a:a + span]]
                        continue
                    base = rng.choice("AaTt")
                    k = max(0, (3 * span + 3) // 4 + rng.choice([-2, -1, -1, 0, 0, 0, 1, 1]) if rng.random() < 0.7 else rng.choice([0, span]))
                    for p in rng.sample(range(span), min(k, span)):
                        if 0 <= a + p < lseq:
                            seq[a + p] = base
                qual = []
                while len(qual) < lseq:
                    lo = ln(33, 120)
                    qual += [chr(ln(lo, lo + 4)) for _ in range(ln(1, 30))]
                r["seq"], r["qual"] = "".join(seq), "".join(qual[:lseq])
            recs.append(r)
    recs.sort(key=lambda r: (r["ref_id"], r["pos"]))
    return F.from_records([1 << 30, 1 << 30], recs)


def build_emul_bam(out_dir) -> str:
    """Compiles tests/emul/emul_bam.cpp into `out_dir` (not into the repository tree, which may be read-only)."""
    out = os.path.join(str(out_dir), "emul_bam")
    srcs = ["tests/emul/emul_bam.cpp", "squid_b200/csrc/host/bam.cpp", "squid_b200/csrc/host/readrec.cpp", "squid_b200/csrc/host/chimeric.cpp"]
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-fopenmp", "-I", "include", "-I", "squid_b200/csrc", "-o", out] + srcs + ["-lz", "-lpthread"],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def names_files(case, d):
    blob, off = case.chim_names()
    bp, op = os.path.join(d, "names.blob"), os.path.join(d, "names.off")
    open(bp, "wb").write(blob)
    np.asarray(off, np.int64).tofile(op)
    return bp, op
