"""The rules of the device BAM decode (sq_inflate.cuh, sq_bam.cuh; sqg_load_concordant_bam) stepped on the CPU by
tests/emul/emul_bam.cpp: inflate against zlib on random data x levels x strategies and on damaged streams, and the windowed
record boundaries + decode against the host front end (sqh_open_bam_case) on every layout.  Plus sqh_open_bam_chimeric."""
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

from squid_b200 import api
from tests import bam_device_cases as cases
from tests import common


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return cases.build_emul_bam(tmp_path_factory.mktemp("emul_bam"))


def _payloads(seed):
    rng = random.Random(seed)
    text = b" ".join(rng.choice([b"ACGT", b"chr1", b"q12345/1", b"IIIIIIII", b"\x00\x01", b"MD:Z:50"]) for _ in range(20000))
    return {"random": bytes(rng.getrandbits(8) for _ in range(70000)), "text": text, "runs": b"A" * 30000 + b"CA" * 9000 + bytes(range(256)) * 40,
            "short": b"x", "mixed": bytes(rng.getrandbits(8) for _ in range(3000)) + text[:50000]}


def _inflate(emul, data: bytes, d):
    p, o = os.path.join(d, "in.bgzf"), os.path.join(d, "out.bin")
    open(p, "wb").write(data)
    r = subprocess.run([emul, "inflate", p, o], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return int(r.stdout.split()[1]), open(o, "rb").read()


@pytest.mark.parametrize("strategy", sorted(cases.STRATEGIES))
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_inflate_matches_zlib(emul, tmp_path, level, strategy):
    """Stored, fixed-Huffman and dynamic-Huffman blocks, overlapping matches of every distance: the stepped warp inflate and its
    sliced CRC32 give zlib's bytes."""
    for name, data in _payloads(level * 7 + len(strategy)).items():
        bg = cases.bgzf_cut(data, range(0xFF00, len(data), 0xFF00), level, cases.STRATEGIES[strategy])
        status, out = _inflate(emul, bg, str(tmp_path))
        assert status == 0 and out == data, name


def _zlib_verdict(cdata: bytes, isize: int, crc: int) -> int:
    """What the host inflater decides about one member: 0 ok, 1 corrupt deflate stream (ISIZE mismatch included), 2 CRC."""
    try:
        d = zlib.decompressobj(-15)
        out = d.decompress(cdata, isize + 1)
    except zlib.error:
        return 1
    if not d.eof or len(out) != isize:
        return 1
    return 0 if (zlib.crc32(out) & 0xFFFFFFFF) == crc else 2


@pytest.mark.parametrize("strategy", ["default", "fixed", "huffman"])
def test_inflate_refuses_what_zlib_refuses(emul, tmp_path, strategy):
    """Single-member files with one, two or eight bytes of the deflate payload or the trailer changed: the stepped inflate
    reaches zlib's verdict on every one (corrupt, CRC mismatch or, where the damage is harmless, accepted)."""
    rng = random.Random(hash(strategy) & 0xFFFF)
    data = _payloads(3)["mixed"][:40000]
    good = cases.member(data, 6, cases.STRATEGIES[strategy])
    seen = set()
    for trial in range(150):
        m = bytearray(good)
        for _ in range(rng.choice([1, 2, 8])):
            k = rng.randrange(18, len(m) - 4 if trial % 5 else len(m))  # mostly the payload, sometimes the CRC / ISIZE too
            m[k] ^= 1 << rng.randrange(8)
        isize, crc = int.from_bytes(m[-4:], "little"), int.from_bytes(m[-8:-4], "little")
        if isize > 65536:
            continue
        want = _zlib_verdict(bytes(m[18:-8]), isize, crc)
        status, _ = _inflate(emul, bytes(m), str(tmp_path))
        assert status == want, (trial, status, want)
        seen.add(want)
    assert 1 in seen and 2 in seen


def _decode(emul, bam, case, d, window=1 << 30, env=None):
    bp, op = cases.names_files(case, d)
    o = case.options
    r = subprocess.run([emul, "decode", bam, bp, op, str(o.phred33), str(o.min_phred), str(window), d], capture_output=True, text=True)
    assert r.returncode in (0, 3), r.stdout + r.stderr
    if r.returncode == 3:
        return r.stdout.strip(), None
    info = dict(zip(r.stdout.split()[0::2], map(int, r.stdout.split()[1::2])))
    return info, {k: np.fromfile(os.path.join(d, k + ".bin"), dt) for k, dt in api.BATCH_DTYPES.items()}


def _assert_batch(want, got):
    for k in api.BATCH_DTYPES:
        assert np.array_equal(want.a[k], got[k]), k


@pytest.fixture(scope="module")
def case6k(tmp_path_factory):
    d = tmp_path_factory.mktemp("case6k")
    cp, hp, conc, chim, info = common.write_case(str(d), 6000, 17, 0.05)
    from squid_b200 import bamio
    hb = str(d / "chim.bam")
    bamio.write_bam(hb, chim)
    return d, conc, hb


@pytest.mark.parametrize("window", [1 << 30, 20000])
@pytest.mark.parametrize("layout", ["htslib", "straddle_997", "straddle_1500", "straddle_ff00", "uncompressed"])
def test_decode_matches_host(emul, case6k, tmp_path, layout, window):
    """Windowed boundaries (20 kB windows: records straddle windows, tails carried) and the record decode against the batch the
    host front end packs from the same file."""
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(conc)[layout])
    host = api.HostCase(cb, hb, bam=True)
    dev = api.HostCase(cb, hb, bam=True, header_only=True)
    info, got = _decode(emul, cb, dev, str(tmp_path), window)
    assert got is not None, info
    _assert_batch(host.batch, got)
    assert info["windows"] >= (2 if window < 1 << 20 else 1)


def test_decode_adversarial_member_start(emul, case6k, tmp_path):
    """A member that starts inside a B-array tag whose bytes are a chain of valid-looking records: the speculative start is
    wrong, the proof rejects it, a repair round walks the member again from its true entry, and the batch is still the host's."""
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.adversarial(conc))
    host = api.HostCase(cb, hb, bam=True)
    info, got = _decode(emul, cb, api.HostCase(cb, hb, bam=True, header_only=True), str(tmp_path))
    assert got is not None, info
    _assert_batch(host.batch, got)
    assert info["rounds"] > 0


@pytest.mark.parametrize("opts", [{}, dict(min_phred=50), dict(phred33=0, min_phred=10)])
def test_decode_known_answers(emul, tmp_path, opts):
    """Clips, I/D/N/=/X, poly-A/T, low-quality runs, missing qualities, every IH type, XA, ChimName with and without /1 /2."""
    from squid_b200 import bamio, sqmb
    t, ch = cases.known_answer_tables()
    cb, hb = str(tmp_path / "c.bam"), str(tmp_path / "h.bam")
    bamio.write_bam(cb, t, block=64); bamio.write_bam(hb, ch)
    host = api.HostCase(cb, hb, bam=True, **opts)
    info, got = _decode(emul, cb, api.HostCase(cb, hb, bam=True, header_only=True, **opts), str(tmp_path))
    assert got is not None, info
    _assert_batch(host.batch, got)
    assert (got["aux"] & 8).any() and (got["aux"] & 2).any()


def test_open_bam_chimeric_matches_full_open(case6k, tmp_path):
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(conc)["straddle_997"])
    full, part = api.HostCase(cb, hb, bam=True), api.HostCase(cb, hb, bam=True, header_only=True)
    for k in full.chimeric.a:
        assert np.array_equal(full.chimeric.a[k], part.chimeric.a[k]), k
    assert full.config == part.config and np.array_equal(full.ref_len, part.ref_len)
    assert part.batch.n_rec == 0 and part.batch.a["blk_off"].tolist() == [0]
    blob, off = part.chim_names()
    names = {blob[a:b] for a, b in zip(off[:-1], off[1:])}
    assert b"" in names and len(names) == off.shape[0] - 1 == full.chim_names()[1].shape[0] - 1


def test_decode_refuses_damage_like_host(emul, case6k, tmp_path):
    """Each damage of test_cpu_bam.py::test_damaged_files_fail_loudly: the stepped decode gives the host's message."""
    from squid_b200 import bamio
    d, conc, hb = case6k
    good = bamio.bgzf_compress(bamio.bam_bytes(conc), 4096)
    for k, bad in enumerate((good[: len(good) // 2], good[:200] + bytes([good[200] ^ 0x55]) + good[201:], zlib.compress(bamio.bam_bytes(conc)),
                             b"BAM\1" + b"\xff" * 40)):
        p = str(tmp_path / ("x%d.bam" % k))
        open(p, "wb").write(bad)
        with pytest.raises(api.SquidB200Error) as e:
            api.HostCase(p, hb, bam=True)
        try:
            case = api.HostCase(p, hb, bam=True, header_only=True)
        except api.SquidB200Error:
            case = api.HostCase(hb, hb, bam=True, header_only=True)  # the header itself is refused: options and names of any case
        info, got = _decode(emul, p, case, str(tmp_path))
        assert got is None and info.endswith(str(e.value).split(": ", 1)[1]), (k, info, str(e.value))
