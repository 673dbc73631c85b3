"""The concordant BAM decoded on the device (sqg_load_concordant_bam, SegmentGraph.load_concordant_bam): the resident batch it
leaves, fetched with sqg_download_concordant, equals what sqh_open_bam_case packs from the same file -- all 15 arrays -- on every
layout, compressor, window size and the known-answer records; the phases after it equal the reference; damaged files are refused
with the host's code and message and leave the context usable."""
import concurrent.futures
import os
import zlib

import numpy as np
import pytest

from squid_b200 import api, bamio, synth
from tests import bam_device_cases as cases
from tests import common

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def case6k(tmp_path_factory):
    d = tmp_path_factory.mktemp("dev6k")
    cp, hp, conc, chim, info = common.write_case(str(d), 6000, 17, 0.05, synth.GRCH38_LEN)
    hb = str(d / "chim.bam")
    bamio.write_bam(hb, chim)
    return d, conc, hb


def _device_batch(cb, hb, window_mb=None, **opts):
    case = api.HostCase(cb, hb, bam=True, header_only=True, **opts)
    g = api.SegmentGraph(case.config, case.ref_len)
    old = os.environ.get("SQG_BAM_WINDOW_MB")
    if window_mb is not None:
        os.environ["SQG_BAM_WINDOW_MB"] = str(window_mb)
    try:
        g.load_concordant_bam(cb, case)
    finally:
        if window_mb is not None:
            if old is None:
                del os.environ["SQG_BAM_WINDOW_MB"]
            else:
                os.environ["SQG_BAM_WINDOW_MB"] = old
    return g, g.download_concordant()


def _assert_same(host, got):
    assert host.n_rec == got.n_rec and host.n_blk == got.n_blk
    for k in api.BATCH_DTYPES:
        assert np.array_equal(host.a[k], got.a[k]), k


@pytest.mark.parametrize("layout", ["htslib", "straddle_997", "straddle_1500", "straddle_ff00", "uncompressed"])
def test_layouts(case6k, tmp_path, built_lib, layout):
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(conc)[layout])
    g, got = _device_batch(cb, hb)
    _assert_same(api.HostCase(cb, hb, bam=True).batch, got)
    assert g.stat("bam_windows") == 1 and g.stat("bam_members") > 0
    for ph in ("bam_h2d", "bam_inflate", "bam_records", "bam_decode"):
        assert g.phase_ms(ph) >= 0, ph


@pytest.mark.parametrize("level,strategy", [(0, "default"), (1, "default"), (6, "default"), (9, "default"), (6, "fixed"), (6, "huffman"), (6, "rle")])
def test_compressors(case6k, tmp_path, built_lib, level, strategy):
    """Stored (level 0), fixed-Huffman and dynamic-Huffman blocks."""
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(conc, level, cases.STRATEGIES[strategy])["straddle_1500"])
    _assert_same(api.HostCase(cb, hb, bam=True).batch, _device_batch(cb, hb)[1])


@pytest.mark.parametrize("layout", ["htslib", "straddle_997", "uncompressed"])
def test_windows_of_1mb(case6k, tmp_path, built_lib, layout):
    """1 MB windows: records straddle windows and the tail of each is carried to the front of the next."""
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(conc)[layout])
    g, got = _device_batch(cb, hb, window_mb=1)
    _assert_same(api.HostCase(cb, hb, bam=True).batch, got)
    assert g.stat("bam_windows") >= 2


@pytest.mark.parametrize("opts", [{}, dict(min_phred=50), dict(phred33=0, min_phred=10)])
def test_known_answers(tmp_path, built_lib, opts):
    """Clips, I/D/N/=/X, poly-A/T, low-quality runs, missing qualities, every IH type, XA, ChimName with and without /1 /2."""
    t, ch = cases.known_answer_tables()
    cb, hb = str(tmp_path / "c.bam"), str(tmp_path / "h.bam")
    bamio.write_bam(cb, t, block=64); bamio.write_bam(hb, ch)
    host = api.HostCase(cb, hb, bam=True, **opts).batch
    got = _device_batch(cb, hb, **opts)[1]
    _assert_same(host, got)
    assert (got.a["aux"] & 8).any() and (got.a["aux"] & 2).any()


@pytest.mark.parametrize("opts", [{}, dict(phred33=0, min_phred=70)])
def test_random_cigars(tmp_path, built_lib, opts):
    """Random CIGARs over all nine ops (bam_device_cases.random_cigar_table), records straddling members, 1 MB windows."""
    t = cases.random_cigar_table(2024)
    cb = str(tmp_path / "c.bam")
    open(cb, "wb").write(cases.layouts(t)["straddle_997"])
    g, got = _device_batch(cb, cb, window_mb=1, **opts)
    _assert_same(api.HostCase(cb, cb, bam=True, **opts).batch, got)


def test_adversarial_member_start(case6k, tmp_path, built_lib):
    """A member that starts inside a B-array tag whose bytes form a chain of valid-looking records."""
    d, conc, hb = case6k
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.adversarial(conc))
    g, got = _device_batch(cb, hb)
    _assert_same(api.HostCase(cb, hb, bam=True).batch, got)
    assert g.stat("bam_repair_rounds") > 0


def tiled_bam(t, copies: int, level: int = 1, cut: int = 0xFF00, threads: int = 16) -> bytes:
    """The records of `t` repeated `copies` times behind one header, cut into members every `cut` bytes (records straddle them)
    and compressed on `threads` threads (zlib releases the GIL)."""
    parts = bamio.bam_parts(t)
    raw = parts[0] + b"".join(parts[1:]) * copies
    edges = list(range(0, len(raw), cut)) + [len(raw)]
    with concurrent.futures.ThreadPoolExecutor(threads) as ex:
        members = list(ex.map(lambda ab: cases.member(raw[ab[0]:ab[1]], level), zip(edges[:-1], edges[1:])))
    return b"".join(members) + bamio._BGZF_EOF


def test_scale_one_million_pairs(tmp_path, built_lib):
    conc, chim, _ = synth.make_case(125000, ref_len=synth.CHR17_LEN, seed=5, disc_frac=0.02)
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    open(cb, "wb").write(tiled_bam(conc, 9))
    bamio.write_bam(hb, chim)
    host = api.HostCase(cb, hb, bam=True).batch
    assert host.n_rec >= 2_000_000
    _assert_same(host, _device_batch(cb, hb)[1])


def test_end_to_end_matches_reference(tmp_path, built_lib, ref_oracle):
    """The case of test_gpu_parity.py::test_bam_input_matches_reference through load_concordant_bam."""
    from oracle import pyref
    cp, hp, conc, chim, info = common.write_case(str(tmp_path), 8000, 19, 0.03)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, conc, block=8191); bamio.write_bam(hb, chim)
    case = api.HostCase(cb, hb, bam=True, header_only=True)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant_bam(cb, case)
    nodes = g.BuildNode_STAR(case.chimeric)
    edges = g.BuildEdges()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": case.chimeric.block_table()}
    common.assert_same(ref, got)
    assert g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref)) == pyref.support_map(ref)


def test_damaged_files_then_a_good_one(case6k, tmp_path, built_lib):
    """Each damage of test_cpu_bam.py::test_damaged_files_fail_loudly: the host's error code and message, then the same context
    loads a good file correctly."""
    d, conc, hb = case6k
    good = bamio.bgzf_compress(bamio.bam_bytes(conc), 4096)
    gp = str(tmp_path / "good.bam")
    open(gp, "wb").write(good)
    case = api.HostCase(gp, hb, bam=True, header_only=True)
    g = api.SegmentGraph(case.config, case.ref_len)
    damages = (good[: len(good) // 2], good[:200] + bytes([good[200] ^ 0x55]) + good[201:], zlib.compress(bamio.bam_bytes(conc)), b"BAM\1" + b"\xff" * 40)
    for k, bad in enumerate(damages):
        p = str(tmp_path / ("bad%d.bam" % k))
        open(p, "wb").write(bad)
        with pytest.raises(api.SquidB200Error) as host_err:
            api.HostCase(p, hb, bam=True)
        with pytest.raises(api.SquidB200Error) as dev_err:
            g.load_concordant_bam(p, case)
        assert (dev_err.value.code, str(dev_err.value)) == (host_err.value.code, str(host_err.value)), k
    with pytest.raises(api.SquidB200Error):
        g.load_concordant_bam(str(tmp_path / "missing.bam"), case)
    g.load_concordant_bam(gp, case)
    _assert_same(api.HostCase(gp, hb, bam=True).batch, g.download_concordant())
    g.BuildNode_STAR(case.chimeric)
