"""The classification pass (sq_phase1.cuh: k_classify_tiles, k_tile_scan, k_finish_gaps, k_compact_lists) against the
restatement's per-record preamble of BuildNode_STAR (pyref.run_restate_classify), reduced in numpy to the pass's own outputs
(common.expected_phase1).  The stream families of common.stream_families reach the paths a synthetic case does not: runs of
more than 32 gate-failing records in front of a tile (the look-back over the tiles' gate words), tiles without a gate-passing
record, unmapped records and tiles across chromosomes (the one-thread literal branch), duplicates whose previous gate-passing
record lies before the tile (classify_from_hbm), first blocks of 65535 bp and more, tiles too dense to stage, and more
coverage-gap candidates than the first candidate buffer holds (the retry of run_classify)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["cls", "first_len", "gap_rec", "gap_key", "pc_rec", "dp_rec", "okmax_excl", "ccmax", "cov_nq", "cov_qmax", "qstage_key", "qstage_end"]
STATS = ["lmax", "first_kept", "classify_attempts", "gap_records", "partial_records", "displaced_records"]


@pytest.fixture(scope="module")
def streams(tmp_path_factory):
    """{family: (conc path, chim path, concordant AlnTable, expected phase-1 outputs)}"""
    from oracle import pyref
    d = tmp_path_factory.mktemp("streams")
    out = {}
    for name, (cp, hp, tab) in common.write_stream_families(d).items():
        rc = pyref.run_restate_classify(cp, hp, os.path.join(os.path.dirname(cp), "rc"))
        out[name] = (cp, hp, tab, common.expected_phase1(rc, tab.ref_id, tab.pos))
    return out


def _graph(case, load):
    from squid_b200 import api
    g = api.SegmentGraph(case.config, case.ref_len)
    keep = None
    if load == "host":
        g.load_concordant(case.batch)
    elif load == "wire":
        g.load_concordant_wire(api.WireBatch(case.batch))
    else:
        from tests.test_gpu_set_nodes import _unaligned_device_batch
        st, keep = _unaligned_device_batch(case)
        g.attach_concordant_device(st, keep)
    return g, keep


def dumps(g) -> dict:
    """Every phase-1 array and the classification stats of a context (before BuildNode_STAR)."""
    d = {k: g.classify_dump(k) for k in NAMES}
    d.update({k: g.stat(k) for k in STATS})
    return d


def _wire_dumps_in_subprocess(cp, hp, env, out_npz):
    """SQG_WIRE_CLASSIFY and SQG_WIRE_CHUNKS are read once per process: those legs load the wire batch in a process of their own."""
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from squid_b200 import api\n"
            "from tests import test_gpu_classify as t\n"
            "c = api.HostCase(%r, %r)\n"
            "g = api.SegmentGraph(c.config, c.ref_len)\n"
            "g.load_concordant_wire(api.WireBatch(c.batch))\n"
            "d = t.dumps(g)\n"
            "np.savez(%r, **{k: np.asarray(v) for k, v in d.items()})\n") % (ROOT, cp, hp, out_npz)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    z = np.load(out_npz)
    return {k: (z[k] if z[k].ndim else int(z[k])) for k in z.files}


def assert_phase1(want, got, where=""):
    for k in ("cls", "first_len", "gap_rec", "gap_key", "pc_rec", "dp_rec", "okmax_excl", "ccmax", "cov_nq", "cov_qmax"):
        a, b = np.asarray(want[k]), np.asarray(got[k])
        assert a.shape == b.shape, "%s %s: shape %s vs %s" % (where, k, a.shape, b.shape)
        bad = np.flatnonzero(a != b.astype(a.dtype))
        assert bad.size == 0, "%s %s differs at %d entries, first %s: restatement %s device %s" % (where, k, bad.size, bad[:5], a[bad[:5]], b[bad[:5]])
    for t, (wk, we) in enumerate(zip(want["qstage_key"], want["qstage_end"])):  # tile t owns [t * 512, t * 512 + cov_nq[t])
        s = slice(t * common.TILE, t * common.TILE + wk.shape[0])
        assert np.array_equal(got["qstage_key"][s], wk) and np.array_equal(got["qstage_end"][s], we), "%s qstage tile %d" % (where, t)
    assert got["lmax"] == want["lmax"] and got["first_kept"] == want["first_kept"], where
    assert got["gap_records"] == want["gap_rec"].shape[0] and got["partial_records"] == want["pc_rec"].shape[0], where
    assert got["displaced_records"] == want["dp_rec"].shape[0], where


@pytest.mark.parametrize("family", common.FAMILY_STREAMS)
@pytest.mark.parametrize("load", ["host", "wire", "unaligned"])
def test_classify_matches_restatement(streams, family, load, built_lib):
    from squid_b200 import api
    cp, hp, tab, want = streams[family]
    case = api.HostCase(cp, hp)
    g, keep = _graph(case, load)
    got = dumps(g)
    assert_phase1(want, got, "%s/%s" % (family, load))
    assert got["classify_attempts"] == 1


@pytest.mark.parametrize("family", ["filtered_runs", "dup_shapes", "many_chr", "unmapped_tail", "long_first_block", "dense_tiles"])
@pytest.mark.parametrize("env", [{"SQG_WIRE_CLASSIFY": "0"}, {"SQG_WIRE_CHUNKS": "3"}, {"SQG_WIRE_CHUNKS": "7"}], ids=["no_pre_classify", "chunks3", "chunks7"])
def test_classify_wire_settings(streams, family, env, tmp_path, built_lib):
    """The wire upload with the tile kernel run after the upload, and with 3 or 7 chunks, so that chunk ends fall inside the stream
    and a chunk's last tile waits for the next chunk."""
    cp, hp, tab, want = streams[family]
    got = _wire_dumps_in_subprocess(cp, hp, env, str(tmp_path / "d.npz"))
    assert_phase1(want, got, "%s/%s" % (family, env))


def test_paths_reached(streams, built_lib):
    """Each path the families exist for occurs in them (otherwise the comparisons above do not test it)."""
    from squid_b200 import api
    T = common.TILE
    # a tile whose first gate-passing record follows a run of more than 32 gate-failing records that crosses its start
    cls = streams["filtered_runs"][3]["cls"]
    gate = np.flatnonzero(cls & common.CLS_GATE)
    nt = (cls.shape[0] + T - 1) // T
    lookback = empty = 0
    for t in range(nt):
        inside = gate[(gate >= t * T) & (gate < (t + 1) * T)]
        before = gate[gate < t * T]
        if inside.size == 0:
            empty += 1
        elif t > 0 and (before.size == 0 or t * T - before[-1] > 32):
            lookback += 1
    assert lookback >= 4 and empty >= 3, (lookback, empty)
    # multi-chromosome tiles and tiles that start with an unmapped record: the one-thread literal branch
    for fam in ("many_chr", "unmapped_tail"):
        cp, hp, tab, want = streams[fam]
        g, _ = _graph(api.HostCase(cp, hp), "host")
        assert (g.classify_dump("ccmax") == common.K_CC_WALK_TILE).sum() >= 3, fam
    cp, hp, tab, want = streams["long_first_block"]
    g, _ = _graph(api.HostCase(cp, hp), "host")
    assert (g.classify_dump("first_len") == 65535).sum() >= 30 and g.stat("lmax") == 70100
    # a tile with more blocks than a tile stages (sq_stream.cuh kTileBlkCap): classified from HBM
    case = api.HostCase(*streams["dense_tiles"][:2])
    off = case.batch.a["blk_off"].astype(np.int64)
    n = case.batch.n_rec
    per_tile = np.array([off[min((t + 1) * T, n)] - off[t * T] for t in range((n + T - 1) // T)])
    assert (per_tile > 1152).sum() >= 1, per_tile.max()


@pytest.mark.parametrize("family", common.FAMILY_STREAMS)
def test_stream_families_end_to_end(streams, family, tmp_path, built_lib):
    """Segments, Support, AvgDepth, edges, trimmed chimeric blocks and the breakpoint coverage of a uniform list against the
    restatement, on every stream family."""
    from oracle import pyref
    cp, hp, tab, _ = streams[family]
    want = pyref.Restated.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp)
    common.assert_same(want, got)
    bps = common.bp_families(tab.ref_len, want["nodes"], tab, 5)["uniform"]
    cov = pyref.run_restate(cp, hp, str(tmp_path / "cov"), bps=bps, stop_after=-1)["cov"]
    assert np.array_equal(got["graph"].BPCoverage(bps[:, 0], bps[:, 1]), cov)


def sparse_gap_case(d, n_frag=1_500_000):
    """About 3 M records, nearly every fragment a coverage gap: pairs of 100-bp mates 50 bp apart, fragments spread over the
    GRCh38 chromosomes evenly, about 2 kb apart.  More gap candidates than max(n / 16, 2^20), the first candidate buffer."""
    from squid_b200 import sqmb, synth
    rl = np.asarray(synth.GRCH38_LEN, np.int64)
    share = np.floor(n_frag * rl / rl.sum()).astype(np.int64)
    chr_ = np.repeat(np.arange(rl.shape[0]), share)
    pos = np.concatenate([np.arange(share[c]) * (rl[c] // (share[c] + 1)) + 500 for c in range(rl.shape[0])])
    m = chr_.shape[0]
    t = sqmb.empty(rl.astype(np.int32), 2 * m)
    t.ref_id[0::2] = chr_; t.ref_id[1::2] = chr_
    t.pos[0::2] = pos; t.pos[1::2] = pos + 50
    t.mate_ref_id[:] = t.ref_id
    t.mate_pos[0::2] = pos + 50; t.mate_pos[1::2] = pos
    t.flag[0::2] = 0x1 | 0x2 | 0x20 | 0x40; t.flag[1::2] = 0x1 | 0x2 | 0x10 | 0x80
    t.mapq[:] = 255
    t.name_id[0::2] = np.arange(m); t.name_id[1::2] = np.arange(m)
    t.cigar = np.full(2 * m, (100 << 4), np.uint32)
    t.cigar_off = np.arange(2 * m + 1, dtype=np.uint32)
    _, chim, _ = synth.make_case(2000, ref_len=synth.GRCH38_LEN, seed=5, disc_frac=0.2)
    cp, hp = os.path.join(d, "conc.sqmb"), os.path.join(d, "chim.sqmb")
    sqmb.write_sqmb(cp, t); sqmb.write_sqmb(hp, chim)
    return cp, hp, t


@pytest.mark.parametrize("load", ["host", "wire"])
def test_candidate_overflow_retry(load, tmp_path, built_lib):
    from oracle import pyref
    from squid_b200 import api
    cp, hp, tab = sparse_gap_case(str(tmp_path))
    rc = pyref.run_restate_classify(cp, hp, str(tmp_path / "rc"))
    want = common.expected_phase1(rc, tab.ref_id, tab.pos)
    n = tab.n
    assert want["gap_rec"].shape[0] > max(n // 16, 1 << 20)
    case = api.HostCase(cp, hp)
    g, _ = _graph(case, load)
    got = dumps(g)
    assert got["classify_attempts"] == 2
    assert_phase1(want, got, load)
    ref = pyref.run_restate(cp, hp, str(tmp_path / "ref"), stop_after=3)
    nodes = g.BuildNode_STAR(case.chimeric, None)
    e = g.BuildEdges()
    common.assert_same(ref, {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], 1).astype(np.int32),
                             "avgdepth": nodes.AvgDepth, "edges": e.table(), "chim_after_edges": case.chimeric.block_table()})


def _bad_batches(batch):
    """Batches that break a rule of the batch validation, with the code and the message each is refused with."""
    from squid_b200 import api
    a = {k: v.copy() for k, v in batch.a.items()}
    n = batch.n_rec
    out = {}
    b = {k: v.copy() for k, v in a.items()}; b["ref_id"][700] = 10 ** 6
    out["ref_id_range"] = (b, api.SQG_EINVAL, "ref_id outside")
    b = {k: v.copy() for k, v in a.items()}; b["ref_id"][700] = -1
    out["mapped_without_ref"] = (b, api.SQG_EUNSUPPORTED, "ref_id -1")
    b = {k: v.copy() for k, v in a.items()}
    r = 900
    o0, o1 = int(b["blk_off"][r]), int(b["blk_off"][r + 1])
    extra = 17 - (o1 - o0)
    for k in ("blk_ref_pos", "blk_match_ref", "blk_read_pos", "blk_match_read"):
        b[k] = np.concatenate([b[k][:o1], np.repeat(b[k][o0:o0 + 1], extra), b[k][o1:]])
    b["blk_off"][r + 1:] += extra
    out["17_blocks"] = (b, api.SQG_EUNSUPPORTED, "more than 16")
    b = {k: v.copy() for k, v in a.items()}
    r = int(np.flatnonzero(np.diff(b["blk_off"].astype(np.int64))[1000:] > 0)[0]) + 1000
    b["blk_off"][r + 1] = b["blk_off"][r] - 1
    out["decreasing_blk_off"] = (b, api.SQG_EUNSUPPORTED, "decreasing blk_off")
    b = {k: v.copy() for k, v in a.items()}; b["pos"][512] = b["pos"][511] - 1
    assert b["ref_id"][511] == b["ref_id"][512]
    out["unsorted_511_512"] = (b, api.SQG_EINVAL, "not sorted")
    b = {k: v.copy() for k, v in a.items()}; b["ref_id"][1300] = -1; b["flag"][1300] |= 0x4
    out["unmapped_then_mapped"] = (b, api.SQG_EINVAL, "not sorted")
    assert all(v[0]["blk_off"].shape[0] == n + 1 for v in out.values())
    return out


def test_batch_validation(streams, built_lib):
    """Every batch-validation flag of k_classify_tiles is refused with its code and message, and the same context then classifies a
    valid batch as the restatement does."""
    from squid_b200 import api
    cp, hp, tab, want = streams["base"]
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    for name, (arrays, code, msg) in _bad_batches(case.batch).items():
        g.load_concordant(api.RecordBatch(arrays))
        with pytest.raises(api.SquidB200Error) as ei:
            g.classify_dump("cls")
        assert ei.value.code == code and msg in str(ei.value), (name, ei.value.code, str(ei.value))
        g.load_concordant(case.batch)
        got = dumps(g)
        assert_phase1(want, got, name)
