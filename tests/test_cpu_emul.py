"""The device-side rules (squid_b200/csrc/*.cuh, `SQ_HD`) stepped on the CPU by tests/emul and compared with the golden
dumps: the event-driven seed machine with island cuts, the closed-form LocateRead with the hint fix-up, the depth
cursor and the coverage chain are all exercised here without a GPU."""
import os
import subprocess

import numpy as np
import pytest

from oracle import pyref
from tests import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def emul_bin(tmp_path_factory):
    return common.build_emul(tmp_path_factory.mktemp("emul"))


@pytest.mark.parametrize("case", ["chr17_3k", "fourchr_6k"])
@pytest.mark.parametrize("one_island,bin_shift,chunks", [(False, 12, 1), (True, 12, 1), (False, 4, 7), (False, 0, 64)])
def test_stepped_rules_match_golden(case, one_island, bin_shift, chunks, emul_bin, tmp_path):
    g = pyref.load_dumps(os.path.join(GOLD, case, "ref"))
    bps = pyref.breakpoints_of(g)
    bps.tofile(str(tmp_path / "bps.bin"))
    env = dict(os.environ)
    env["SQH_PREPASS_CHUNKS"] = str(chunks)    # chimeric pre-pass: read loop split into this many chunks
    env["SQ_EMUL_BIN_SHIFT"] = str(bin_shift)  # segment-table position index: 0 = plain binary searches, 4 = many tiny bins
    if one_island:
        env["SQ_EMUL_ONE_ISLAND"] = "1"
        env["SQ_EMUL_NO_FAST_EDGES"] = "1"  # this variant runs every read through the generic read_edges
    r = subprocess.run([emul_bin, os.path.join(GOLD, case, "conc.sqmb"), os.path.join(GOLD, case, "chim.sqmb"), str(tmp_path), str(tmp_path / "bps.bin")],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    me = pyref.load_dumps(str(tmp_path))
    common.assert_same(g, me, ("nodes", "avgdepth", "edges", "chim_after_edges"))
    cov = np.fromfile(str(tmp_path / "cov_i32.bin"), dtype=np.int32)
    assert pyref.support_from_cov(g, bps, cov) == pyref.support_map(g)


@pytest.mark.parametrize("n,seed,disc,ref_len,kw", [
    (600, 303, 0.3, [3000000, 2000000], dict(n_genes=40, fusion_support=8)),
    (600, 302, 0.3, [3000000, 2000000], dict(n_genes=40, fusion_support=8)),
    (10000, 36, 0.02, None, dict(n_genes=20, fusion_support=20)),
    (30000, 38, 0.05, [3000000, 2000000, 500000, 16569], dict(n_genes=100, fusion_support=60, exon_len=(20, 170), intron_len=(60, 400))),
])
@pytest.mark.parametrize("dense", [False, True])
def test_stepped_rules_with_short_blocks(n, seed, disc, ref_len, kw, dense, emul_bin, ref_oracle, tmp_path):
    """Aligned blocks of 1-3 bp (min_block=1: nothing filtered out): the ReadsOther start masks, the replayed tie order of
    sort(ReadsOther), the short-block branches of the seed windows and of LocateRead, stepped on the CPU against the reference."""
    from squid_b200 import synth
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, ref_len if ref_len is not None else synth.CHR17_LEN, min_block=1, **kw)
    g = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    bps = pyref.breakpoints_of(g)
    bps.tofile(str(tmp_path / "bps.bin"))
    env = dict(os.environ)
    if dense:
        env["SQ_EMUL_DENSE"] = "100000"; env["SQ_EMUL_CC_TILE"] = "8"
    os.makedirs(str(tmp_path / "emu"))
    r = subprocess.run([emul_bin, cp, hp, str(tmp_path / "emu"), str(tmp_path / "bps.bin")], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "short ReadsOther blocks" in r.stderr and " 0 short ReadsOther" not in r.stderr
    me = pyref.load_dumps(str(tmp_path / "emu"))
    common.assert_same(g, me, ("nodes", "avgdepth", "edges", "chim_after_edges"))
    cov = np.fromfile(str(tmp_path / "emu" / "cov_i32.bin"), dtype=np.int32)
    assert pyref.support_from_cov(g, bps, cov) == pyref.support_map(g)


@pytest.fixture(scope="module")
def cov_case(tmp_path_factory):
    """Four chromosomes (one of 16569 bp), 30 k pairs, and the breakpoint list families of common.bp_families on its restated graph."""
    d = str(tmp_path_factory.mktemp("cov_case"))
    ref_len = [3000000, 2000000, 500000, 16569]
    cp, hp, conc, _, _ = common.write_case(d, 30000, 29, 0.05, ref_len, n_genes=20)
    g = pyref.run_restate(cp, hp, os.path.join(d, "graph"), stop_after=3)
    g["final_nodes"], g["final_edges"], g["exactbp"] = g["nodes"], g["edges"], np.zeros((0, 6), np.int32)
    fam = common.bp_families(ref_len, g["nodes"], conc, 29)
    fam["segment_ends"] = pyref.breakpoints_of(g)
    return cp, hp, ref_len, fam


@pytest.mark.parametrize("dp", [50000, 0, 3000, 100000000, -100, -5000])
@pytest.mark.parametrize("family", ["segment_ends", "uniform", "dups", "dense", "before", "after", "one", "empty"])
def test_coverage_chain_matches_restatement(cov_case, family, dp, emul_bin, tmp_path):
    """The stepped coverage rules (r0 over running maxima, the literal indBP chain, the count) against the literal BAM pass of the
    restatement (SegmentGraph.cpp:3124-3166) on the same list, at several -dp.  Every list also holds breakpoints at 0, 1, 99 and
    4999 of every chromosome (except the lists whose shape that would change): with a negative -dp, pos + dist < 0 there and every
    record of the chromosome passes the breakpoint."""
    cp, hp, ref_len, fam = cov_case
    bps = fam[family]
    if family not in ("before", "after", "one", "empty"):
        bps = common.bp_array(np.concatenate([bps, common.chr_start_bps(ref_len)]))
    if family == "before":
        assert bps.shape[0] > 0
    want = pyref.run_restate(cp, hp, str(tmp_path / "ref"), bps=bps, opts=pyref.restate_opts(["-dp", str(dp)]))
    bps.tofile(str(tmp_path / "bps.bin"))
    os.makedirs(str(tmp_path / "emu"))
    r = subprocess.run([emul_bin, cp, hp, str(tmp_path / "emu"), str(tmp_path / "bps.bin")], capture_output=True, text=True,
                       env=dict(os.environ, SQ_EMUL_DP=str(dp)))
    assert r.returncode == 0, r.stderr[-2000:]
    common.assert_same(want, pyref.load_dumps(str(tmp_path / "emu")), ("nodes", "edges"))  # -dp also gates edges (sq_locate.cuh)
    got = np.fromfile(str(tmp_path / "emu" / "cov_i32.bin"), dtype=np.int32)
    assert got.shape == want["cov"].shape
    bad = np.flatnonzero(got != want["cov"])
    assert bad.size == 0, "%d of %d breakpoints differ, first %s: restatement %s emul %s" % (
        bad.size, got.size, bps[bad[:3]].tolist(), want["cov"][bad[:3]].tolist(), got[bad[:3]].tolist())


@pytest.fixture(scope="module")
def family_cases(tmp_path_factory):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = common.family_case(tmp_path_factory.mktemp(name), name)
        return cache[name]
    return get


FAMILIES = ["built", "block_edges", "near_edges", "micro", "bins", "coarse", "random"]


@pytest.mark.parametrize("case,family,opts", [(c, f, []) for c in ("chr17_s17", "short_s37") for f in FAMILIES] +
                         [("chr17_s17", f, common.FAMILY_OPTS) for f in ("near_edges", "micro")])
@pytest.mark.parametrize("bin_shift", [0, 4, 9, 12])
@pytest.mark.parametrize("fast", [True, False])
def test_edges_on_injected_tables(family_cases, case, family, opts, bin_shift, fast, emul_bin, tmp_path):
    """BuildEdges on a segment table the caller installs (the graph-reload seam): the closed-form LocateRead, the hint replay and
    the position index stepped on the CPU against the restatement's literal LocateRead, on tables with segments on and beside
    block ends, runs of 1-6 bp segments, segments of one bin's size and one segment per chromosome.  Depth is not compared: the
    reload seam keeps the stored values."""
    cp, hp, ref_len, fam = family_cases(case)
    nodes = fam[family]
    want = pyref.run_restate_on_nodes(cp, hp, str(tmp_path / "ref"), nodes, opts=pyref.restate_opts(opts))
    nodes.tofile(str(tmp_path / "nodes.bin"))
    env = dict(os.environ, SQ_EMUL_NODES=str(tmp_path / "nodes.bin"), SQ_EMUL_BIN_SHIFT=str(bin_shift))
    if not fast:
        env["SQ_EMUL_NO_FAST_EDGES"] = "1"
    if opts:
        env["SQ_EMUL_DP"], env["SQ_EMUL_DI"] = opts[1], opts[3]
    os.makedirs(str(tmp_path / "emu"))
    r = subprocess.run([emul_bin, cp, hp, str(tmp_path / "emu")], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    common.assert_same(want, pyref.load_dumps(str(tmp_path / "emu")), ("edges", "chim_after_edges"))


@pytest.fixture(scope="module")
def stream_families(tmp_path_factory):
    return common.write_stream_families(tmp_path_factory.mktemp("streams"))


def _emul_phase1(emul_bin, cp, hp, d):
    os.makedirs(d)
    r = subprocess.run([emul_bin, cp, hp, d], capture_output=True, text=True, env=dict(os.environ, SQ_EMUL_CLASSIFY=d))
    assert r.returncode == 0, r.stderr[-2000:]
    rd = lambda f: np.fromfile(os.path.join(d, f), np.int32)
    gk = rd("gap_key_2xi32.bin").reshape(-1, 2).astype(np.int64)
    lm = rd("lmax_first_kept_i32.bin")
    return {"cls": rd("cls_i32.bin"), "first_len": rd("first_len_i32.bin"), "gap_rec": rd("gap_rec_i32.bin"),
            "gap_key": ((gk[:, 0] << 32) | (gk[:, 1] & 0xFFFFFFFF)).astype(np.uint64), "pc_rec": rd("pc_rec_i32.bin"),
            "dp_rec": rd("dp_rec_i32.bin"), "lmax": int(lm[0]), "first_kept": int(lm[1])}


@pytest.mark.parametrize("family", common.FAMILY_STREAMS)
def test_classify_rules_match_restatement(stream_families, family, emul_bin, tmp_path):
    """The classification rules (sq_classify.cuh) stepped record by record against the restatement's own per-record preamble of
    BuildNode_STAR (sqo_classify) on every stream family: class bytes, first-block lengths, the coverage-gap list and its
    otherrightmost keys, the partial and displaced lists, lmax and the first kept record.  A difference here is a wrong rule; a
    difference only on the device (tests/test_gpu_classify.py) is a wrong decomposition."""
    cp, hp, tab = stream_families[family]
    want = common.expected_phase1(pyref.run_restate_classify(cp, hp, str(tmp_path / "ref")), tab.ref_id, tab.pos)
    got = _emul_phase1(emul_bin, cp, hp, str(tmp_path / "emu"))
    for k in ("cls", "first_len", "gap_rec", "gap_key", "pc_rec", "dp_rec"):
        a, b = want[k].astype(np.int64), got[k].astype(np.int64)
        assert a.shape == b.shape, (k, a.shape, b.shape)
        bad = np.flatnonzero(a != b)
        assert bad.size == 0, "%s differs at %s: restatement %s emul %s" % (k, bad[:5], a[bad[:5]], b[bad[:5]])
    assert (got["lmax"], got["first_kept"]) == (want["lmax"], want["first_kept"])
    if family == "long_first_block":
        assert want["lmax"] == 70100 and (want["first_len"] == 65535).sum() > 0
    if family == "dup_shapes":
        assert want["first_kept"] == 1  # the leading empty record equals the default-constructed ReadRec_t


@pytest.mark.parametrize("family", common.FAMILY_STREAMS)
def test_stream_families_end_to_end(stream_families, family, emul_bin, tmp_path):
    """Segments, AvgDepth, edges and trimmed chimeric blocks of the stepped rules against sqo_run on every stream family."""
    cp, hp, _ = stream_families[family]
    want = pyref.run_restate(cp, hp, str(tmp_path / "ref"), stop_after=3)
    os.makedirs(str(tmp_path / "emu"))
    r = subprocess.run([emul_bin, cp, hp, str(tmp_path / "emu")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    common.assert_same(want, pyref.load_dumps(str(tmp_path / "emu")))
