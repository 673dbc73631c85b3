"""Breakpoint coverage on the GPU (sqg_bp_coverage: the r0 search over tile maxima, the max-plus scan and its verification, the
chunked literal chain with its repair rounds, the whole-list replay, the 256-wide breakpoint windows of k_cov_count_tiles) against
independent numbers: the reference's own golden dumps, and the literal BAM pass of the CPU restatement (oracle/restate,
SegmentGraph.cpp:3124-3166) run on the same records and the same breakpoint list.  The lists have the shapes the product passes
(ExactBreakpoint + CountTop: interior positions, many duplicates around a fusion hub), not only segment ends."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
FOURCHR = [3000000, 2000000, 500000, 16569]


@pytest.fixture(scope="module")
def restate():
    from oracle import pyref
    pyref.build_restate()
    return pyref


def restated_cov(pyref, cp, hp, outdir, bps, args=()):
    return pyref.run_restate(cp, hp, outdir, bps=bps, opts=pyref.restate_opts(args), stop_after=-1)["cov"]


def assert_cov(got, want, bps, what=""):
    assert got.shape == want.shape, "%s: %s vs %s breakpoints" % (what, got.shape, want.shape)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, "%s: %d of %d breakpoints differ, first %s: restatement %s CUDA %s" % (
        what, bad.size, got.size, bps[bad[:3]].tolist(), want[bad[:3]].tolist(), got[bad[:3]].tolist())


def table(nodes):
    return np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32)


def qualifying_keys(batch, min_mapq):
    """(chr + 1) << 32 | fragment start of the records the BAM pass counts (:3136-3155), in stream order: the device's rank space."""
    a = batch.a
    f = a["flag"].astype(np.int64)
    rid, pos = a["ref_id"].astype(np.int64), a["pos"].astype(np.int64)
    mrid, mpos = a["mate_ref_id"].astype(np.int64), a["mate_pos"].astype(np.int64)
    gate = ((a["aux"] & 11) == 0) & (a["mapq"].astype(np.int64) >= min_mapq) & ((f & 0x400) == 0) & ((f & 4) == 0) & (rid >= 0)
    same = ((f & 8) == 0) & (mrid == rid)
    q = gate & ~(same & (mpos > pos)) & ~(same & (mpos == pos) & ((f & 0x80) != 0))
    return ((rid[q] + 1) << 32) | np.where(same, mpos, pos)[q]


def lag_clusters(case, n_clusters, size=5200, gap=4700, first=20000):
    """`n_clusters` clusters of `size` copies of one breakpoint whose r0 (first qualifying rank past pos + Concord_Dist_Pos) lie
    `gap` ranks apart: more than kChainGap (4096), so every cluster starts a chunk of the literal chain, but fewer than the `size`
    ranks of lag each cluster builds up, so every chunk's chain runs into the next one and the repair needs one round per cluster.
    Returns the list and the r0 of the clusters."""
    M = np.maximum.accumulate(qualifying_keys(case.batch, case.config.Min_MapQual))
    assert M.shape[0] > first + n_clusters * gap
    bp, r0 = [], []
    for i in range(n_clusters):
        T = int(M[first + i * gap - 1])
        bp += [((T >> 32) - 1, (T & 0xffffffff) - case.config.Concord_Dist_Pos)] * size
        r0.append(int(np.searchsorted(M, T, side="right")))
    bp = common.bp_array(bp)
    assert (bp[:, 1] >= 0).all()
    return bp, np.array(r0)


# ---- a. golden cases, end to end, against the reference's own numbers -------------------------------------------------------

@pytest.mark.parametrize("case", ["chr17_3k", "fourchr_6k"])
def test_golden_exact_breakpoint_support(case, built_lib):
    """Segments, edges and trimmed blocks from the CUDA path; ExactBreakpoint on the reference's final graph from the blocks the
    CUDA path trimmed; the coverage at those exact breakpoints: all equal to the reference's own dumps."""
    from oracle import pyref
    from squid_b200 import api
    d = os.path.join(GOLD, case)
    ref = pyref.load_dumps(os.path.join(d, "ref"))
    got = common.run_cuda(os.path.join(d, "conc.sqmb"), os.path.join(d, "chim.sqmb"))
    common.assert_same(ref, got)
    chim = got["case"].chimeric
    rows = api.ExactBreakpoint(ref["final_nodes"], chim)
    assert np.array_equal(rows, ref["exactbp"])
    assert np.array_equal(chim.block_table(), np.fromfile(os.path.join(d, "ref", "chim_after_exactbp.bin"), dtype=np.int32).reshape(-1, 8))
    assert rows.shape[0] > 0
    sup = got["graph"].ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map({"exactbp": rows}))
    assert sup == pyref.support_map(ref)


# ---- b. differential: BPCoverage(list) == the restatement's BAM pass on the same list -----------------------------------------

SHAPES = [
    # n_pairs, seed, disc_frac, ref_len, kwargs
    (20000, 17, 0.02, None, {}),
    (30000, 29, 0.05, FOURCHR, {"n_genes": 20}),
    (100000, 1003, 0.02, "grch38", {}),
    (60000, 77, 0.05, FOURCHR, {"n_genes": 30, "exon_len": (20, 170), "intron_len": (60, 400)}),
]
FAMILIES = ["product", "segment_ends", "uniform", "dups", "dense", "before", "after", "one", "empty"]


@pytest.fixture(scope="module", params=SHAPES, ids=["chr17", "fourchr", "grch38", "short_exons"])
def shape(request, tmp_path_factory, built_lib, restate):
    """One case on one context after BuildNode_STAR + BuildEdges, with its breakpoint lists.  "product" is the list the product
    passes: ExactBreakpoint on the CUDA graph (its raw segments and edges taken as the final graph), assembled as the reference
    does (pyref.breakpoints_of)."""
    from squid_b200 import api, synth
    n, seed, disc, rl, kw = request.param
    rl = synth.GRCH38_LEN if rl == "grch38" else (rl if rl is not None else synth.CHR17_LEN)
    d = str(tmp_path_factory.mktemp("shape"))
    cp, hp, conc, _, _ = common.write_case(d, n, seed, disc, rl, **kw)
    case = api.HostCase(cp, hp)
    chim0 = api.ChimericReads(case.chimeric.a)  # a copy: BuildEdges and ExactBreakpoint trim case.chimeric in place
    g = api.SegmentGraph(case.config, case.ref_len)
    nodes = table(g.BuildNode_STAR(case.chimeric, case.batch))
    edges = g.BuildEdges().table()
    rows = api.ExactBreakpoint(nodes, case.chimeric)
    graph = {"final_nodes": nodes, "final_edges": edges, "exactbp": rows}
    fam = common.bp_families(rl, nodes, conc, seed)
    fam["product"] = restate.breakpoints_of(graph)
    fam["segment_ends"] = restate.breakpoints_of({"final_nodes": nodes, "final_edges": edges, "exactbp": np.zeros((0, 6), np.int32)})
    assert rows.shape[0] > 0 and np.unique(fam["product"], axis=0).shape[0] < fam["product"].shape[0]
    want = {}

    def cov(f):  # the restatement's coverage of list f, computed once
        if f not in want:
            want[f] = restated_cov(restate, cp, hp, os.path.join(d, "ref_" + f), fam[f])
        return want[f]
    yield {"case": case, "chim0": chim0, "g": g, "graph": graph, "fam": fam, "cov": cov, "idx": SHAPES.index(request.param)}
    g.close()


@pytest.mark.parametrize("family", FAMILIES)
def test_coverage_lists_match_restatement(shape, family, restate):
    g, bps = shape["g"], shape["fam"][family]
    want = shape["cov"](family)
    got = g.BPCoverage(bps[:, 0], bps[:, 1])
    assert_cov(got, want, bps, family)
    if family == "product":
        gr = shape["graph"]
        sup = g.ExactBPConcordantSupport(gr["final_nodes"], gr["final_edges"], restate.exactbp_map(gr))
        assert sup == restate.support_from_cov(gr, bps, want)
    if family == "dense":  # more than 256 breakpoints under one block of 1024 ranks: several windows of k_cov_count_tiles
        assert bps.shape[0] >= 2900


def test_chain_repaired_in_rounds(tmp_path, built_lib, restate):
    """Four lagging clusters: the max-plus shortcut fails, the chunked literal chain is repaired in a few rounds (cov_chain_chunks
    stays > 1: no whole-list replay)."""
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 60000, 41, 0.02)
    case = api.HostCase(cp, hp)
    bps, r0 = lag_clusters(case, 4)
    assert (np.diff(r0) > 4096).all() and (np.diff(r0) < 5200).all()
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    got = g.BPCoverage(bps[:, 0], bps[:, 1])
    assert g.stat("cov_chain_fallback") == 1 and g.stat("cov_chain_chunks") > 1
    assert_cov(got, restated_cov(restate, cp, hp, str(tmp_path / "ref"), bps), bps)


def test_chain_whole_list_replay(tmp_path, built_lib, restate):
    """24 lagging clusters: each repair round settles one more chunk, 16 rounds do not settle them all, and the whole list is
    replayed by one warp (cov_chain_chunks == 1 after the fallback)."""
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 200000, 43, 0.02)
    case = api.HostCase(cp, hp)
    bps, r0 = lag_clusters(case, 24)
    assert (np.diff(r0) > 4096).all() and (np.diff(r0) < 5200).all()
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    got = g.BPCoverage(bps[:, 0], bps[:, 1])
    assert g.stat("cov_chain_fallback") == 1 and g.stat("cov_chain_chunks") == 1
    assert_cov(got, restated_cov(restate, cp, hp, str(tmp_path / "ref"), bps), bps)


# ---- c. options ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("opts,args", [
    (dict(concord_dist_pos=0), ["-dp", "0"]),
    (dict(concord_dist_pos=3000), ["-dp", "3000"]),
    # pos + dist < 0 for breakpoints near a chromosome start: every record of the chromosome passes them (an unsigned threshold
    # key used to stall indBP there, and every later breakpoint's coverage was wrong)
    (dict(concord_dist_pos=-100), ["-dp", "-100"]),
    (dict(concord_dist_pos=-5000), ["-dp", "-5000"]),
    (dict(min_mapq=3, max_lowphred_len=25, min_phred=10), ["-mq", "3", "-pl", "25", "-pm", "10"]),
])
def test_options(opts, args, tmp_path, built_lib, restate):
    from squid_b200 import api
    cp, hp, conc, _, _ = common.write_case(str(tmp_path), 30000, 29, 0.05, FOURCHR, n_genes=20)
    case = api.HostCase(cp, hp, **opts)
    g = api.SegmentGraph(case.config, case.ref_len)
    nodes = table(g.BuildNode_STAR(case.chimeric, case.batch))
    edges = g.BuildEdges().table()
    fam = common.bp_families(FOURCHR, nodes, conc, 29)
    ends = restate.breakpoints_of({"final_nodes": nodes, "final_edges": edges, "exactbp": np.zeros((0, 6), np.int32)})
    for name, bps in (("segment_ends", ends), ("dups", fam["dups"]), ("uniform", fam["uniform"])):
        bps = common.bp_array(np.concatenate([bps, common.chr_start_bps(FOURCHR)]))
        got = g.BPCoverage(bps[:, 0], bps[:, 1])
        assert_cov(got, restated_cov(restate, cp, hp, str(tmp_path / ("ref_" + name)), bps, args), bps, name)


def test_chimname_gated_records(tmp_path, built_lib, restate):
    """Concordant records that carry the name of a chimeric read fail the gate (SegmentGraph.cpp:302 via :3136): the host packer
    sets SQG_AUX_CHIMNAME, the restatement looks the raw names up itself."""
    from squid_b200 import api, sqmb, synth
    conc, chim, _ = synth.make_case(30000, ref_len=FOURCHR, seed=31, disc_frac=0.05, n_genes=20)
    rng = np.random.default_rng(5)
    take = rng.choice(conc.n, size=3000, replace=False)
    conc.name_id[take] = rng.choice(chim.name_id, size=take.shape[0])
    cp, hp = str(tmp_path / "conc.sqmb"), str(tmp_path / "chim.sqmb")
    sqmb.write_sqmb(cp, conc); sqmb.write_sqmb(hp, chim)
    case = api.HostCase(cp, hp)
    assert ((case.batch.a["aux"] & 8) != 0).sum() > 500
    g = api.SegmentGraph(case.config, case.ref_len)
    nodes = table(g.BuildNode_STAR(case.chimeric, case.batch))
    fam = common.bp_families(FOURCHR, nodes, conc, 31)
    for name in ("dups", "dense", "uniform"):
        bps = fam[name]
        got = g.BPCoverage(bps[:, 0], bps[:, 1])
        assert_cov(got, restated_cov(restate, cp, hp, str(tmp_path / ("ref_" + name)), bps), bps, name)


# ---- d. batch shapes ------------------------------------------------------------------------------------------------------------

def test_batch_shapes(tmp_path, built_lib, restate):
    """Prefixes around the 512-record classification tile and the 2048-record coverage tile, and a batch without any qualifying
    record (left-hand mates only), each written as its own SQMB so that both sides read the same records."""
    from squid_b200 import api, sqmb
    _, hp, conc, _, _ = common.write_case(str(tmp_path), 20000, 53, 0.02, FOURCHR, n_genes=20)
    same = ((conc.flag & 8) == 0) & (conc.mate_ref_id == conc.ref_id)
    left = np.flatnonzero(same & (conc.mate_pos > conc.pos))[:3000]
    rng = np.random.default_rng(7)
    for name, idx in [("p%d" % n, np.arange(n)) for n in (1, 511, 513, 2047, 2049)] + [("left_only", left)]:
        sub = conc.take(idx)
        cp = str(tmp_path / (name + ".sqmb"))
        sqmb.write_sqmb(cp, sub)
        starts = np.stack([sub.ref_id, sub.pos], 1).astype(np.int64)
        bps = common.bp_array(np.concatenate([starts, starts + [0, 50], starts + [0, 150], np.repeat(starts[:1] + [0, 20], 40, axis=0),
                                              common.chr_start_bps(FOURCHR)]))
        case = api.HostCase(cp, hp)
        g = api.SegmentGraph(case.config, case.ref_len)
        g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
        got = g.BPCoverage(bps[:, 0], bps[:, 1])
        want = restated_cov(restate, cp, hp, str(tmp_path / ("ref_" + name)), bps)
        assert_cov(got, want, bps, name)
        if name == "left_only":
            assert qualifying_keys(case.batch, case.config.Min_MapQual).shape[0] == 0 and not want.any()
        g.close(); case.close()


# ---- e. input paths and context state ------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def small(tmp_path_factory, restate):
    """A 4-chromosome case with its list families (from the restated segment table) and their restated coverage."""
    d = str(tmp_path_factory.mktemp("small"))
    cp, hp, conc, chim, _ = common.write_case(d, 30000, 61, 0.03, FOURCHR, n_genes=20)
    gr = restate.run_restate(cp, hp, os.path.join(d, "graph"), stop_after=3)
    fam = common.bp_families(FOURCHR, gr["nodes"], conc, 61)
    want = {f: restated_cov(restate, cp, hp, os.path.join(d, "ref_" + f), fam[f]) for f in ("dups", "dense", "uniform")}
    return {"cp": cp, "hp": hp, "conc": conc, "chim": chim, "fam": fam, "want": want}


def check_small(g, small, families=("dups", "dense", "uniform")):
    fam, want = small["fam"], small["want"]
    for f in families:
        assert_cov(g.BPCoverage(fam[f][:, 0], fam[f][:, 1]), want[f], fam[f], f)


def test_after_wire_upload(small, built_lib):
    from squid_b200 import api
    cp, hp = small["cp"], small["hp"]
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant_wire(api.WireBatch(case.batch, pinned=True)); g.load_chimeric(case.chimeric)
    check_small(g, small)


def test_after_wire_upload_without_tile_classification(small, built_lib, tmp_path):
    """SQG_WIRE_CLASSIFY=0 (read once per process, so in a process of its own): the wire upload leaves classification to run_classify."""
    cp, hp, fam, want = small["cp"], small["hp"], small["fam"], small["want"]
    script = ("import sys, numpy as np\nsys.path.insert(0, %r)\nfrom squid_b200 import api\n"
              "case = api.HostCase(%r, %r)\ng = api.SegmentGraph(case.config, case.ref_len)\n"
              "g.load_concordant_wire(api.WireBatch(case.batch)); g.load_chimeric(case.chimeric)\n"
              "for f in ('dups', 'dense', 'uniform'):\n"
              "    bp = np.load(%r + '/' + f + '.npy'); np.save(%r + '/got_' + f + '.npy', g.BPCoverage(bp[:, 0], bp[:, 1]))\n"
              ) % (ROOT, cp, hp, str(tmp_path), str(tmp_path))
    for f in ("dups", "dense", "uniform"):
        np.save(str(tmp_path / (f + ".npy")), fam[f])
    r = subprocess.run([sys.executable, "-c", script], cwd=ROOT, capture_output=True, text=True, env=dict(os.environ, SQG_WIRE_CLASSIFY="0"))
    assert r.returncode == 0, r.stderr[-3000:]
    for f in ("dups", "dense", "uniform"):
        assert_cov(np.load(str(tmp_path / ("got_" + f + ".npy"))), want[f], fam[f], f)


def test_after_unaligned_device_attach(small, built_lib):
    import torch
    from squid_b200 import api
    cp, hp = small["cp"], small["hp"]
    case = api.HostCase(cp, hp)
    keep, st = {}, api.sqg_batch()
    st.n_rec, st.n_blk = case.batch.n_rec, case.batch.n_blk
    for k, a in case.batch.a.items():
        dt = {"uint16": "int16", "uint32": "int32"}.get(a.dtype.name, a.dtype.name)
        t = torch.zeros(a.shape[0] + 3, dtype=getattr(torch, dt), device="cuda")
        v = t[1:1 + a.shape[0]]  # one element off the allocation's alignment
        v.copy_(torch.from_numpy(a.view(dt)))
        keep[k] = t
        setattr(st, k, v.data_ptr())
    g = api.SegmentGraph(case.config, case.ref_len)
    g.attach_concordant_device(st, keepalive=keep); g.load_chimeric(case.chimeric)
    check_small(g, small)


def test_from_bam_input(small, built_lib, tmp_path):
    from squid_b200 import api, bamio
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, small["conc"], block=8191); bamio.write_bam(hb, small["chim"])
    case = api.HostCase(cb, hb, bam=True)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    check_small(g, small)


def test_before_and_after_build_nodes(small, built_lib):
    """Before BuildNode_STAR the coverage pass classifies the records itself (cov_prepare); after it, it reuses that compaction."""
    from squid_b200 import api
    cp, hp = small["cp"], small["hp"]
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    check_small(g, small)
    g.BuildNode_STAR()
    check_small(g, small)
    g.BuildEdges()
    check_small(g, small, ("dense",))


def test_context_reuse(small, built_lib, tmp_path, restate):
    """One context: a long list, a short list, then a different batch and another list (buffers reused, cov_compacted reset)."""
    from squid_b200 import api
    cp, hp, fam, want = small["cp"], small["hp"], small["fam"], small["want"]
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    check_small(g, small, ("dups", "dense"))
    one = fam["dups"][:1]
    assert_cov(g.BPCoverage(one[:, 0], one[:, 1]), restated_cov(restate, cp, hp, str(tmp_path / "ref_one"), one), one, "short")
    cp2, hp2, conc2, _, _ = common.write_case(str(tmp_path), 12000, 62, 0.03, FOURCHR, n_genes=10)
    case2 = api.HostCase(cp2, hp2)
    g.load_concordant(case2.batch); g.load_chimeric(case2.chimeric)
    starts = np.stack([conc2.ref_id, conc2.pos], 1).astype(np.int64)
    bps = common.bp_array(np.concatenate([starts[::7] + [0, 30], common.chr_start_bps(FOURCHR)]))
    assert_cov(g.BPCoverage(bps[:, 0], bps[:, 1]), restated_cov(restate, cp2, hp2, str(tmp_path / "ref2"), bps), bps, "reloaded")


# ---- f. sharded -----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("family", ["dups", "dense", "product"])
def test_sharded_matches_restatement(shape, family, built_lib):
    """The range-sharded coverage chain (speculative hand-over between shards, repaired in rounds) against the restatement on the
    whole stream, with 2 to 5 shards."""
    import types
    from squid_b200 import api
    from tests.tools import gpu_sharded_diag as diag
    c, bps = shape["case"], shape["fam"][family]
    case = types.SimpleNamespace(batch=c.batch, chimeric=shape["chim0"], config=c.config, ref_len=c.ref_len)  # untrimmed Chimrecord
    ns = 2 + shape["idx"] % 4
    cuts = api.plan_shards(case.batch, case.chimeric, case.config, len(case.ref_len), ns)
    assert len(cuts) - 1 >= 2, "the planner found no clean cut"
    got = diag.run_sharded(case, cuts, None, bps)
    got["sg"].close()
    assert_cov(got["cov"], shape["cov"](family), bps, family)
