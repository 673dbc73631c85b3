"""GPU parity tests proper: the CUDA path through the C ABI against the oracle (the reference's own sources
built against shims, oracle/_ref) on the same seeded synthetic inputs.  Bit-exact: everything is integer work
(AvgDepth is an int sum divided once on the host, so it is compared with == as well)."""
import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu

CASES = [
    # n_pairs, seed, disc_frac, ref_len, kwargs
    (3000, 3, 0.05, None, {}),
    (20000, 17, 0.02, None, {}),
    (30000, 29, 0.005, [3000000, 2000000, 500000, 16569], {"n_genes": 20}),
    (100000, 1003, 0.02, "grch38", {}),
    (200000, 1022, 0.005, [30000000, 20000000, 5000000, 16569], {"n_genes": 300}),
    (400000, 1020, 0.05, "grch38", {"fusion_support": 10}),
    # many multi-block records: the deferred-record list overflows and the edge pass runs twice; a chimeric block that the
    # first pass trimmed to 1 bp at a 1-bp segment would fit another segment the second time (found by tests/tools/fuzz_sharded.py)
    (60000, 418, 0.1, [30000000, 20000000, 5000000, 16569], {"fusion_support": 100, "exon_len": (20, 170), "intron_len": (60, 400)}),
]


@pytest.mark.parametrize("n_pairs,seed,disc,ref_len,kw", CASES)
def test_hot_path_matches_reference(tmp_path, built_lib, ref_oracle, n_pairs, seed, disc, ref_len, kw):
    from oracle import pyref
    from squid_b200 import synth
    rl = synth.GRCH38_LEN if ref_len == "grch38" else ref_len
    cp, hp, conc, chim, info = common.write_case(str(tmp_path), n_pairs, seed, disc, rl, **kw)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp, do_cov_with=ref)
    assert got["read_len"] == ref["read_len"]
    common.assert_same(ref, got)
    assert got["support"] == pyref.support_map(ref)
    g = got["graph"]
    assert g.launch_count() > 0
    if seed == 1020:  # several block-sized islands: k_seed_islands' whole-block path, longest island first
        assert g.stat("heavy_islands") > 1
    for ph in ("classify", "seed", "depth_edges", "edge_sort", "coverage"):
        assert g.phase_ms(ph) >= 0.0


def test_set_nodes_then_edges(tmp_path, built_lib, ref_oracle):
    """Edges and coverage on an injected segment table (the graph-reload seam, SegmentGraph.cpp:126-157)."""
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 20000, 5, 0.02)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    g.set_nodes(ref["nodes"][:, 0], ref["nodes"][:, 1], ref["nodes"][:, 2])
    e = g.BuildEdges()
    assert np.array_equal(e.table(), ref["edges"])
    assert np.array_equal(case.chimeric.block_table(), ref["chim_after_edges"])


def test_errors_are_loud(tmp_path, built_lib):
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 2000, 9, 0.05)
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len)
    with pytest.raises(api.SquidB200Error):
        g.BuildEdges()  # nothing loaded
    bad = case.batch.slice(0, case.batch.n_rec)
    bad.a["pos"] = bad.a["pos"][::-1].copy()
    g.load_concordant(bad)  # unsorted: the validation kernel's verdict surfaces at the next synchronising call
    g.load_chimeric(case.chimeric)
    with pytest.raises(api.SquidB200Error) as ei:
        g.BuildNode_STAR()
    assert "sorted" in str(ei.value)


def test_many_blocks_per_record(tmp_path, built_lib, ref_oracle):
    """Short exons: ~3 aligned blocks per record, so most tiles hold more blocks than the staging buffer takes and run the
    HBM path of the tile kernels; nearly every read goes through the generic multi-block rules."""
    from oracle import pyref
    cp, hp, conc, chim, info = common.write_case(str(tmp_path), 60000, 77, 0.02, [3000000, 2000000, 500000, 16569], n_genes=30, exon_len=(20, 170), intron_len=(60, 400))
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp, do_cov_with=ref)
    b = got["case"].batch
    assert b.n_blk > 1.5 * b.n_rec  # dense enough that tiles overflow the staging buffer
    common.assert_same(ref, got)
    assert got["support"] == pyref.support_map(ref)


def test_unaligned_device_batch(tmp_path, built_lib, ref_oracle):
    """A caller-owned device batch whose arrays start at odd offsets: no TMA bulk copies, the tiles are staged with plain
    loads.  Same answers."""
    import torch
    from oracle import pyref
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 30000, 41, 0.02)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    case = api.HostCase(cp, hp)
    keep, st = {}, api.sqg_batch()
    st.n_rec, st.n_blk = case.batch.n_rec, case.batch.n_blk
    for k, a in case.batch.a.items():
        t = torch.zeros(a.shape[0] + 3, dtype=getattr(torch, {"uint16": "int16", "uint32": "int32"}.get(a.dtype.name, a.dtype.name)), device="cuda")
        v = t[1:1 + a.shape[0]]  # one element off the allocation's alignment
        v.copy_(torch.from_numpy(a.view({"uint16": "int16", "uint32": "int32"}.get(a.dtype.name, a.dtype.name))))
        keep[k] = t
        setattr(st, k, v.data_ptr())
        assert v.data_ptr() % 16 != 0
    g = api.SegmentGraph(case.config, case.ref_len)
    g.attach_concordant_device(st, keepalive=keep)
    g.load_chimeric(case.chimeric)
    nodes = g.BuildNode_STAR()
    edges = g.BuildEdges()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": case.chimeric.block_table()}
    common.assert_same(ref, got)
    sup = g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref))
    assert sup == pyref.support_map(ref)


def test_degenerate_batches(tmp_path, built_lib):
    """Ragged inputs: an empty concordant batch, a batch that is not a multiple of the tile size, unsorted input."""
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 3000, 13, 0.05)
    case = api.HostCase(cp, hp)
    # 1. batch sizes around tile boundaries (512 records per tile): two contexts agree, and agree with the full batch on the prefix
    n = case.batch.n_rec

    def run(cut):
        g = api.SegmentGraph(case.config, case.ref_len)
        g.load_concordant(case.batch.slice(0, cut)); g.load_chimeric(api.ChimericReads(case.chimeric.a))
        try:
            nd = g.BuildNode_STAR(); ed = g.BuildEdges()
        except api.SquidB200Error as e:  # a stream that ends before the first group triggers: undefined in the reference, reported here
            assert e.code == api.SQG_EUNSUPPORTED
            return None
        return nd.Position.copy(), nd.Support.copy(), ed.table().copy()
    for cut in (n, n - 1, (n // 512) * 512, (n // 512) * 512 + 1, (n // 512) * 512 - 1, 1025, 512, 511):
        a, b2 = run(cut), run(cut)
        assert (a is None) == (b2 is None)
        if a is not None:
            assert all(np.array_equal(x, y) for x, y in zip(a, b2))
    # 2. no concordant record at all: the chimeric reads alone still give a graph
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch.slice(0, 0)); g.load_chimeric(api.ChimericReads(case.chimeric.a))
    try:
        n0 = g.BuildNode_STAR()
        assert n0.Chr.shape[0] >= len(case.ref_len)
    except api.SquidB200Error as e:  # BuildNode_STAR is undefined when nothing triggers a group; that must be reported, not crash
        assert e.code in (api.SQG_EUNSUPPORTED, api.SQG_ESTATE)
    # 3. unsorted input is refused
    bad = case.batch.slice(0, case.batch.n_rec)
    bad.a["pos"][10], bad.a["pos"][11] = bad.a["pos"][11] + 5, bad.a["pos"][10]
    if bad.a["ref_id"][10] == bad.a["ref_id"][11]:
        g = api.SegmentGraph(case.config, case.ref_len)
        g.load_concordant(bad); g.load_chimeric(api.ChimericReads(case.chimeric.a))
        with pytest.raises(api.SquidB200Error):
            g.BuildNode_STAR()


def test_dense_breakpoints_lagging_chain(tmp_path, built_lib):
    """Tens of thousands of breakpoints packed into expressed regions: indBP lags far behind the stream (one breakpoint per
    qualifying record, SegmentGraph.cpp:3157-3158), so the max-plus shortcut fails and the chunked literal chain has to repair
    chunks that run into each other.  Checked against the literal chain of the CPU stepping harness."""
    import subprocess
    from squid_b200 import api
    emul = common.build_emul(tmp_path / "bin")
    cp, hp, *_ = common.write_case(str(tmp_path), 60000, 23, 0.02, [3000000, 2000000, 500000, 16569], n_genes=40)
    case = api.HostCase(cp, hp)
    a = case.batch.a
    keys = np.unique((a["ref_id"].astype(np.int64) << 32) | a["pos"].astype(np.int64))
    keys = keys[keys >= 0]
    # every distinct record position, plus runs of consecutive positions behind each of them: very dense lists
    dense = np.unique(np.concatenate([keys, keys + 1, keys + 2, keys + 37]))
    bp = np.stack([(dense >> 32).astype(np.int32), (dense & 0xffffffff).astype(np.int32)], axis=1)
    bp = bp[bp[:, 1] < np.asarray(case.ref_len)[bp[:, 0]]]
    assert bp.shape[0] > 20000
    bp.astype(np.int32).tofile(str(tmp_path / "bps.bin"))
    out = tmp_path / "emul"
    out.mkdir()
    r = subprocess.run([emul, cp, hp, str(out), str(tmp_path / "bps.bin")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    want = np.fromfile(str(out / "cov_i32.bin"), dtype=np.int32)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch); g.load_chimeric(case.chimeric)
    got = g.BPCoverage(bp[:, 0], bp[:, 1])
    assert g.stat("cov_chain_fallback") == 1  # the shortcut must have failed, else this test does not test the chain
    assert np.array_equal(got, want)


def test_bam_input_matches_reference(tmp_path, built_lib, ref_oracle):
    """The same case fed as real BGZF-compressed BAM files through the library's own BAM front end (sqh_open_bam_case)."""
    from oracle import pyref
    from squid_b200 import api, bamio
    cp, hp, conc, chim, info = common.write_case(str(tmp_path), 8000, 19, 0.03)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, conc, block=8191); bamio.write_bam(hb, chim)
    case = api.HostCase(cb, hb, bam=True)
    g = api.SegmentGraph(case.config, case.ref_len)
    nodes = g.BuildNode_STAR(case.chimeric, case.batch)
    edges = g.BuildEdges()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": case.chimeric.block_table()}
    common.assert_same(ref, got)
    assert g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref)) == pyref.support_map(ref)


@pytest.mark.parametrize("opts,args", [
    (dict(min_mapq=3, max_lowphred_len=25, min_phred=10), ["-mq", "3", "-pl", "25", "-pm", "10"]),
    (dict(concord_dist_pos=3000, concord_dist_idx=2, max_lowphred_len=5), ["-dp", "3000", "-di", "2", "-pl", "5"]),
    # Phred64 (-pt 0 means offset 64 in the code, ReadRec.cpp:19-38, contrary to the README): threshold 'J' > every quality
    (dict(phred33=0, min_phred=10), ["-pt", "0", "-pm", "10"]),
])
def test_non_default_parameters(tmp_path, built_lib, ref_oracle, opts, args):
    """-mq / -pl / -pm gate and classify differently, -dp moves the point at which a breakpoint stops being counted
    (SegmentGraph.cpp:3157): the same options on both sides, same answers."""
    from oracle import pyref
    from squid_b200 import api
    cp, hp, *_ = common.write_case(str(tmp_path), 50000, 47, 0.03)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"), extra_args=args)
    base = ref_oracle.run(cp, hp, str(tmp_path / "ref0"))
    assert not (np.array_equal(ref["edges"], base["edges"]) and pyref.support_map(ref) == pyref.support_map(base)), "the options must change something"
    case = api.HostCase(cp, hp, **opts)
    g = api.SegmentGraph(case.config, case.ref_len)
    nodes = g.BuildNode_STAR(case.chimeric, case.batch)
    edges = g.BuildEdges()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": case.chimeric.block_table()}
    common.assert_same(ref, got)
    assert g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref)) == pyref.support_map(ref)


@pytest.mark.parametrize("n,seed,disc,ref_len,kw,want_unstable", [
    # aligned blocks of 1-3 bp (STAR's alignSJDBoverhangMin is 3): short NON-first blocks feed ReadsOther, whose merge loop
    # (SegmentGraph.cpp:806-825) counts them in the segment LEFT of the one they start in when that one still contains them
    # within +-3 -- unless an entry sorted before them has moved the cursor on
    (600, 303, 0.3, [3000000, 2000000], dict(n_genes=40, fusion_support=8), False),   # short blocks, no tie that matters: start masks only
    (600, 327, 0.3, [3000000, 2000000], dict(n_genes=40, fusion_support=8), False),
    (600, 302, 0.3, [3000000, 2000000], dict(n_genes=40, fusion_support=8), True),    # ties at a splice junction: the reference's answer
    (30000, 37, 0.2, None, dict(n_genes=100, fusion_support=20), True),               # is its unstable sort's tie order, replayed
    (30000, 38, 0.05, [3000000, 2000000, 500000, 16569], dict(n_genes=100, fusion_support=60), True),
    (120000, 39, 0.05, None, dict(n_genes=300, fusion_support=20, exon_len=(20, 170), intron_len=(60, 400)), True),
])
def test_short_blocks_match_reference(n, seed, disc, ref_len, kw, want_unstable, tmp_path, built_lib, ref_oracle):
    """min_block=1: nothing is filtered out of the generator.  Support / AvgDepth with 1-3 bp blocks, including the case the
    reference's own source leaves to std::sort's tie order (sqg_stat "unstable_depth_blocks" > 0: the sort is replayed)."""
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, ref_len, min_block=1, **kw)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp, do_cov_with=ref)
    common.assert_same(ref, got)
    g = got["graph"]
    assert g.stat("short_other_blocks") > 0
    assert (g.stat("unstable_depth_blocks") > 0) == want_unstable
    if want_unstable:
        assert g.stat("other_sort_status") == 0  # std::sort's permutation came from the device
    from oracle import pyref
    assert got["support"] == pyref.support_map(ref)
