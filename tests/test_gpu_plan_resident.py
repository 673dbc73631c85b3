"""Range shards of a concordant BAM decoded on the device: the planner on the resident batch (sqg_plan_shards_resident) gives the
host planner's cuts, sqg_keep_records leaves exactly one shard's records, and ShardedSegmentGraph.load_bam -- every context
decodes the whole file, plans, keeps its range -- reproduces the reference on the whole stream."""
import numpy as np
import pytest

from squid_b200 import api, bamio, sharded
from tests import bam_device_cases as bcases
from tests import common
from tests import plan_cases as pc
from tests.test_gpu_sharded import CASES as SHARDED_CASES

pytestmark = pytest.mark.gpu


def _device_cuts(g, max_shards=8):
    return {ns: g.plan_shards(ns) for ns in range(1, max_shards + 1)}


def _ctx(case, batch=None, shard=None):
    g = api.SegmentGraph(case.config, case.ref_len)
    if shard is not None:
        g.set_shard(*shard)
    g.load_concordant(batch if batch is not None else case.batch)
    g.load_chimeric(api.ChimericReads(case.chimeric.a))
    return g


@pytest.mark.parametrize("shape", list(pc.SHAPES))
def test_device_plan_matches_host(shape, tmp_path, built_lib):
    """Loaded from the host batch and decoded from the BAM file; twice on one context; on a context declared a shard."""
    cp, hp, conc, chim, _ = pc.write_shape(tmp_path, shape)
    case = api.HostCase(cp, hp)
    want = pc.host_cuts(case.batch, case)
    g = _ctx(case)
    assert _device_cuts(g) == want
    assert _device_cuts(g) == want
    g.close()
    g = _ctx(case, shard=(1, 2))
    assert _device_cuts(g) == want
    g.close()
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, conc); bamio.write_bam(hb, chim)
    hcase = api.HostCase(cb, hb, bam=True)
    dcase = api.HostCase(cb, hb, bam=True, header_only=True)
    g = api.SegmentGraph(dcase.config, dcase.ref_len)
    g.load_concordant_bam(cb, dcase)
    g.load_chimeric(api.ChimericReads(dcase.chimeric.a))
    assert _device_cuts(g) == pc.host_cuts(hcase.batch, hcase)
    g.close()


def test_device_plan_special_streams(tmp_path, built_lib):
    """Golden cases, an unmapped tail, no clean cut, dense groups, and runs longer than the look-back window."""
    import os
    for name in pc.golden_cases():
        case = api.HostCase(os.path.join(pc.GOLD, name, "conc.sqmb"), os.path.join(pc.GOLD, name, "chim.sqmb"))
        g = _ctx(case)
        assert _device_cuts(g) == pc.host_cuts(case.batch, case), name
        g.close()
    (tmp_path / "a").mkdir()
    cp, hp, *_ = pc.write_shape(tmp_path / "a", "fourchr")
    case = api.HostCase(cp, hp)
    streams = [pc.unmapped_tail(case.batch, 0.34), pc.no_gap_batch(case.batch)]
    a = case.batch.a
    c0 = pc.host_cuts(case.batch, case, 2)[2][1]
    gate = ((a["aux"] & 11) == 0) & (a["mapq"] >= case.config.Min_MapQual) & ((a["flag"] & 0x404) == 0) & (a["ref_id"] >= 0)
    k1 = int(np.flatnonzero(gate[:c0])[-1])
    for run in (pc.LOOK_BACK - 2000, pc.LOOK_BACK):
        streams += [pc.with_records(case.batch, k1 + 1, k1, run), pc.with_records(case.batch, k1 + 1, k1, run, 0)]
    for b in streams:
        g = _ctx(case, b)
        assert _device_cuts(g) == pc.host_cuts(b, case)
        g.close()
    (tmp_path / "d").mkdir()
    cp, hp, *_ = common.write_case(str(tmp_path / "d"), 8000, 303, 0.3, [3000000, 2000000], n_genes=40, fusion_support=8)
    case = api.HostCase(cp, hp)
    g = _ctx(case)
    assert _device_cuts(g) == pc.host_cuts(case.batch, case)
    g.close()


def _assert_batch(want: api.RecordBatch, got: api.RecordBatch):
    assert (want.n_rec, want.n_blk) == (got.n_rec, got.n_blk)
    for k in api.BATCH_DTYPES:
        assert np.array_equal(want.a[k], got.a[k]), k


def test_keep_records_matches_slice(tmp_path, built_lib):
    """download_concordant after keep_records(lo, hi) is case.batch.slice(lo, hi); the class bytes are then those of the slice
    loaded on its own (the whole stream's classification is dropped), from the host batch and from the BAM file."""
    cp, hp, conc, chim, _ = common.write_case(str(tmp_path), 6000, 17, 0.05)
    case = api.HostCase(cp, hp)
    n = case.batch.n_rec
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, conc); bamio.write_bam(hb, chim)
    dcase = api.HostCase(cb, hb, bam=True, header_only=True)
    ranges = [(0, n // 3), (n // 3, n), (n // 2, n // 2), (5, n - 3), (4099, 4100), (1, n), (n - 1, n), (0, n), (n, n)]
    for lo, hi in ranges:
        for from_bam in (False, True):
            g = api.SegmentGraph(case.config, case.ref_len)
            if from_bam:
                g.load_concordant_bam(cb, dcase)
            else:
                g.load_concordant(case.batch)
            g.classify_dump("cls")
            g.keep_records(lo, hi)
            want = case.batch.slice(lo, hi)
            _assert_batch(want, g.download_concordant())
            if hi > lo:
                g1 = api.SegmentGraph(case.config, case.ref_len)
                g1.load_concordant(want)
                assert np.array_equal(g.classify_dump("cls"), g1.classify_dump("cls")), (lo, hi)
                g1.close()
            g.close()


def _run_bam(cb, dcase, ns, ref):
    sg = sharded.ShardedSegmentGraph(dcase.config, dcase.ref_len, ns, list(range(ns)))
    cuts = sg.load_bam(cb, dcase)
    nodes = sg.BuildNode_STAR()
    edges = sg.BuildEdges()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": sg.Chimrecord.block_table()}
    common.assert_same(ref, got)
    from oracle import pyref
    assert api.SegmentGraph.ExactBPConcordantSupport(sg, ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref)) == pyref.support_map(ref)
    sg.close()
    return cuts


@pytest.mark.parametrize("n_pairs,seed,disc,ref_len,kw,shards", SHARDED_CASES)
@pytest.mark.parametrize("layout", ["htslib", "straddle_997"])
def test_load_bam_matches_reference(tmp_path, built_lib, ref_oracle, n_pairs, seed, disc, ref_len, kw, shards, layout):
    from squid_b200 import synth
    rl = synth.GRCH38_LEN if ref_len == "grch38" else ref_len
    cp, hp, conc, chim, _ = common.write_case(str(tmp_path), n_pairs, seed, disc, rl, **kw)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    open(cb, "wb").write(bcases.layouts(conc)[layout])
    bamio.write_bam(hb, chim)
    dcase = api.HostCase(cb, hb, bam=True, header_only=True)
    hcase = api.HostCase(cb, hb, bam=True)
    for ns in shards:
        cuts = _run_bam(cb, dcase, ns, ref)
        assert cuts == api.plan_shards(hcase.batch, hcase.chimeric, hcase.config, len(hcase.ref_len), ns) and len(cuts) == ns + 1


def test_load_bam_options_and_refusal(tmp_path, built_lib, ref_oracle):
    """Non-default -mq / -pl / -pm, 2 to 8 shards; a shard count the stream cannot give is refused with ValueError."""
    cp, hp, conc, chim, _ = common.write_case(str(tmp_path), 40000, 23, 0.02)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"), extra_args=pc.OPTS_ARGS)
    cb, hb = str(tmp_path / "conc.bam"), str(tmp_path / "chim.bam")
    bamio.write_bam(cb, conc); bamio.write_bam(hb, chim)
    dcase = api.HostCase(cb, hb, bam=True, header_only=True, **pc.OPTS)
    for ns in range(2, 9):
        _run_bam(cb, dcase, ns, ref)
    sg = sharded.ShardedSegmentGraph(dcase.config, dcase.ref_len, 100000, [0])  # far more shards than the stream has clean cuts
    with pytest.raises(ValueError):
        sg.load_bam(cb, dcase)
    sg.close()


def test_refusals_leave_context_usable(tmp_path, built_lib):
    cp, hp, *_ = common.write_case(str(tmp_path), 6000, 17, 0.05)
    case = api.HostCase(cp, hp)
    want = api.plan_shards(case.batch, case.chimeric, case.config, len(case.ref_len), 3)
    g = api.SegmentGraph(case.config, case.ref_len)
    with pytest.raises(api.SquidB200Error) as e:
        g.plan_shards(2)
    assert e.value.code == api.SQG_ESTATE
    with pytest.raises(api.SquidB200Error) as e:
        g.keep_records(0, 0)
    assert e.value.code == api.SQG_ESTATE
    g.load_concordant(case.batch)
    with pytest.raises(api.SquidB200Error) as e:
        g.plan_shards(2)  # no chimeric reads yet
    assert e.value.code == api.SQG_ESTATE
    g.load_chimeric(api.ChimericReads(case.chimeric.a))
    with pytest.raises(api.SquidB200Error) as e:
        g.plan_shards(0)
    assert e.value.code == api.SQG_EINVAL
    n = case.batch.n_rec
    for lo, hi in ((-1, 5), (5, 4), (0, n + 1)):
        with pytest.raises(api.SquidB200Error) as e:
            g.keep_records(lo, hi)
        assert e.value.code == api.SQG_EINVAL
    assert g.plan_shards(3) == want
    g.keep_records(want[1], want[2])
    with pytest.raises(api.SquidB200Error) as e:
        g.plan_shards(3)
    assert e.value.code == api.SQG_ESTATE
    _assert_batch(case.batch.slice(want[1], want[2]), g.download_concordant())
    g.close()
    # an attached (caller-owned) batch is not the context's to cut
    import torch
    t = {k: torch.from_numpy(np.ascontiguousarray(case.batch.a[k]).view(np.int8).copy()).cuda() for k in api.BATCH_DTYPES}
    s = api.sqg_batch()
    s.n_rec, s.n_blk = case.batch.n_rec, case.batch.n_blk
    for k in api.BATCH_DTYPES:
        setattr(s, k, t[k].data_ptr())
    torch.cuda.synchronize()
    g = api.SegmentGraph(case.config, case.ref_len)
    g.attach_concordant_device(s, keepalive=t)
    with pytest.raises(api.SquidB200Error) as e:
        g.keep_records(0, 10)
    assert e.value.code == api.SQG_ESTATE
    g.load_concordant(case.batch)  # still usable
    g.keep_records(0, 10)
    _assert_batch(case.batch.slice(0, 10), g.download_concordant())
    g.close()
