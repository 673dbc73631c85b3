"""BuildEdges on injected segment tables (sqg_set_nodes, the graph reload of SegmentGraph_t(string), SegmentGraph.cpp:126-157)
against the restatement's literal LocateRead / RawEdgesChim / RawEdgesOther on the same table.  The families of
common.node_families put segment boundaries on and beside block ends, pack hundreds of segments into one position bin and
leave one segment per chromosome: the closed-form LocateRead, the hint fix-up chains, the position index, the tile's edge table
and the capacity retry of the edge pass all run on tables the seed machine never builds."""

import numpy as np
import pytest

from tests import common

pytestmark = pytest.mark.gpu

FAMILIES = ["built", "block_edges", "near_edges", "micro", "bins", "coarse", "random"]


@pytest.fixture(scope="module")
def family_cases(tmp_path_factory):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = common.family_case(tmp_path_factory.mktemp(name), name)
        return cache[name]
    return get


def _host(cp, hp, opts=()):
    from squid_b200 import api
    kw = {}
    if opts:
        kw = dict(concord_dist_pos=int(opts[1]), concord_dist_idx=int(opts[3]))
    return api.HostCase(cp, hp, **kw)


def _edges_on(case, nodes, load="host"):
    """Fresh context: concordant batch + chimeric reads + set_nodes + BuildEdges.  Returns (edges, chim_after_edges, graph)."""
    from squid_b200 import api
    g = api.SegmentGraph(case.config, case.ref_len)
    if load == "host":
        g.load_concordant(case.batch)
    elif load == "wire":
        g.load_concordant_wire(api.WireBatch(case.batch))
    else:
        g.attach_concordant_device(*_unaligned_device_batch(case))
    chim = api.ChimericReads(case.chimeric.a)
    g.load_chimeric(chim)
    g.set_nodes(nodes[:, 0], nodes[:, 1], nodes[:, 2])
    return g.BuildEdges().table(), chim.block_table(), g


def _unaligned_device_batch(case):
    """The batch in device arrays that start one element off their allocation (test_gpu_parity.py::test_unaligned_device_batch):
    the tiles are staged with plain loads instead of bulk copies."""
    import torch
    from squid_b200 import api
    keep, st = {}, api.sqg_batch()
    st.n_rec, st.n_blk = case.batch.n_rec, case.batch.n_blk
    for k, a in case.batch.a.items():
        dt = {"uint16": "int16", "uint32": "int32"}.get(a.dtype.name, a.dtype.name)
        t = torch.zeros(a.shape[0] + 3, dtype=getattr(torch, dt), device="cuda")
        v = t[1:1 + a.shape[0]]
        v.copy_(torch.from_numpy(a.view(dt)))
        keep[k] = t
        setattr(st, k, v.data_ptr())
        assert v.data_ptr() % 16 != 0
    return st, keep


def _max_tile_keys(raw, n_rec, tile=512):
    """Most distinct edge keys RawEdgesOther emits from one tile of `tile` consecutive records."""
    t = raw[:, 0] // tile
    best = 0
    for k in range(int(n_rec + tile - 1) // tile):
        sel = raw[t == k, 1]
        best = max(best, np.unique(sel).size)
    return best


@pytest.mark.parametrize("case,family,opts", [(c, f, []) for c in common.FAMILY_CASES for f in FAMILIES] +
                         [("chr17_s17", f, common.FAMILY_OPTS) for f in ("near_edges", "micro")])
def test_edges_on_injected_table(family_cases, case, family, opts, tmp_path, built_lib):
    from oracle import pyref
    cp, hp, ref_len, fam = family_cases(case)
    nodes = fam[family]
    want = pyref.run_restate_on_nodes(cp, hp, str(tmp_path / "ref"), nodes, opts=pyref.restate_opts(opts), dump_raw=family == "micro")
    hc = _host(cp, hp, opts)
    edges, chim, g = _edges_on(hc, nodes)
    common.assert_same(want, {"edges": edges, "chim_after_edges": chim}, ("edges", "chim_after_edges"))
    stats = {k: g.stat(k) for k in ("sensitive_reads", "edges_generic_path", "edge_pass_attempts", "raw_edges", "n_rec")}
    assert 1 <= stats["edge_pass_attempts"] <= 4, stats
    if family in ("near_edges", "micro"):
        assert stats["sensitive_reads"] > 0, stats
    if family != "coarse":
        assert stats["edges_generic_path"] > 0, stats
    if family == "micro" and case != "fourchr_s418":
        # the tile's 256-slot edge table must have spilled: some tile emits more distinct keys than it holds.  (Not in the
        # four-chromosome case: its genes are a few hundred bp long, so the records of a tile share too few start segments.)
        assert stats["n_rec"] == hc.batch.n_rec
        assert _max_tile_keys(want["raw_edges"], hc.batch.n_rec) > 256
    if case == "fourchr_s418" and family != "coarse":
        # many multi-block records leave their tile's segment: the deferred-record list overflows, and the next attempt trims
        # the chimeric blocks again from their pristine copies.  On block_edges and near_edges the first attempt's counts miss
        # the deferred records' raw pairs, so the second attempt overflowed again and the pass failed with SQG_ENOMEM.
        assert stats["edge_pass_attempts"] >= 2, stats


def test_context_reuse_across_tables(family_cases, tmp_path, built_lib):
    """set_nodes(A) -> BuildEdges -> set_nodes(B) -> BuildEdges -> set_nodes(A) -> BuildEdges on one context, with the same
    caller-owned chimeric arrays throughout: every result equals a fresh context's and the restatement's (the undo list of the
    chimeric-block patch puts back the blocks the previous table trimmed)."""
    from oracle import pyref
    from squid_b200 import api
    cp, hp, ref_len, fam = family_cases("chr17_s17")
    hc = _host(cp, hp)
    seq = ["near_edges", "micro", "near_edges"]
    want = {f: pyref.run_restate_on_nodes(cp, hp, str(tmp_path / f), fam[f]) for f in set(seq)}
    g = api.SegmentGraph(hc.config, hc.ref_len)
    g.load_concordant(hc.batch)
    chim = api.ChimericReads(hc.chimeric.a)
    g.load_chimeric(chim)
    for f in seq:
        nodes = fam[f]
        g.set_nodes(nodes[:, 0], nodes[:, 1], nodes[:, 2])
        got = {"edges": g.BuildEdges().table(), "chim_after_edges": chim.block_table()}
        common.assert_same(want[f], got, ("edges", "chim_after_edges"))
        e0, c0, _ = _edges_on(hc, nodes)
        common.assert_same({"edges": e0, "chim_after_edges": c0}, got, ("edges", "chim_after_edges"))


@pytest.mark.parametrize("load", ["wire", "unaligned"])
def test_injected_table_staging_paths(family_cases, load, tmp_path, built_lib):
    """The micro family through the wire upload and through a caller-owned device batch at odd offsets: the staging paths
    without bulk copies."""
    from oracle import pyref
    cp, hp, ref_len, fam = family_cases("chr17_s17")
    want = pyref.run_restate_on_nodes(cp, hp, str(tmp_path / "ref"), fam["micro"])
    edges, chim, _ = _edges_on(_host(cp, hp), fam["micro"], load)
    common.assert_same(want, {"edges": edges, "chim_after_edges": chim}, ("edges", "chim_after_edges"))


@pytest.mark.parametrize("family", ["micro", "bins"])
def test_coverage_after_reload(family_cases, family, tmp_path, built_lib):
    """BPCoverage after set_nodes + BuildEdges, on the injected table's segment ends: the coverage pass reads no segments, so the
    reload must leave it as the restatement's literal BAM pass computes it."""
    from oracle import pyref
    cp, hp, ref_len, fam = family_cases("chr17_s17")
    nodes = fam[family]
    want = pyref.run_restate_on_nodes(cp, hp, str(tmp_path / "ref"), nodes)
    d = {"final_nodes": nodes, "final_edges": want["edges"], "exactbp": np.zeros((0, 6), np.int32)}
    bps = pyref.breakpoints_of(d)
    assert bps.shape[0] > 0
    cov = pyref.run_restate(cp, hp, str(tmp_path / "cov"), bps=bps, stop_after=-1)["cov"]
    edges, _, g = _edges_on(_host(cp, hp), nodes)
    assert np.array_equal(edges, want["edges"])
    got = g.BPCoverage(bps[:, 0], bps[:, 1])
    assert np.array_equal(got, cov)


def _bad_tables(ref_len):
    """Tables that break the contract of sqg_set_nodes, each from a valid one-segment-per-chromosome table."""
    rl = [int(x) for x in ref_len]
    ok = [[c, 0, L] for c, L in enumerate(rl)]
    n = len(rl)
    out = {
        "chr_out_of_range": ok + [[n, 0, 10]],
        "negative_chr": [[-1, 0, 10]] + ok,
        "zero_length": [[0, 0, 0]] + ok,
        "negative_length": [[0, 0, 100], [0, 100, -5]] + [[0, 95, rl[0] - 95]] + ok[1:],
        "not_at_zero": [[0, 7, rl[0] - 7]] + ok[1:],
        "past_the_end": [[0, 0, rl[0] + 1]] + ok[1:],
        "short_of_the_end": [[0, 0, rl[0] - 1]] + ok[1:],
        "missing_last_chromosome": ok[:-1],
        "unsorted": [ok[1], ok[0]] + ok[2:],
        "gap": [[0, 0, 100], [0, 101, rl[0] - 101]] + ok[1:],
    }
    if n > 2:
        out["missing_chromosome"] = ok[:1] + ok[2:]
    return {k: np.array(v, np.int32) for k, v in out.items()}


def test_set_nodes_refuses_tables_that_do_not_tile(family_cases, tmp_path, built_lib):
    """Every shape that breaks "the table must tile the genome" is refused with SQG_EINVAL and a message, and the same context
    then accepts a valid table and gives the restatement's edges on it."""
    from oracle import pyref
    from squid_b200 import api
    cp, hp, ref_len, fam = family_cases("fourchr_s418")
    hc = _host(cp, hp)
    g = api.SegmentGraph(hc.config, hc.ref_len)
    g.load_concordant(hc.batch)
    chim = api.ChimericReads(hc.chimeric.a)
    g.load_chimeric(chim)
    good = fam["near_edges"]
    want = pyref.run_restate_on_nodes(cp, hp, str(tmp_path / "ref"), good)
    bad = _bad_tables(ref_len)
    assert "missing_chromosome" in bad
    for name, t in bad.items():
        with pytest.raises(api.SquidB200Error) as ei:
            g.set_nodes(t[:, 0], t[:, 1], t[:, 2])
        assert ei.value.code == api.SQG_EINVAL, name
        assert str(ei.value), name
        g.set_nodes(good[:, 0], good[:, 1], good[:, 2])
        got = {"edges": g.BuildEdges().table(), "chim_after_edges": chim.block_table()}
        common.assert_same(want, got, ("edges", "chim_after_edges"))
