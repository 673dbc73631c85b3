"""CPU tests of the oracle: the restatement (oracle/restate) must reproduce the committed golden dumps, which were
produced by the reference's own sources (oracle/_ref; script: tests/golden/make_golden.py).  When oracle/_ref is
present (development container / GPU box with the prebuilt binary) the goldens are re-derived and fresh fuzzed cases
are compared as well."""
import os

import numpy as np
import pytest

from oracle import pyref
from tests import common

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["chr17_3k", "fourchr_6k"]


def _gold(case):
    return pyref.load_dumps(os.path.join(GOLD, case, "ref"))


@pytest.mark.parametrize("case", CASES)
def test_restatement_reproduces_golden(case, tmp_path):
    g = _gold(case)
    bps = pyref.breakpoints_of(g)
    me = pyref.run_restate(os.path.join(GOLD, case, "conc.sqmb"), os.path.join(GOLD, case, "chim.sqmb"), str(tmp_path), bps=bps)
    assert me["read_len"] == g["read_len"]
    common.assert_same(g, me, ("chim_loaded", "chim_loaded_meta", "nodes", "avgdepth", "edges", "chim_after_edges"))
    assert pyref.support_from_cov(g, bps, me["cov"]) == pyref.support_map(g)


@pytest.mark.parametrize("case", CASES)
def test_restatement_edges_on_given_nodes(case, tmp_path):
    """BuildEdges of the restatement on an injected table (sqo_edges_on_nodes): on the reference's own segments it must give the
    reference's edges and trimmed chimeric blocks, so the reload entry shares the pinned path."""
    g = _gold(case)
    me = pyref.run_restate_on_nodes(os.path.join(GOLD, case, "conc.sqmb"), os.path.join(GOLD, case, "chim.sqmb"), str(tmp_path), g["nodes"], dump_raw=True)
    common.assert_same(g, me, ("edges", "chim_after_edges"))
    # every RawEdgesOther emission is one weight-1 row: their keys are a sub-multiset of the reduced table
    raw = me["raw_edges"]
    assert raw.shape[0] > 0 and np.all(np.diff(raw[:, 0]) >= 0)
    e = g["edges"].astype(np.int64)
    keys = (e[:, 0] << 33) | (e[:, 1] << 2) | (e[:, 2] << 1) | e[:, 3]
    k, c = np.unique(raw[:, 1], return_counts=True)
    at = np.searchsorted(keys, k)
    assert np.all(keys[at] == k) and np.all(c <= e[at, 4])


def test_restatement_decoder_kat(tmp_path):
    g = pyref.load_dumps(os.path.join(GOLD, "kat_decode", "ref"))
    me = pyref.run_restate(os.path.join(GOLD, "kat_decode", "conc.sqmb"), os.path.join(GOLD, "kat_decode", "chim.sqmb"), str(tmp_path), stop_after=1)
    common.assert_same(g, me, ("chim_loaded", "chim_loaded_meta"))
    assert me["read_len"] == g["read_len"]


@pytest.mark.parametrize("case", CASES)
def test_reference_build_reproduces_golden(case, tmp_path, reference_build):
    """The goldens are what oracle/_ref produces today (guards against stale fixtures)."""
    g = _gold(case)
    r = reference_build.run(os.path.join(GOLD, case, "conc.sqmb"), os.path.join(GOLD, case, "chim.sqmb"), str(tmp_path))
    common.assert_same(g, r, ("chim_loaded", "nodes", "avgdepth", "edges", "chim_after_edges", "final_nodes", "final_edges", "exactbp", "support"))


@pytest.mark.parametrize("seed,n,disc,ref_len", [(101, 4000, 0.05, None), (202, 20000, 0.01, [3000000, 2000000, 500000, 16569]), (303, 30000, 0.02, "grch38")])
def test_restatement_matches_reference_on_fuzz(seed, n, disc, ref_len, tmp_path, reference_build):
    from squid_b200 import synth
    rl = synth.GRCH38_LEN if ref_len == "grch38" else ref_len
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, rl)
    r = reference_build.run(cp, hp, str(tmp_path / "ref"))
    bps = pyref.breakpoints_of(r)
    me = pyref.run_restate(cp, hp, str(tmp_path / "me"), bps=bps)
    common.assert_same(r, me, ("chim_loaded", "nodes", "avgdepth", "edges", "chim_after_edges"))
    assert pyref.support_from_cov(r, bps, me["cov"]) == pyref.support_map(r)


@pytest.mark.parametrize("opts,args", [
    ((1, 25, 10, 3, 50000, 20), ["-mq", "3", "-pl", "25", "-pm", "10"]),
    ((1, 5, 4, -1, 3000, 2), ["-dp", "3000", "-di", "2", "-pl", "5"]),
    # -pt 0 selects offset 64 (ReadRec.cpp:19-38; the README says the opposite, SURVEY App. A-1): with -pm 10 the threshold
    # is 'J', above every synthetic quality, so every read has a low-phred run -- with offset 33 it would be '+'
    ((0, 10, 10, -1, 50000, 20), ["-pt", "0", "-pm", "10"]),
])
def test_restatement_matches_reference_with_options(opts, args, tmp_path, reference_build):
    """The -mq / -pl / -pm / -dp / -di rules (Config.cpp:18-25) on both sides; the options must change the outputs."""
    cp, hp, *_ = common.write_case(str(tmp_path), 20000, 47, 0.03)
    base = reference_build.run(cp, hp, str(tmp_path / "ref0"))
    r = reference_build.run(cp, hp, str(tmp_path / "ref"), extra_args=args)
    assert not (np.array_equal(r["edges"], base["edges"]) and pyref.support_map(r) == pyref.support_map(base))
    bps = pyref.breakpoints_of(r)
    me = pyref.run_restate(cp, hp, str(tmp_path / "me"), bps=bps, opts=opts)
    common.assert_same(r, me, ("chim_loaded", "nodes", "avgdepth", "edges", "chim_after_edges"))
    assert pyref.support_from_cov(r, bps, me["cov"]) == pyref.support_map(r)


@pytest.mark.parametrize("n,seed,disc,kw", [
    (30000, 37, 0.2, dict(n_genes=100, fusion_support=20)),
    (20000, 36, 0.05, dict(n_genes=20, fusion_support=20, exon_len=(20, 170), intron_len=(60, 400))),
])
def test_restatement_matches_reference_with_short_blocks(n, seed, disc, kw, tmp_path, reference_build):
    """min_block=1: aligned blocks of 1-3 bp are left in (the generators' default drops them)."""
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, None, min_block=1, **kw)
    r = reference_build.run(cp, hp, str(tmp_path / "ref"))
    bps = pyref.breakpoints_of(r)
    me = pyref.run_restate(cp, hp, str(tmp_path / "me"), bps=bps)
    common.assert_same(r, me, ("chim_loaded", "nodes", "avgdepth", "edges", "chim_after_edges"))
    assert pyref.support_from_cov(r, bps, me["cov"]) == pyref.support_map(r)
