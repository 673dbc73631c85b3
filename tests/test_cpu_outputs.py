"""Host twins of the stages between the device path and the files a SQUID user reads (SURVEY.md §8 rows a17, a20):
ExactBreakpoint + CountTop and the `_graph.txt` / `_sv.txt` writers, against the reference's own sources (oracle/_ref, run
with --write-outputs; golden copies under tests/golden/*/ref).  Pure host code: no GPU needed."""
import filecmp
import os

import numpy as np
import pytest

from oracle import pyref
from tests import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _chim_from_dump(api, rows8: np.ndarray, meta: np.ndarray):
    """ChimericReads from the harness's Chimrecord dump: rows (read, mate, RefID, RefPos, ReadPos, MatchRef, MatchRead, IsReverse)."""
    n_reads = int(meta.shape[0])
    read = rows8[:, 0].astype(np.int64)
    order = np.lexsort((np.arange(rows8.shape[0]), rows8[:, 1], read))  # first-mate blocks before second-mate blocks, dump order kept
    assert np.array_equal(order, np.arange(rows8.shape[0])), "the dump lists FirstRead before SecondMate per read"
    read_off = np.zeros(n_reads + 1, np.uint32)
    np.add.at(read_off, read + 1, 1)
    read_off = np.cumsum(read_off).astype(np.uint32)
    n_first = np.zeros(n_reads, np.uint16)
    np.add.at(n_first, read[rows8[:, 1] == 0], 1)
    a = {
        "read_off": read_off, "n_first": n_first,
        "first_total_len": meta[:, 0].astype(np.int32), "second_total_len": meta[:, 1].astype(np.int32),
        "first_lowphred": (meta[:, 2] > 0).astype(np.uint8), "second_lowphred": (meta[:, 3] > 0).astype(np.uint8),
        "multi_filter": np.zeros(n_reads, np.uint8),
        "blk_ref_id": rows8[:, 2].astype(np.int32), "blk_ref_pos": rows8[:, 3].astype(np.int32), "blk_read_pos": rows8[:, 4].astype(np.int32),
        "blk_match_ref": rows8[:, 5].astype(np.int32), "blk_match_read": rows8[:, 6].astype(np.int32), "blk_is_reverse": rows8[:, 7].astype(np.uint8),
    }
    return api.ChimericReads(a)


def _check_dir(refdir, tmp_path, n_ref, min_sv_lines=0):
    from squid_b200 import api
    d = pyref.load_dumps(refdir)
    i32 = lambda name, cols: np.fromfile(os.path.join(refdir, name), dtype=np.int32).reshape(-1, cols)
    # ---- a17: ExactBreakpoint + CountTop on the final graph, from the Chimrecord BuildEdges left behind
    chim = _chim_from_dump(api, d["chim_after_edges"], d["chim_loaded_meta"])
    rows = api.ExactBreakpoint(d["final_nodes"], chim)
    assert np.array_equal(rows, d["exactbp"]), "ExactBP map differs from the reference"
    assert np.array_equal(chim.block_table(), i32("chim_after_exactbp.bin", 8)), "LocateRead on the final graph trims differently"
    # ---- a20: _graph.txt
    avg = np.fromfile(os.path.join(refdir, "final_nodes_f64.bin"))
    labels = np.fromfile(os.path.join(refdir, "labels_i32.bin"), dtype=np.int32)
    gp = str(tmp_path / "graph.txt")
    api.OutputGraph(gp, d["final_nodes"], avg, labels, d["final_edges"])
    assert filecmp.cmp(gp, os.path.join(refdir, "ref_graph.txt"), shallow=False), "_graph.txt differs"
    # ---- a20: _sv.txt under the harness's stand-in ordering
    flat = np.fromfile(os.path.join(refdir, "components_i32.bin"), dtype=np.int32)
    comps, at = [], 1
    for _ in range(int(flat[0])):
        k = int(flat[at]); comps.append(flat[at + 1: at + 1 + k].tolist()); at += 1 + k
    sp = str(tmp_path / "sv.txt")
    api.WriteBEDPE(sp, ["chr%d" % i for i in range(n_ref)], d["final_nodes"], i32("edges_before_demultiply_i32.bin", 5), comps, rows, d["support"])
    assert filecmp.cmp(sp, os.path.join(refdir, "ref_sv.txt"), shallow=False), "_sv.txt differs"
    n_lines = sum(1 for _ in open(sp))
    assert n_lines >= 1 + min_sv_lines
    return n_lines


@pytest.mark.parametrize("case,n_ref", [("chr17_3k", 1), ("fourchr_6k", 4)])
def test_twins_match_golden_outputs(case, n_ref, built_lib, tmp_path):
    _check_dir(os.path.join(GOLD, case, "ref"), tmp_path, n_ref)


@pytest.mark.parametrize("n,seed,disc,kw", [
    (40000, 61, 0.05, dict(n_genes=40, fusion_support=30)),
    (25000, 62, 0.1, dict(n_genes=12, fusion_support=60)),
])
def test_twins_match_reference_on_fresh_cases(n, seed, disc, kw, built_lib, reference_build, tmp_path):
    """Denser graphs than the goldens: several breakpoint pairs per edge (CountTop's top-5 and its extreme-position fallback),
    ties in the weight sort of WriteBEDPE, tens of BEDPE lines."""
    from squid_b200 import synth
    ref_len = [30000000, 20000000, 5000000, 16569]
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, ref_len, **kw)
    reference_build.run(cp, hp, str(tmp_path / "ref"), extra_args=("--write-outputs",))
    lines = _check_dir(str(tmp_path / "ref"), tmp_path, len(ref_len), min_sv_lines=3)
    print("sv lines", lines)
