"""Drop-in proof (SURVEY.md §8 rows a20 / b): integration/_build/squid_b200_ref is the reference's own, unmodified host code
(ReadRec.cpp, SegmentGraph.cpp, WriteIO.cpp, Config.cpp compiled in place) with BuildNode_STAR, BuildEdges, ExactBreakpoint and
ExactBPConcordantSupport replaced at link time by integration/binding.cpp, i.e. by calls into libsquid_b200.so.  It must write
the same files as the unpatched reference build (oracle/_ref/squid_ref) driven by the same harness: every seam dump, the
`_graph.txt` of OutputGraph and the `_sv.txt` of WriteBEDPE, byte for byte.  (`_sv.txt` under the harness's stand-in ordering:
the GLPK ordering stage is host code out of scope and GLPK is not installed; equality with a real GLPK run stays unpinned.)"""
import filecmp
import os
import subprocess

import numpy as np
import pytest

from tests import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "integration", "_build", "squid_b200_ref")
pytestmark = pytest.mark.gpu

FILES = ["nodes_i32.bin", "nodes_f64.bin", "edges_i32.bin", "chim_after_edges.bin", "final_nodes_i32.bin", "final_nodes_f64.bin", "final_edges_i32.bin", "labels_i32.bin",
         "exactbp_i32.bin", "chim_after_exactbp.bin", "support_i32.bin", "components_i32.bin", "edges_before_demultiply_i32.bin", "ref_graph.txt", "ref_sv.txt"]


@pytest.fixture(scope="module")
def dropin_bin(built_lib):
    subprocess.run(["make", "-C", os.path.join(ROOT, "integration")], capture_output=True, text=True)
    assert os.path.exists(BIN), "integration/_build/squid_b200_ref is missing (built by __graft_entry__.build() where /root/reference exists)"
    return BIN


@pytest.mark.parametrize("n,seed,disc,ref_len,kw,extra", [
    (3000, 3, 0.05, None, {}, []),
    (60000, 71, 0.04, [30000000, 20000000, 5000000, 16569], dict(n_genes=60, fusion_support=25), []),
    (40000, 72, 0.08, None, dict(n_genes=25, fusion_support=40), ["-mq", "3", "-pl", "25", "-dp", "3000", "-di", "2"]),
])
def test_dropin_writes_the_reference_files(n, seed, disc, ref_len, kw, extra, reference_build, dropin_bin, tmp_path):
    cp, hp, *_ = common.write_case(str(tmp_path), n, seed, disc, ref_len, **kw)
    reference_build.run(cp, hp, str(tmp_path / "ref"), extra_args=["--write-outputs"] + extra)
    out = str(tmp_path / "ours")
    os.makedirs(out)
    r = subprocess.run([dropin_bin, cp, hp, out, "--quiet", "--write-outputs"] + extra, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, "rc=%d %s" % (r.returncode, r.stderr[-2000:])
    for f in FILES:
        a, b = os.path.join(str(tmp_path / "ref"), f), os.path.join(out, f)
        assert os.path.exists(a) and os.path.exists(b), f
        assert filecmp.cmp(a, b, shallow=False), "%s differs between the reference build and the drop-in build" % f
    assert sum(1 for _ in open(os.path.join(out, "ref_sv.txt"))) > 1
