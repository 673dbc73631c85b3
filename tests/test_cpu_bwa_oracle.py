"""BWA mode (SURVEY.md §8 rows a8 / a14: BuildNode_BWA, RawEdges) is not on the device yet.  What exists is its checker: the
reference's own sources run in BWA mode on merged synthetic input (oracle/ref_harness.cpp --bwa), with the seam dumps
committed as golden fixtures (tests/golden/bwa_*).  These tests keep that pin honest: where the reference build is available it
must reproduce the committed dumps bit for bit, the fixtures must be structurally sound, and the library must refuse
using_star = 0 loudly instead of answering with the STAR rules."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
CASES = ["bwa_chr17_3k", "bwa_fourchr_6k"]


@pytest.mark.parametrize("case", CASES)
def test_reference_build_reproduces_bwa_golden(case, reference_build, tmp_path):
    got = reference_build.run(os.path.join(GOLD, case, "all.sqmb"), "-", str(tmp_path), extra_args=("--bwa",))
    want = reference_build.load_dumps(os.path.join(GOLD, case, "ref"))
    for k in ("nodes", "avgdepth", "edges", "chim_after_edges", "final_nodes", "final_edges", "exactbp", "support"):
        assert want[k].shape == got[k].shape and np.array_equal(want[k], got[k]), k
    assert got["read_len"] == want["read_len"] == 100


@pytest.mark.parametrize("case", CASES)
def test_bwa_golden_is_a_graph(case):
    from oracle import pyref
    from squid_b200 import sqmb  # noqa: F401  (the fixture's input format)
    d = pyref.load_dumps(os.path.join(GOLD, case, "ref"))
    n = d["nodes"]
    assert n.shape[0] > 10 and (n[:, 2] > 0).all()
    for c in np.unique(n[:, 0]):  # segments tile every chromosome (SegmentGraph.cpp:1120-1175)
        m = n[n[:, 0] == c]
        assert m[0, 1] == 0 and np.array_equal(m[1:, 1], (m[:-1, 1] + m[:-1, 2]))
    e = d["edges"]
    assert e.shape[0] > 10 and (e[:, 0] <= e[:, 1]).all() and (e[:, 4] > 0).all() and e[:, :2].max() < n.shape[0]
    assert d["chim_after_edges"].shape[0] > 0  # RawEdges rebuilt Chimrecord from the partially aligned reads (:1883-1926)


def test_library_refuses_bwa_mode(built_lib):
    from squid_b200 import api
    L = api.lib()
    cfg = api.Config(UsingSTAR=False, ReadLen=100).as_struct()
    ref_len = np.array([1000000], np.int32)
    h = C.c_void_p()
    rc = L.sqg_create(C.byref(h), C.byref(cfg), ref_len.ctypes.data, 1, 0)
    assert rc in (api.SQG_EUNSUPPORTED, api.SQG_ENODEVICE)  # (no device in the CPU container: refused even earlier)
    if h:
        L.sqg_destroy(h)
