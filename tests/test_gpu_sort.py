"""The device twin of the chimeric pre-pass sort (squid_b200/csrc/sq_gpusort.cuh) against std::sort on the host: the same
permutation, payload included, for keys with many ties (what decides which equal (RefID,RefPos) block the reference sees
first, SURVEY.md App. A-11), sorted, reversed and organ-pipe inputs, across the leaf / multi-level size boundaries."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(n, seed, rng, pattern):
    from squid_b200 import api
    L = api.lib()
    L.sqg_selftest_gpu_sort.argtypes = [C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_float)]
    ms = C.c_float(-1)
    return L.sqg_selftest_gpu_sort(0, n, seed, rng, pattern, C.byref(ms)), ms.value


@pytest.mark.parametrize("n", [2, 3, 16, 17, 100, 1024, 1025, 2049, 5000, 40000, 300000, 1200000])
def test_random_keys_with_ties(built_lib, n):
    for seed, rng in ((1, 0), (2, 3), (3, 50), (4, max(2, n // 7)), (5, 1 << 40)):  # range 0: every key equal
        v, ms = _run(n, seed, rng, 0)
        assert v == 1, "n=%d range=%d: verdict %d" % (n, rng, v)


@pytest.mark.parametrize("pattern", [1, 2, 3])
def test_structured_inputs(built_lib, pattern):
    for n in (1000, 1025, 70000, 900000):
        v, ms = _run(n, 7, 0, pattern)
        # organ-pipe inputs can exhaust std::sort's depth budget: the device then declines (2) and the CPU twin takes over
        assert v == 1 or (pattern == 3 and v == 2), "pattern %d n=%d: verdict %d" % (pattern, n, v)


def test_prepass_uses_the_device_sort(tmp_path, built_lib, ref_oracle):
    """End to end on a small input: the pre-pass sort runs on the device, same segments / edges as the reference build."""
    from tests import common
    cp, hp, *_ = common.write_case(str(tmp_path), 60000, 1031, 0.05, fusion_support=10)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp)
    assert got["graph"].stat("device_sort_status") == 0
    common.assert_same(ref, got)


def _organ_pipe_case(tmpdir, n_pairs=30000, seed=41, n_pipe=2500):
    """A concordant stream whose ReadsOther keys (the non-first blocks in record order) are in organ-pipe order, on which
    std::sort's quicksort exhausts its depth budget: n_pipe single-block records on chromosome 0 become spliced records whose
    second block starts at 2.2 Mb + 40 * min(i, n_pipe - 1 - i).  Every 7th second block is 3 bp long, so the depth pass has
    short ReadsOther blocks; long exons keep the generator's own spliced records few."""
    from squid_b200 import sqmb, synth
    conc, chim, _ = synth.make_case(n_pairs, ref_len=[3000000, 2000000], seed=seed, disc_frac=0.05, n_genes=12, fusion_support=10,
                                    exon_len=(15000, 30000), intron_len=(200, 2000))
    off = conc.cigar_off.astype(np.int64)
    first = conc.cigar[off[:-1]]
    cand = np.flatnonzero((off[1:] - off[:-1] == 1) & (first & 15 == sqmb.OP_M) & (first >> 4 >= 40) & (conc.ref_id == 0) & (conc.pos < 2000000))
    pick = cand[np.linspace(0, cand.size - 1, n_pipe).astype(np.int64)]
    assert np.unique(pick).size == n_pipe
    cig = [conc.cigar[off[r]:off[r + 1]] for r in range(conc.n)]
    for i, r in enumerate(pick):
        read, b = int(first[r] >> 4), 3 if i % 7 == 0 else 20
        a, s = read - b, 2200000 + 40 * min(i, n_pipe - 1 - i)
        cig[r] = np.array([(a << 4) | sqmb.OP_M, ((s - int(conc.pos[r]) - a) << 4) | sqmb.OP_N, (b << 4) | sqmb.OP_M], np.uint32)
    conc.cigar_off = np.concatenate([[0], np.cumsum([c.size for c in cig])]).astype(np.uint32)
    conc.cigar = np.concatenate(cig).astype(np.uint32)
    cp, hp = os.path.join(tmpdir, "conc.sqmb"), os.path.join(tmpdir, "chim.sqmb")
    sqmb.write_sqmb(cp, conc); sqmb.write_sqmb(hp, chim)
    return cp, hp


def test_reads_other_sort_falls_back_to_the_cpu_twin(tmp_path, built_lib, ref_oracle):
    """The replayed sort(ReadsOther) of the depth pass on keys the device sort declines: the CPU twin sorts them, and nodes,
    Support, AvgDepth and edges still equal the oracle's.  SQG_OTHER_SORT=1 (the replay even without order-dependent ties) is
    read once per process, so the CUDA path runs in a process of its own."""
    from tests import common
    cp, hp = _organ_pipe_case(str(tmp_path))
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    out = str(tmp_path / "got.npz")
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from tests import common\n"
            "got = common.run_cuda(%r, %r)\n"
            "g = got['graph']\n"
            "np.savez(%r, other_sort_status=g.stat('other_sort_status'), short_other_blocks=g.stat('short_other_blocks'),\n"
            "         **{k: got[k] for k in ('nodes', 'avgdepth', 'edges', 'chim_after_edges')})\n") % (ROOT, cp, hp, out)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, SQG_OTHER_SORT="1"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    z = np.load(out)
    assert int(z["short_other_blocks"]) > 0
    assert int(z["other_sort_status"]) in (2, 3), "the device sort did not decline: status %d" % int(z["other_sort_status"])
    common.assert_same(ref, {k: z[k] for k in ("nodes", "avgdepth", "edges", "chim_after_edges")})
