"""Shared helpers of the parity tests: make a synthetic case, run the oracle, run the CUDA path, compare."""
import os
import tempfile

import numpy as np

from squid_b200 import sqmb, synth


def write_case(tmpdir, n_pairs, seed, disc_frac=0.02, ref_len=None, **kw):
    conc, chim, info = synth.make_case(n_pairs, ref_len=ref_len if ref_len is not None else synth.CHR17_LEN, seed=seed, disc_frac=disc_frac, **kw)
    cp, hp = os.path.join(tmpdir, "conc.sqmb"), os.path.join(tmpdir, "chim.sqmb")
    sqmb.write_sqmb(cp, conc); sqmb.write_sqmb(hp, chim)
    return cp, hp, conc, chim, info


def build_emul(out_dir) -> str:
    """Compiles the CPU stepping harness (tests/emul) into `out_dir` (not into the repository tree, which may be read-only)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    os.makedirs(str(out_dir), exist_ok=True)
    out = os.path.join(str(out_dir), "emul")
    srcs = ["tests/emul/emul_main.cpp", "squid_b200/csrc/host/readrec.cpp", "squid_b200/csrc/host/chimeric.cpp", "squid_b200/csrc/host/prepass.cpp"]
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-fopenmp", "-I", "include", "-I", "squid_b200/csrc", "-o", out] + srcs + ["-lpthread"],
                       cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def run_cuda(cp, hp, device=0, do_cov_with=None):
    """Full hot path through the C ABI.  Returns dict with nodes/avgdepth/edges/chim_after_edges (+coverage map)."""
    from squid_b200 import api
    case = api.HostCase(cp, hp)
    g = api.SegmentGraph(case.config, case.ref_len, device=device)
    nodes = g.BuildNode_STAR(case.chimeric, case.batch)
    edges = g.BuildEdges()
    out = {
        "nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32),
        "avgdepth": nodes.AvgDepth, "edges": edges.table(), "chim_after_edges": case.chimeric.block_table(),
        "read_len": case.config.ReadLen, "graph": g, "case": case,
    }
    if do_cov_with is not None:
        ref = do_cov_with
        from oracle import pyref
        out["support"] = g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref))
    return out


def bp_array(chr_pos) -> np.ndarray:
    """Sorted (chr, pos) int32 rows, duplicates kept (a breakpoint list as ExactBPConcordantSupport builds it)."""
    a = np.asarray(chr_pos, dtype=np.int64).reshape(-1, 2)
    a = a[np.lexsort((a[:, 1], a[:, 0]))]
    return np.ascontiguousarray(a.astype(np.int32))


def chr_start_bps(ref_len, offsets=(0, 1, 99, 4999)) -> np.ndarray:
    """Breakpoints just right of every chromosome start: there a negative -dp makes pos + dist negative."""
    return bp_array([(c, p) for c in range(len(ref_len)) for p in offsets if p < ref_len[c]])


def bp_families(ref_len, nodes, conc, seed) -> dict:
    """Breakpoint lists of the shapes that drive the coverage chain (DESIGN §7), from a case's segment table `nodes` (rows chr,
    pos, len, support) and its concordant records `conc` (AlnTable):
      uniform   random positions over every chromosome (also those without records), plus 0, ref_len-1 and ref_len
      dups      runs of 1..60 copies of one breakpoint at record starts and segment ends (a fusion hub)
      dense     every position of a 3000-bp window in the highest-Support segment (> 256 breakpoints under one rank block)
      before    every breakpoint before the first record
      after     every breakpoint on the last record's chromosome or later (t unresolved by the stream)
      one       K = 1
      empty     K = 0"""
    rng = np.random.default_rng(seed)
    rl = np.asarray(ref_len, np.int64)
    n_ref = rl.shape[0]
    out = {}
    c = rng.integers(0, n_ref, 3000)
    u = [np.stack([c, (rng.random(3000) * rl[c]).astype(np.int64)], 1)]
    u += [np.array([(k, 0), (k, rl[k] - 1), (k, rl[k])]) for k in range(n_ref)]
    out["uniform"] = bp_array(np.concatenate(u))
    m = conc.ref_id >= 0
    starts = np.stack([conc.ref_id[m], conc.pos[m]], 1).astype(np.int64)
    ends = np.stack([nodes[:, 0], nodes[:, 1] + nodes[:, 2]], 1).astype(np.int64)
    hubs = np.concatenate([starts[rng.integers(0, starts.shape[0], 200)], ends[rng.integers(0, ends.shape[0], 100)]])
    out["dups"] = bp_array(np.repeat(hubs, rng.integers(1, 61, hubs.shape[0]), axis=0))
    top = nodes[np.argmax(nodes[:, 3])]
    w0 = max(0, int(top[1]) + int(top[2]) // 2 - 1500)
    out["dense"] = bp_array([(int(top[0]), p) for p in range(w0, min(w0 + 3000, int(rl[top[0]])))])
    first, last = starts[0], int(starts[:, 0].max())  # the stream is coordinate-sorted
    out["before"] = bp_array([(k, p) for k in range(int(first[0])) for p in (0, 5, int(rl[k]) - 1)] +
                             [(int(first[0]), p) for p in rng.integers(0, max(1, int(first[1])), 50) if p < first[1]])
    out["after"] = bp_array([(k, int(p)) for k in range(last, n_ref) for p in rng.integers(0, rl[k], 100)])
    out["one"] = bp_array(starts[rng.integers(0, starts.shape[0], 1)])
    out["empty"] = bp_array(np.zeros((0, 2)))
    return out


def assert_same(ref, got, what=("nodes", "avgdepth", "edges", "chim_after_edges")):
    for k in what:
        a, b = ref[k], got[k]
        assert a.shape == b.shape, "%s: shape %s vs %s" % (k, a.shape, b.shape)
        if not np.array_equal(a, b):
            bad = np.flatnonzero((a != b).reshape(a.shape[0], -1).any(axis=1))[:5]
            raise AssertionError("%s differs at rows %s: ref %s got %s" % (k, bad, a[bad], b[bad]))
