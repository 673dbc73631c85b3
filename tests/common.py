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


# Cases of the segment-table families (tests/test_cpu_emul.py, tests/test_gpu_set_nodes.py): n_pairs, seed, disc_frac, ref_len, kwargs
FAMILY_CASES = {
    "chr17_s17": (20000, 17, 0.02, None, {}),
    "fourchr_s418": (60000, 418, 0.1, [30000000, 20000000, 5000000, 16569], {"fusion_support": 100, "exon_len": (20, 170), "intron_len": (60, 400)}),
    "grch38_s1003": (100000, 1003, 0.02, "grch38", {}),
    "short_s37": (30000, 37, 0.2, None, {"n_genes": 100, "fusion_support": 20, "min_block": 1}),  # 1-3 bp blocks meet 1-6 bp segments
}
# -dp 3000 -di 2: the index distance of an edge decides IsDiscordant on the dense tables
FAMILY_OPTS = ["-dp", "3000", "-di", "2"]


def family_case(tmpdir, name):
    """Writes case `name` of FAMILY_CASES; returns (conc path, chim path, ref_len, families)."""
    from oracle import pyref
    n, seed, disc, rl, kw = FAMILY_CASES[name]
    cp, hp, conc, chim, _ = write_case(str(tmpdir), n, seed, disc, synth.GRCH38_LEN if rl == "grch38" else rl, **kw)
    built = pyref.run_restate(cp, hp, os.path.join(str(tmpdir), "built"), stop_after=2)["nodes"]
    return cp, hp, np.asarray(conc.ref_len, np.int64), node_families((conc.ref_len, conc, chim), built, seed)


def aligned_blocks(tab) -> np.ndarray:
    """(chr, start, end) rows of the aligned blocks of every mapped record of an AlnTable: maximal runs of M/I/D/=/X
    operations between S, H and N, as the record decoder cuts them (ReadRec.cpp:46-87)."""
    cig = np.asarray(tab.cigar, np.int64)
    op, ln = cig & 15, cig >> 4
    off = np.asarray(tab.cigar_off, np.int64)
    rec = np.repeat(np.arange(tab.n, dtype=np.int64), np.diff(off))
    adv = np.where(np.isin(op, (0, 2, 3, 7, 8)), ln, 0)  # reference-consuming operations
    ex = np.cumsum(adv) - adv
    gp = np.asarray(tab.pos, np.int64)[rec] + ex - ex[off[rec]]  # reference position at each operation
    inb = np.isin(op, (0, 1, 2, 7, 8))
    start = inb & (np.r_[True, rec[1:] != rec[:-1]] | ~np.r_[False, inb[:-1]])
    run = np.cumsum(start) - 1
    keep = inb & (np.asarray(tab.ref_id)[rec] >= 0) & ((np.asarray(tab.flag)[rec] & 4) == 0)
    if not keep.any():
        return np.zeros((0, 3), np.int64)
    r = run[keep]
    first = np.r_[True, r[1:] != r[:-1]]
    last = np.r_[r[1:] != r[:-1], True]
    g0, g1 = gp[keep], gp[keep] + adv[keep]
    return np.stack([np.asarray(tab.ref_id, np.int64)[rec[keep]][first], g0[first], g1[last]], 1)


def _tile(ref_len, cuts_by_chr) -> np.ndarray:
    """Segment table (chr, pos, len) of each chromosome cut at the given positions (those inside (0, ref_len) are used)."""
    rows = []
    for c, L in enumerate(np.asarray(ref_len, np.int64)):
        cu = np.asarray(cuts_by_chr.get(c, ()), np.int64)
        b = np.unique(np.concatenate([[0, L], cu[(cu > 0) & (cu < L)]]))
        rows.append(np.stack([np.full(b.shape[0] - 1, c), b[:-1], np.diff(b)], 1))
    return np.ascontiguousarray(np.concatenate(rows).astype(np.int32))


def _starts(nodes) -> dict:
    out = {}
    for c in np.unique(nodes[:, 0]):
        out[int(c)] = nodes[nodes[:, 0] == c, 1].astype(np.int64)
    return out


MICRO_SPAN = 20000


def node_families(case, nodes, seed) -> dict:
    """Segment tables for the graph-reload seam (sqg_set_nodes), built from a case's own segment table `nodes` (rows chr, pos,
    len, ...) and records.  `case` = (ref_len, concordant AlnTable, chimeric AlnTable).  Every table tiles every chromosome
    from 0 to its length with segments of positive length:
      built        the table BuildNode_STAR built (the control)
      block_edges  built, cut at the exact start and end of a random 20 % of the aligned blocks: boundaries on block ends
                   (the spanning-block fallback, SegmentGraph.cpp:1408-1409)
      near_edges   built, cut 1..6 bp beside the start or end of a random 20 % of the blocks: blocks fit two or three segments
                   within LocateRead's tolerance of 5, so reads become hint-sensitive
      micro        built, with the spans of 3 record tiles re-cut into segments of cycling length 1..6 bp:
                   ~150 segments per 512-bp bin, long hint chains, more distinct edges per tile than its table holds
      bins         built, with up to 2 Mb of the most-read chromosome re-cut into segments of 512, 511, 513, ... bp from a
                   multiple of 512: segment ends on and beside the bin boundaries of the position index
      coarse       one segment per chromosome
      random       cuts of a seeded process whose mean spacing changes region by region between 10 bp and 100 kb"""
    ref_len, conc, chim = case
    rl = np.asarray(ref_len, np.int64)
    nodes = np.asarray(nodes)
    rng = np.random.default_rng(seed)
    blk = np.concatenate([aligned_blocks(conc), aligned_blocks(chim)])
    base = _starts(nodes)

    def with_cuts(extra):  # extra: (chr, pos) rows added to the built table's boundaries
        d = {c: [v] for c, v in base.items()}
        for c in np.unique(extra[:, 0]):
            d.setdefault(int(c), []).append(extra[extra[:, 0] == c, 1])
        return _tile(rl, {c: np.concatenate(v) for c, v in d.items()})

    def replace_window(tab, c, lo, hi, cuts):  # tab's boundaries on chromosome c inside [lo, hi) replaced by `cuts`
        d = _starts(tab)
        s = d[c]
        d[c] = np.concatenate([s[(s < lo) | (s >= hi)], [lo, hi], cuts])
        return _tile(rl, d)

    out = {"built": np.ascontiguousarray(nodes[:, :3].astype(np.int32))}
    pick = blk[rng.random(blk.shape[0]) < 0.2]
    out["block_edges"] = with_cuts(np.concatenate([pick[:, [0, 1]], pick[:, [0, 2]]]))
    pick = blk[rng.random(blk.shape[0]) < 0.2]
    side = np.where(rng.random(pick.shape[0]) < 0.5, pick[:, 1], pick[:, 2])
    out["near_edges"] = with_cuts(np.stack([pick[:, 0], side + rng.choice([-6, -5, -4, -3, -2, -1, 1, 2, 3, 4, 5, 6], pick.shape[0])], 1))
    t = out["built"]
    # windows over whole 512-record tiles (the edge pass's tile) whose records span about MICRO_SPAN bp: re-cut, such a tile
    # sees thousands of segments and can emit more distinct keys than its table holds (where all its reads pile up in a few
    # hundred bp, a tile cannot)
    pos, rid = np.asarray(conc.pos, np.int64), np.asarray(conc.ref_id, np.int64)
    nt = rid.shape[0] // 512
    t0, t1 = np.arange(nt) * 512, np.arange(nt) * 512 + 511
    ok = (rid[t0] >= 0) & (rid[t0] == rid[t1])
    span = np.where(ok, pos[t1] - pos[t0], 1 << 40)
    taken = []
    for k in np.argsort(np.abs(span - MICRO_SPAN), kind="stable"):
        if len(taken) == 3 or not ok[k]:
            break
        c, lo, hi = int(rid[t0[k]]), max(0, int(pos[t0[k]]) - 200), min(int(rl[rid[t0[k]]]), int(pos[t1[k]]) + 400)
        if any(c == q[0] and lo < q[2] and q[1] < hi for q in taken):
            continue
        taken.append((c, lo, hi))
        cuts = lo + np.cumsum(np.tile(np.arange(1, 7), (hi - lo) // 3 + 1))
        t = replace_window(t, c, lo, hi, cuts[cuts < hi])
    out["micro"] = t
    c = int(np.bincount(blk[:, 0], minlength=rl.shape[0]).argmax())
    mid = int(np.median(blk[blk[:, 0] == c, 1]))
    lo = max(0, min(mid - (1 << 20), int(rl[c]) - (2 << 20))) // 512 * 512
    hi = min(int(rl[c]), lo + (2 << 20))
    cuts = lo + np.cumsum(np.tile([512, 511, 513, 512, 513, 511], (hi - lo) // 3000 + 1))
    out["bins"] = replace_window(out["built"], c, lo, hi, cuts[cuts < hi])
    out["coarse"] = _tile(rl, {})
    d = {}
    for k, L in enumerate(rl):
        cu, x = [], 0.0
        while x < L:
            m = 10.0 ** rng.uniform(1, 5)  # mean spacing of this region
            g = rng.exponential(m, int(rng.integers(20, 400)))
            cu.append(x + np.cumsum(np.maximum(g, 1.0)))
            x = cu[-1][-1]
        d[k] = np.concatenate(cu).astype(np.int64)
    out["random"] = _tile(rl, d)
    for tab in out.values():
        check_tiling(rl, tab)
    return out


def check_tiling(ref_len, tab):
    """Asserts the contract of sqg_set_nodes: sorted, positive lengths, contiguous, every chromosome from 0 to its length."""
    tab = np.asarray(tab, np.int64)
    assert np.all(tab[:, 2] > 0)
    assert np.array_equal(np.unique(tab[:, 0]), np.arange(len(ref_len)))
    for c, L in enumerate(ref_len):
        s = tab[tab[:, 0] == c]
        assert s[0, 1] == 0 and s[-1, 1] + s[-1, 2] == L and np.array_equal(s[1:, 1], s[:-1, 1] + s[:-1, 2])
    assert np.all(np.diff(tab[:, 0]) >= 0)


def assert_same(ref, got, what=("nodes", "avgdepth", "edges", "chim_after_edges")):
    for k in what:
        a, b = ref[k], got[k]
        assert a.shape == b.shape, "%s: shape %s vs %s" % (k, a.shape, b.shape)
        if not np.array_equal(a, b):
            bad = np.flatnonzero((a != b).reshape(a.shape[0], -1).any(axis=1))[:5]
            raise AssertionError("%s differs at rows %s: ref %s got %s" % (k, bad, a[bad], b[bad]))
