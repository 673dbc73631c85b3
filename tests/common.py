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


# ---- concordant-stream families of the classification pass (tests/test_cpu_emul.py, tests/test_gpu_classify.py) -------------
TILE = 512  # records per classification tile (sq_stream.cuh kTile)
FAMILY_STREAMS = ["base", "unmapped_mates", "unmapped_tail", "filtered_runs", "dup_shapes", "many_chr", "long_first_block", "dense_tiles"]
FILTERED_RUN_LENGTHS = (31, 32, 33, 64, 511, 512, 513, 1500)


def _cigar_str(tab, r) -> str:
    c = np.asarray(tab.cigar[int(tab.cigar_off[r]):int(tab.cigar_off[r + 1])], np.int64)
    return "".join("%d%s" % (x >> 4, sqmb.CIGAR_OPS[x & 15]) for x in c)


def _record(tab, r) -> dict:
    """Record r of an AlnTable as a sqmb.from_records row."""
    a = int(tab.aux[r])
    d = dict(ref_id=int(tab.ref_id[r]), pos=int(tab.pos[r]), cigar=_cigar_str(tab, r), flag=int(tab.flag[r]), mate_ref_id=int(tab.mate_ref_id[r]),
             mate_pos=int(tab.mate_pos[r]), mapq=int(tab.mapq[r]), xa=bool(a & sqmb.AUX_XA), name_id=int(tab.name_id[r]),
             name_suffix=bool(a & sqmb.AUX_NAME_SUFFIX), lowrun=int(tab.lowrun[r]), polya=int(tab.polya[r]))
    if a & sqmb.AUX_IH:
        d["ih"] = int(tab.ih[r])
    return d


def _passes_gate(rec, chim_names) -> bool:
    """SegmentGraph.cpp:302 at the default -mq (255), for a from_records row whose name has no /1 /2 suffix."""
    return not (rec.get("xa") or rec.get("ih", 0) > 1 or rec["mapq"] < 255 or rec["flag"] & (sqmb.FLAG_DUP | sqmb.FLAG_UNMAPPED) or
                rec["ref_id"] < 0 or (not rec.get("name_suffix") and rec["name_id"] in chim_names))


def _gate_failing_clone(rec, k, chim_name):
    """A copy of `rec` that fails the record gate, the reason cycling with k: DUP flag, mapq below -mq, XA, IH > 1, ChimName."""
    c = dict(rec)
    c.pop("ih", None)
    c["name_suffix"] = False
    why = k % 5
    if why == 0: c["flag"] = rec["flag"] | sqmb.FLAG_DUP
    elif why == 1: c["mapq"] = 3
    elif why == 2: c["xa"] = True
    elif why == 3: c["ih"] = 2
    else: c["name_id"] = chim_name
    return c


def stream_families(conc, chim, seed) -> dict:
    """Coordinate-sorted concordant streams (AlnTable) that drive the classification pass (sq_phase1.cuh) down the paths a
    synthetic case does not reach, each derived from the case's concordant records `conc` (chimeric records `chim` give the
    ChimName gate's names):
      base              the case as generated
      unmapped_mates    5 % of the proper pairs lose one mate, SAM convention: flag 0x4 at the mate's position, no CIGAR; the
                        partner gets 0x8
      unmapped_tail     2.5 tiles of unmapped records (ref_id -1) at the end; the last mapped tile holds unmapped records too
      filtered_runs     runs of 31..1500 gate-failing clones (DUP, mapq, XA, IH, ChimName) at -40..+40 around tile starts and over
                        records 0..600, each followed by a duplicate of the last gate-passing record before it
      dup_shapes        hand-built Equal pairs and near-misses (mate-swapped 15-bp blocks, multi-block lists whose CIGAR order
                        is not their read order, empty lists with and without a mate block) across tile boundaries and filtered
                        runs; the stream starts with an empty record that equals the default-constructed ReadRec_t
      many_chr          48 contigs of a few hundred records each, chromosome boundaries at tile start -1, 0 and +1
      long_first_block  concordant records whose first block is 65534, 65535, 65536 or 70100 bp long
    (dense_tiles, tiles with more than kTileBlkCap blocks, is a case of its own: dense_tiles_case.)"""
    rng = np.random.default_rng(seed)
    chim_names = set(int(x) for x in np.asarray(chim.name_id))
    chim_name = int(np.asarray(chim.name_id)[0])
    ref_len = np.asarray(conc.ref_len)
    n = conc.n
    out = {"base": conc}

    # unmapped_mates
    order = np.argsort(np.asarray(conc.name_id), kind="stable")
    nid = np.asarray(conc.name_id)[order]
    pair = np.flatnonzero(nid[1:] == nid[:-1])
    a, b = order[pair], order[pair + 1]
    ok = ((conc.flag[a] & sqmb.FLAG_PROPER) != 0) & ((conc.flag[b] & sqmb.FLAG_PROPER) != 0)
    a, b = a[ok], b[ok]
    pick = rng.random(a.shape[0]) < 0.05
    swap = rng.random(a.shape[0]) < 0.5
    lost, kept = np.where(swap, b, a)[pick], np.where(swap, a, b)[pick]
    t = conc.take(np.arange(n))
    t.flag[lost] = (t.flag[lost] | sqmb.FLAG_UNMAPPED) & ~np.uint16(sqmb.FLAG_PROPER | sqmb.FLAG_MATE_REVERSE)
    t.ref_id[lost], t.pos[lost] = t.ref_id[kept], t.pos[kept]
    t.mate_ref_id[lost], t.mate_pos[lost] = t.ref_id[kept], t.pos[kept]
    t.flag[kept] = (t.flag[kept] | sqmb.FLAG_MATE_UNMAPPED) & ~np.uint16(sqmb.FLAG_PROPER)
    t.mate_pos[kept] = t.pos[kept]
    lens = np.diff(t.cigar_off.astype(np.int64))
    t.cigar = t.cigar[np.repeat(~np.isin(np.arange(n), lost), lens)]
    lens[lost] = 0
    t.cigar_off = np.r_[0, np.cumsum(lens)].astype(np.uint32)
    out["unmapped_mates"] = t.sorted_by_coordinate()

    # unmapped_tail: 2.5 tiles, the mapped records ending inside a tile
    base = conc.take(np.arange(n - (n % TILE) - 200 if n % TILE < 200 else n))
    u = conc.take(rng.integers(0, n, TILE * 5 // 2))
    u.ref_id[:] = -1; u.pos[:] = -1; u.mate_ref_id[:] = -1; u.mate_pos[:] = -1
    u.flag[:] = sqmb.FLAG_PAIRED | sqmb.FLAG_UNMAPPED | sqmb.FLAG_MATE_UNMAPPED | sqmb.FLAG_FIRST
    u.cigar = np.zeros(0, np.uint32); u.cigar_off = np.zeros(u.n + 1, np.uint32)
    out["unmapped_tail"] = sqmb.concat([base, u])

    recs = [_record(conc, r) for r in range(n)]

    # filtered_runs
    starts = {}  # output index -> run length
    offs = [-40, -33, -1, 0, 1, 7, 31, 40]
    t_at = 3
    for k, L in enumerate(FILTERED_RUN_LENGTHS * 2):
        starts[t_at * TILE + offs[k % len(offs)]] = L
        t_at += 2 + (L + 40) // TILE
    outl, last_ok, k = [], None, 0
    outl += [_gate_failing_clone(recs[0], j, chim_name) for j in range(601)]  # records 0..600: the first tile has no gate-passing record
    pending = sorted(starts)
    for r in recs:
        # a run starts at its planned index, or a record later when the record before it is not gate-passing (the duplicate
        # after the run repeats that record, so both must sit at its position)
        if pending and len(outl) >= pending[0] and last_ok is not None and outl[-1] is last_ok:
            L = starts[pending.pop(0)]
            outl += [_gate_failing_clone(last_ok, k + j, chim_name) for j in range(L)]
            k += L
            outl.append(dict(last_ok))
        outl.append(r)
        if _passes_gate(r, chim_names):
            last_ok = r
    assert not pending
    out["filtered_runs"] = sqmb.from_records(ref_len, outl)

    # dup_shapes: (l, r) pairs written next to each other; `equal` says whether Equal(l, r) holds
    def pair_shapes(c, p, q, nm):
        """Pairs at chromosome c, l at position p, r at q > p (nothing else lies between p and q in the stream)."""
        fl, fs = 0x1 | 0x2 | 0x20 | 0x40, 0x1 | 0x2 | 0x10 | 0x80  # forward first mate, reverse second mate
        mk = lambda pos, cig, flag, mpos, **kw: dict(dict(ref_id=c, pos=pos, cigar=cig, flag=flag, mate_ref_id=c, mate_pos=mpos, mapq=255,
                                                          name_id=nm), **kw)
        return [
            # mate-swapped match: own(l) == mate block of r and mate block of l == own(r), 15-bp blocks
            (mk(p, "15M", fl, q), mk(q, "15M", fs, p), True),
            (mk(p, "15M", fl, q), mk(q, "16M", fs, p), False),           # own(r) one base longer
            (mk(p, "15M", fl, q), mk(q, "15M", fs, p + 1), False),       # mate of r one base off
            # several blocks: same CIGAR, forward vs reverse strand => the read-position order of the blocks differs
            (mk(p, "20M100N30M", fl, p + 400), mk(p, "20M100N30M", fl | 0x10, p + 400), False),
            (mk(p, "20M100N30M", fl | 0x10, p + 400), mk(p, "20M100N30M", fl | 0x10, p + 400), True),
            (mk(p, "20M100N30M", fl | 0x10, p + 400), mk(p, "20M101N29M", fl | 0x10, p + 400), False),   # second block one base off
            (mk(p, "5S20M100N30M", fl | 0x10, p + 400), mk(p, "20M100N30M5S", fl | 0x10, p + 400), True),  # read positions differ, blocks equal
            # empty own lists (the block is a poly-A run), with and without a mate block
            (mk(p, "40M", fl, p + 300, polya=1), mk(p, "40M", fl, p + 300, polya=1), True),
            (mk(p, "40M", fl, p + 300, polya=1), mk(p, "40M", fl, p + 301, polya=1), False),
            (mk(p, "40M", fl | 0x8, -1, polya=1, mate_ref_id=-1), mk(p, "40M", fl | 0x8, -1, polya=1, mate_ref_id=-1), True),
            (mk(p, "40M", fl | 0x8, -1, polya=1, mate_ref_id=-1), mk(p, "40M", fl, p + 300, polya=1), False),
        ]
    outl = [dict(ref_id=int(conc.ref_id[0]), pos=int(conc.pos[0]), cigar="40M", flag=0x1 | 0x8 | 0x40, mapq=255, name_id=1 << 40, polya=1)]
    shapes_done, where, nm = 0, 0, 1 << 40
    n_shapes = len(pair_shapes(0, 0, 1, 0))
    for i, r in enumerate(recs):
        nxt = recs[i + 1] if i + 1 < n else None
        if (shapes_done < 3 * n_shapes and nxt is not None and nxt["ref_id"] == r["ref_id"] and nxt["pos"] > r["pos"] + 2 and
                len(outl) >= where):
            at_edge = len(outl) % TILE == TILE - 2  # then l is the tile's last record and r the next tile's first
            mode = shapes_done // n_shapes  # 0: across a tile boundary, 1: inside a tile, 2: a filtered run between l and r
            if mode != 0 or at_edge:
                outl.append(r)
                nm += 1
                l_, r_, eq = pair_shapes(r["ref_id"], r["pos"] + 1, nxt["pos"] - 1, nm)[shapes_done % n_shapes]
                outl.append(dict(l_, equal=eq))
                if mode == 2:
                    outl += [_gate_failing_clone(l_, j, chim_name) for j in range(40)]
                outl.append(dict(r_, equal=eq))
                shapes_done += 1
                where = len(outl) + (TILE if mode == 0 else 97)
                continue
        outl.append(r)
    assert shapes_done == 3 * n_shapes, shapes_done
    out["dup_shapes"] = sqmb.from_records(ref_len, [{k: v for k, v in d.items() if k != "equal"} for d in outl])

    # many_chr: contig boundaries at tile starts -1, 0, +1; every contig as long as the case's first chromosome
    cuts = [k * TILE + (k % 3) - 1 for k in range(1, n // TILE)]
    cuts = [c for c in cuts if c < n][: 47]
    chrom = np.zeros(n, np.int32)
    for c in cuts:
        chrom[c:] += 1
    t = conc.take(np.arange(n))
    mate_of = np.full(n, -1, np.int64)
    mate_of[order[pair]] = order[pair + 1]
    mate_of[order[pair + 1]] = order[pair]
    t.ref_id = chrom.copy()
    has = (mate_of >= 0) & (t.mate_ref_id >= 0)
    t.mate_ref_id = np.where(has, chrom[np.maximum(mate_of, 0)], np.where(t.mate_ref_id >= 0, chrom, -1)).astype(np.int32)
    t.ref_len = np.full(int(chrom[-1]) + 1, int(ref_len[0]), np.int32)
    out["many_chr"] = t

    # long_first_block: first blocks of 65534, 65535, 65536 and 70100 bp (a deletion does not split a block)
    t = [dict(x) for x in recs]
    cand = [i for i, x in enumerate(t) if x["flag"] & 0x2 and x["cigar"].endswith("M") and x["cigar"].count("M") == 1 and
            x["cigar"][:-1].isdigit() and x["flag"] & 0xC0]
    for j, i in enumerate(rng.choice(cand, 60, replace=False)):
        L = int(t[i]["cigar"][:-1])
        want = (65534, 65535, 65536, 70100)[j % 4]
        t[i]["cigar"] = "%dM%dD%dM" % (L // 2, want - L, L - L // 2)
    out["long_first_block"] = sqmb.from_records(ref_len, t)
    for name, tab in out.items():
        check_sorted(tab)
    return out


def check_sorted(tab):
    key = np.where(tab.ref_id < 0, np.int64(1) << 62, (tab.ref_id.astype(np.int64) << 32) | tab.pos.astype(np.int64))
    assert np.all(np.diff(key) >= 0)


def dense_tiles_case():
    """A case whose exons are 20-170 bp: some tiles with more than 1152 aligned blocks are read from HBM instead of being staged."""
    return synth.make_case(12000, ref_len=synth.CHR17_LEN, seed=71, disc_frac=0.02, exon_len=(20, 170), intron_len=(60, 400))


def write_stream_families(tmpdir, seed=17):
    """SQMB files of every stream family (common.stream_families over FAMILY_CASES["chr17_s17"], plus dense_tiles):
    {family: (conc path, chim path, concordant AlnTable)}."""
    n, s, disc, rl, kw = FAMILY_CASES["chr17_s17"]
    conc, chim, _ = synth.make_case(n, ref_len=synth.CHR17_LEN, seed=s, disc_frac=disc, **kw)
    fams = stream_families(conc, chim, seed)
    fams["dense_tiles"] = dense_tiles_case()[:2]
    out = {}
    for name, tab in fams.items():
        ch = chim
        if isinstance(tab, tuple):
            tab, ch = tab
        d = os.path.join(str(tmpdir), name)
        os.makedirs(d, exist_ok=True)
        cp, hp = os.path.join(d, "conc.sqmb"), os.path.join(d, "chim.sqmb")
        sqmb.write_sqmb(cp, tab); sqmb.write_sqmb(hp, ch)
        out[name] = (cp, hp, tab)
    return out


K_NO_CC_END, K_CC_WALK_TILE = -(1 << 30), 0x7FFFFFFF  # sq_classify.cuh kNoCcEnd, kCcWalkTile
CLS_GATE, CLS_KEEP, CLS_CONC, CLS_PART, CLS_HASBLK, CLS_DISPL, CLS_REST = 1, 2, 4, 8, 16, 32, 64


def _key(chr_, pos):
    """sq_depth_cover.cuh chrpos_key: (chr + 1) << 32 | (uint32) pos."""
    return ((np.asarray(chr_, np.int64) + 1).astype(np.uint64) << np.uint64(32)) | (np.asarray(pos, np.int64) & 0xFFFFFFFF).astype(np.uint64)


def expected_phase1(rc, ref_id, pos, tile=TILE) -> dict:
    """The restatement's per-record classification (pyref.run_restate_classify) reduced to the outputs of the classification
    pass, in its conventions: per record, the gap / partial / displaced lists, and per `tile`-record tile the exclusive maximum
    of the otherrightmost keys, the ConcordantCluster maximum (kCcWalkTile for a tile whose first record is unmapped or whose
    first and last records lie on different chromosomes), the coverage pass's count and maximum start key.  `ref_id`, `pos`:
    the records' own fields."""
    ref_id, pos = np.asarray(ref_id, np.int64), np.asarray(pos, np.int64)
    cls = rc["cls"].astype(np.uint8)
    n = cls.shape[0]
    assert ref_id.shape[0] == n
    keep = (cls & CLS_KEEP) != 0
    conc = (cls & CLS_CONC) != 0
    flen = np.where(conc, rc["first_len"], 0)
    gap = keep & ((ref_id != rc["ex_chr"]) | (pos > rc["ex_right"].astype(np.int64) + rc["read_len"]))
    out = {
        "cls": cls, "first_len": np.minimum(flen, 65535).astype(np.uint16),
        "gap_rec": np.flatnonzero(gap).astype(np.int32), "gap_key": _key(rc["ex_chr"], rc["ex_right"])[gap],
        "pc_rec": np.flatnonzero((cls & CLS_PART) != 0).astype(np.int32),
        "dp_rec": np.flatnonzero(conc & ((cls & CLS_DISPL) != 0)).astype(np.int32),
        "lmax": int(flen.max()) if n else 0, "first_kept": int(np.argmax(keep)) if keep.any() else n,
    }
    nt = (n + tile - 1) // tile
    okey = np.where(rc["other_end"] >= 0, _key(ref_id, rc["other_end"]), np.uint64(0))
    q = rc["cover_q"] != 0
    qkey = _key(ref_id, rc["frag_start"])
    okmax, ccmax, nq, qmax = np.zeros(nt, np.uint64), np.zeros(nt, np.int32), np.zeros(nt, np.uint32), np.zeros(nt, np.uint64)
    run = np.uint64(0)
    qk, qe = [], []
    for t in range(nt):
        s = slice(t * tile, min(n, (t + 1) * tile))
        okmax[t] = run
        if s.stop > s.start:
            run = max(run, okey[s].max())
        if ref_id[s.start] < 0 or ref_id[s.start] != ref_id[s.stop - 1]:
            ccmax[t] = K_CC_WALK_TILE
        else:
            c = rc["cc_end"][s]
            c = c[c != np.iinfo(np.int32).min]
            ccmax[t] = c.max() if c.size else K_NO_CC_END
        nq[t] = q[s].sum()
        qmax[t] = qkey[s][q[s]].max() if nq[t] else 0
        qk.append(qkey[s][q[s]]); qe.append(rc["frag_end"][s][q[s]])
    out.update(okmax_excl=okmax, ccmax=ccmax, cov_nq=nq, cov_qmax=qmax, qstage_key=qk, qstage_end=qe)
    return out
