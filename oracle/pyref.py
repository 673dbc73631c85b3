"""TEST INFRASTRUCTURE.  Python driver of the oracle: builds and runs oracle/_ref/squid_ref (the reference's own
sources against shims) and loads its seam dumps.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module; the product (squid_b200/) never does.
"""
from __future__ import annotations

import json
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_BIN = os.path.join(HERE, "_ref", "squid_ref")
REFERENCE_SRC = "/root/reference"


def build(verbose: bool = False) -> None:
    """(Re)builds oracle/_ref when the reference sources are present (development container only);
    on the GPU box the prebuilt binary that travelled with the snapshot is used as is."""
    if os.path.isdir(os.path.join(REFERENCE_SRC, "src")):
        srcs = [os.path.join(HERE, "ref_harness.cpp"), os.path.join(HERE, "Makefile")] + [os.path.join(HERE, "shim", d, f) for d, _, fs in os.walk(os.path.join(HERE, "shim")) for f in fs]
        if os.path.exists(REF_BIN) and all(os.path.getmtime(s) <= os.path.getmtime(REF_BIN) for s in srcs if os.path.exists(s)):
            return
        r = subprocess.run(["make", "-C", HERE, "ref"], capture_output=True, text=True)
        if verbose:
            print(r.stdout[-2000:], r.stderr[-2000:])
        if r.returncode != 0:
            raise RuntimeError("oracle/_ref build failed:\n" + r.stderr[-4000:])


def available() -> bool:
    return os.path.exists(REF_BIN)


def _i32(path: str, cols: int) -> np.ndarray:
    return np.fromfile(path, dtype=np.int32).reshape(-1, cols) if os.path.exists(path) else np.zeros((0, cols), np.int32)


def load_dumps(outdir: str) -> dict:
    d = {
        "nodes": _i32(os.path.join(outdir, "nodes_i32.bin"), 4),
        "avgdepth": np.fromfile(os.path.join(outdir, "nodes_f64.bin")) if os.path.exists(os.path.join(outdir, "nodes_f64.bin")) else np.zeros(0),
        "edges": _i32(os.path.join(outdir, "edges_i32.bin"), 5),
        "chim_loaded": _i32(os.path.join(outdir, "chim_loaded.bin"), 8),
        "chim_loaded_meta": _i32(os.path.join(outdir, "chim_loaded.bin.meta"), 4),
        "chim_after_edges": _i32(os.path.join(outdir, "chim_after_edges.bin"), 8),
        "final_nodes": _i32(os.path.join(outdir, "final_nodes_i32.bin"), 4),
        "final_edges": _i32(os.path.join(outdir, "final_edges_i32.bin"), 5),
        "exactbp": _i32(os.path.join(outdir, "exactbp_i32.bin"), 6),
        "support": _i32(os.path.join(outdir, "support_i32.bin"), 6),
    }
    p = os.path.join(outdir, "timings.json")
    d["timings"] = json.load(open(p)) if os.path.exists(p) else {}
    rl = os.path.join(outdir, "readlen.bin")
    d["read_len"] = int(np.fromfile(rl, dtype=np.int32)[0]) if os.path.exists(rl) else 0
    return d


def run(conc_sqmb: str, chim_sqmb: str, outdir: str, extra_args=(), timeout: float = 3600.0) -> dict:
    if not available():
        raise RuntimeError("oracle/_ref/squid_ref is missing (run oracle.pyref.build() where /root/reference exists)")
    os.makedirs(outdir, exist_ok=True)
    r = subprocess.run([REF_BIN, conc_sqmb, chim_sqmb, outdir, "--quiet", *extra_args], capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference harness failed rc=%d: %s" % (r.returncode, r.stderr[-2000:]))
    return load_dumps(outdir)


RESTATE_LIB = os.path.join(HERE, "liboracle.so")


def build_restate() -> None:
    """Compiles the CPU restatement (oracle/restate/squid_oracle.cpp -> oracle/liboracle.so)."""
    src = os.path.join(HERE, "restate", "squid_oracle.cpp")
    if os.path.exists(RESTATE_LIB) and os.path.getmtime(RESTATE_LIB) >= os.path.getmtime(src):
        return
    r = subprocess.run(["make", "-C", HERE, "restate"], capture_output=True, text=True)
    if r.returncode != 0 or not os.path.exists(RESTATE_LIB):
        raise RuntimeError("oracle restatement build failed:\n" + r.stdout[-2000:] + r.stderr[-4000:])


def run_restate(conc_sqmb: str, chim_sqmb: str, outdir: str, bps=None, opts=None, stop_after: int = 0) -> dict:
    """Runs the CPU restatement; `bps` = sorted (chr,pos) int array for the coverage pass.  Same dump layout as run().
    stop_after: 0 = everything, 1/2/3 = stop after the chimeric loader / nodes / edges, -1 = the coverage pass alone."""
    import ctypes as C
    build_restate()
    lib = C.CDLL(RESTATE_LIB)
    lib.sqo_run.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.c_char_p, C.c_int]
    os.makedirs(outdir, exist_ok=True)
    bf = None
    if bps is not None:
        bf = os.path.join(outdir, "bps_in.bin")
        np.ascontiguousarray(bps, dtype=np.int32).reshape(-1, 2).tofile(bf)
    o = (C.c_int * 6)(*(opts if opts is not None else restate_opts()))
    rc = lib.sqo_run(conc_sqmb.encode(), chim_sqmb.encode(), outdir.encode(), o, bf.encode() if bf else None, stop_after)
    if rc != 0:
        raise RuntimeError("sqo_run failed rc=%d" % rc)
    d = load_dumps(outdir)
    cp = os.path.join(outdir, "cov_i32.bin")
    d["cov"] = np.fromfile(cp, dtype=np.int32) if os.path.exists(cp) else None
    return d


def run_restate_on_nodes(conc_sqmb: str, chim_sqmb: str, outdir: str, nodes, opts=None, dump_raw: bool = False) -> dict:
    """BuildEdges of the CPU restatement on a given segment table `nodes` (rows chr, pos, len[, ...]): the graph reload of
    SegmentGraph_t(string).  Returns {"edges", "chim_after_edges"}; with dump_raw also "raw_edges", int64 rows (concordant
    record index, packed edge key) for every edge RawEdgesOther emits, in emission order."""
    import ctypes as C
    build_restate()
    lib = C.CDLL(RESTATE_LIB)
    lib.sqo_edges_on_nodes.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.c_char_p, C.c_int]
    os.makedirs(outdir, exist_ok=True)
    nf = os.path.join(outdir, "nodes_in.bin")
    np.ascontiguousarray(np.asarray(nodes)[:, :3], dtype=np.int32).tofile(nf)
    o = (C.c_int * 6)(*(opts if opts is not None else restate_opts()))
    rc = lib.sqo_edges_on_nodes(conc_sqmb.encode(), chim_sqmb.encode(), outdir.encode(), o, nf.encode(), int(dump_raw))
    if rc != 0:
        raise RuntimeError("sqo_edges_on_nodes failed rc=%d" % rc)
    d = {"edges": _i32(os.path.join(outdir, "edges_i32.bin"), 5), "chim_after_edges": _i32(os.path.join(outdir, "chim_after_edges.bin"), 8)}
    if dump_raw:
        d["raw_edges"] = np.fromfile(os.path.join(outdir, "raw_edges.bin"), dtype=np.int64).reshape(-1, 2)
    return d


CLASSIFY_COLS = ("cls", "first_len", "cc_end", "other_end", "ex_chr", "ex_right", "cover_q", "frag_start", "frag_end")


def run_restate_classify(conc_sqmb: str, chim_sqmb: str, outdir: str, opts=None) -> dict:
    """The per-record preamble of BuildNode_STAR over the whole concordant stream (sqo_classify): one int32 array per column of
    CLASSIFY_COLS (class bits as sq_common.cuh's CLS_* values; cc_end INT32_MIN and other_end -1 where the record has none;
    (ex_chr, ex_right) = otherChr/otherRight in front of the record), plus "read_len"."""
    import ctypes as C
    build_restate()
    lib = C.CDLL(RESTATE_LIB)
    lib.sqo_classify.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int)]
    os.makedirs(outdir, exist_ok=True)
    o = (C.c_int * 6)(*(opts if opts is not None else restate_opts()))
    rc = lib.sqo_classify(conc_sqmb.encode(), chim_sqmb.encode(), outdir.encode(), o)
    if rc != 0:
        raise RuntimeError("sqo_classify failed rc=%d" % rc)
    a = _i32(os.path.join(outdir, "classify_i32.bin"), len(CLASSIFY_COLS))
    d = {k: np.ascontiguousarray(a[:, i]) for i, k in enumerate(CLASSIFY_COLS)}
    d["read_len"] = int(np.fromfile(os.path.join(outdir, "readlen.bin"), dtype=np.int32)[0])
    return d


_RESTATE_FLAGS = {"-pt": 0, "-pl": 1, "-pm": 2, "-mq": 3, "-dp": 4, "-di": 5}  # the reference's options (Config.cpp:18-25) -> sqo_run opts


def restate_opts(extra_args=()) -> list:
    o = [1, 10, 4, -1, 50000, 20]
    args = list(extra_args)
    if len(args) % 2 or any(f not in _RESTATE_FLAGS for f in args[::2]):
        raise ValueError("the restatement takes only %s, each with a value: %s" % (sorted(_RESTATE_FLAGS), args))
    for f, v in zip(args[::2], args[1::2]):
        o[_RESTATE_FLAGS[f]] = int(v)
    return o


def components(n: int, a, b) -> np.ndarray:
    """Connected-component label per node, components numbered in the order of their smallest node (SegmentGraph.cpp:2986-3003)."""
    parent = list(range(n))

    def root(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x
    for x, y in zip(np.asarray(a).tolist(), np.asarray(b).tolist()):
        rx, ry = root(x), root(y)
        if rx != ry:
            parent[max(rx, ry)] = min(rx, ry)
    label, out = {}, np.empty(n, np.int32)
    for x in range(n):
        out[x] = label.setdefault(root(x), len(label))
    return out


def run_restated(conc_sqmb: str, chim_sqmb: str, outdir: str, extra_args=(), timeout: float = None) -> dict:
    """run() where the reference build is absent: the same dumps from the CPU restatement, which the committed golden dumps
    pin to the reference.  The host stages between BuildEdges and ExactBPConcordantSupport (filters, CompressNode,
    ExactBreakpoint) are not restated, so the final graph is every segment and every edge, without exact breakpoints: each
    edge is covered at its two segment ends.  Writes labels_i32.bin of that graph like the reference harness."""
    opts = restate_opts(extra_args)
    d = run_restate(conc_sqmb, chim_sqmb, outdir, opts=opts, stop_after=3)
    d["final_nodes"], d["final_edges"], d["exactbp"] = d["nodes"], d["edges"], np.zeros((0, 6), np.int32)
    bps = breakpoints_of(d)
    cov = run_restate(conc_sqmb, chim_sqmb, outdir, bps=bps, opts=opts)["cov"]
    sup = support_from_cov(d, bps, cov)
    d["support"] = np.array([k + c for k, v in sup.items() for c in v], np.int32).reshape(-1, 6)
    components(d["nodes"].shape[0], d["edges"][:, 0], d["edges"][:, 1]).tofile(os.path.join(outdir, "labels_i32.bin"))
    return d


class Restated:
    """The oracle interface of this module (run, load_dumps) backed by the CPU restatement."""
    run = staticmethod(run_restated)
    load_dumps = staticmethod(load_dumps)


def breakpoints_of(d: dict) -> np.ndarray:
    """The sorted BPs vector ExactBPConcordantSupport assembles (SegmentGraph.cpp:3091-3109) from a dump of the
    reference harness (final graph + ExactBP map)."""
    fn = d["final_nodes"].astype(np.int64)
    xm = exactbp_map(d)
    bps = []
    for e in d["final_edges"]:
        k = tuple(int(v) for v in e[:4])
        if k in xm:
            for b1, b2 in xm[k]:
                bps.append((int(fn[k[0], 0]), b1)); bps.append((int(fn[k[1], 0]), b2))
        else:
            bps.append((int(fn[k[0], 0]), int(fn[k[0], 1] + (0 if k[2] else fn[k[0], 2]))))
            bps.append((int(fn[k[1], 0]), int(fn[k[1], 1] + (0 if k[3] else fn[k[1], 2]))))
    bps.sort()
    return np.array(bps, dtype=np.int32).reshape(-1, 2)


def support_from_cov(d: dict, bps: np.ndarray, cov: np.ndarray) -> dict:
    """Maps a Coverages vector back to {edge: [(cov1,cov2)]} as SegmentGraph.cpp:3171-3211 does (lower_bound lookups)."""
    fn = d["final_nodes"].astype(np.int64)
    xm = exactbp_map(d)
    key = bps[:, 0].astype(np.int64) * (1 << 32) + bps[:, 1].astype(np.int64)
    look = lambda c, p: int(cov[np.searchsorted(key, int(c) * (1 << 32) + int(p))])
    out = {}
    for e in d["final_edges"]:
        k = tuple(int(v) for v in e[:4])
        if k in xm:
            out[k] = [(look(fn[k[0], 0], b1), look(fn[k[1], 0], b2)) for b1, b2 in xm[k]]
        else:
            out[k] = [(look(fn[k[0], 0], fn[k[0], 1] + (0 if k[2] else fn[k[0], 2])), look(fn[k[1], 0], fn[k[1], 1] + (0 if k[3] else fn[k[1], 2])))]
    return out


def exactbp_map(d: dict) -> dict:
    m = {}
    for row in d["exactbp"]:
        m.setdefault(tuple(int(v) for v in row[:4]), []).append((int(row[4]), int(row[5])))
    return m


def support_map(d: dict) -> dict:
    m = {}
    for row in d["support"]:
        m.setdefault(tuple(int(v) for v in row[:4]), []).append((int(row[4]), int(row[5])))
    return m
