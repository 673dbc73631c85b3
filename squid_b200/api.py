"""ctypes binding of the squid_b200 C ABI (include/squid_b200.h, include/squid_b200_host.h) and a host-side
mirror of the reference's SegmentGraph_t seam for the hot path (same method names and argument meaning:
BuildNode_STAR, BuildEdges, ExactBPConcordantSupport; reference: src/SegmentGraph.h:77-79,104).

The product path is the CUDA library: importing this module never falls back to a CPU implementation,
and `lib()` raises if squid_b200/libsquid_b200.so is missing or a symbol is not exported.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsquid_b200.so")

SQG_OK, SQG_EINVAL, SQG_ENODEVICE, SQG_ECUDA, SQG_ESTATE, SQG_EUNSUPPORTED, SQG_ENOMEM = 0, -1, -2, -3, -4, -5, -6


class SquidB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("squid_b200 error %d: %s" % (code, msg))
        self.code = code


class sqg_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("using_star", "max_lowphred_len", "min_mapq", "concord_dist_pos", "concord_dist_idx", "read_len")]


_P = C.c_void_p


class sqg_batch(C.Structure):
    _fields_ = [("n_rec", C.c_int64), ("n_blk", C.c_int64)] + [(n, _P) for n in (
        "ref_id", "pos", "mate_ref_id", "mate_pos", "end_pos", "flag", "total_len", "lowphred_run", "mapq", "aux", "blk_off",
        "blk_ref_pos", "blk_match_ref", "blk_read_pos", "blk_match_read")]


class sqg_chimeric(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_blk", C.c_int64)] + [(n, _P) for n in (
        "read_off", "n_first", "first_total_len", "second_total_len", "first_lowphred", "second_lowphred", "multi_filter",
        "blk_ref_id", "blk_ref_pos", "blk_read_pos", "blk_match_ref", "blk_match_read", "blk_is_reverse")]


class sqg_wire(C.Structure):  # include/squid_b200.h
    _fields_ = [(k, C.c_int64) for k in ("n_rec", "n_blk", "n_tiles", "n_rec_exc", "n_blk_exc", "n_wblk")] + [(k, C.c_void_p) for k in (
        "tile_ref_id", "tile_pos", "tile_blk_off", "tile_rec_exc_off", "tile_blk_exc_off", "tile_wblk_off", "dpos", "span", "dmate", "flag", "total_len", "lowphred_run", "mapq", "aux_nblk",
        "blk_dref", "blk_match_ref", "blk_read_pos", "blk_match_read", "rec_exc", "blk_exc")]


WIRE_REC_EXC = np.dtype([("idx", "<u4"), ("ref_id", "<i4"), ("pos", "<i4"), ("mate_ref_id", "<i4"), ("mate_pos", "<i4"), ("end_pos", "<i4"), ("lowphred_run", "<u2"), ("n_blk", "<u2")])
WIRE_BLK_EXC = np.dtype([("idx", "<u4"), ("ref_pos", "<i4"), ("match_ref", "<i4")])


class sqg_bam_decode(C.Structure):  # include/squid_b200.h
    _fields_ = [("phred33", C.c_int32), ("min_phred", C.c_int32), ("n_names", C.c_int64), ("names", C.c_void_p), ("name_off", C.c_void_p)]


class sqh_options(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("phred33", "max_lowphred_len", "min_phred", "min_mapq", "concord_dist_pos", "concord_dist_idx")]


BATCH_DTYPES = {
    "ref_id": np.int32, "pos": np.int32, "mate_ref_id": np.int32, "mate_pos": np.int32, "end_pos": np.int32,
    "flag": np.uint16, "total_len": np.uint16, "lowphred_run": np.uint16, "mapq": np.uint8, "aux": np.uint8, "blk_off": np.uint32,
    "blk_ref_pos": np.int32, "blk_match_ref": np.int32, "blk_read_pos": np.uint16, "blk_match_read": np.uint16,
}
CHIM_DTYPES = {
    "read_off": np.uint32, "n_first": np.uint16, "first_total_len": np.int32, "second_total_len": np.int32,
    "first_lowphred": np.uint8, "second_lowphred": np.uint8, "multi_filter": np.uint8,
    "blk_ref_id": np.int32, "blk_ref_pos": np.int32, "blk_read_pos": np.int32, "blk_match_ref": np.int32, "blk_match_read": np.int32,
    "blk_is_reverse": np.uint8,
}

EXPORTS = [
    "sqg_create", "sqg_destroy", "sqg_last_error", "sqg_load_concordant", "sqg_load_concordant_wire", "sqg_load_concordant_bam", "sqg_download_concordant", "sqg_connected_components", "sqg_attach_concordant_device", "sqg_load_chimeric",
    "sqg_build_nodes", "sqg_set_nodes", "sqg_build_edges", "sqg_bp_coverage", "sqg_edges_device_table", "sqg_merge_edge_tables",
    "sqg_phase_ms", "sqg_launch_count", "sqg_stat", "sqg_classify_dump", "sqg_selftest_gpu_sort",
    "sqg_plan_shards", "sqg_set_shard", "sqg_shard_seeds", "sqg_shard_build", "sqg_shard_hint_state", "sqg_shard_redo_edges",
    "sqg_shard_cov_begin", "sqg_shard_cov_chain", "sqg_shard_cov_owned_t", "sqg_shard_cov_count",
    "sqh_default_options", "sqh_open_case", "sqh_open_concordant", "sqh_open_bam_case", "sqh_open_bam_chimeric", "sqh_case_chim_names", "sqh_probe_bam", "sqh_close_case", "sqh_case_batch", "sqh_case_chimeric", "sqh_case_config",
    "sqh_case_n_ref", "sqh_case_ref_len", "sqh_case_blocks",
    "sqh_exact_breakpoint", "sqh_free", "sqh_write_graph", "sqh_write_bedpe", "sqh_pack_wire", "sqh_free_wire", "sqh_wire_bytes",
]

_lib = None


def lib() -> C.CDLL:
    """Loads the CUDA library; never substitutes anything else for it."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SquidB200Error(SQG_ENODEVICE, "%s is missing: run `python -m squid_b200.build` (there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    for s in EXPORTS:
        if not hasattr(L, s):
            raise SquidB200Error(SQG_EINVAL, "library does not export %s" % s)
    pp = C.POINTER
    L.sqg_create.argtypes = [pp(_P), pp(sqg_config), _P, C.c_int32, C.c_int32]
    L.sqg_destroy.argtypes = [_P]; L.sqg_destroy.restype = None
    L.sqg_last_error.argtypes = [_P]; L.sqg_last_error.restype = C.c_char_p
    L.sqg_load_concordant.argtypes = [_P, pp(sqg_batch), C.c_int64]
    L.sqg_attach_concordant_device.argtypes = [_P, pp(sqg_batch), C.c_int64]
    L.sqg_load_concordant_wire.argtypes = [_P, pp(sqg_wire), C.c_int64]
    L.sqg_load_concordant_bam.argtypes = [_P, C.c_char_p, pp(sqg_bam_decode), C.c_int64]
    L.sqg_download_concordant.argtypes = [_P, pp(sqg_batch)]
    L.sqg_connected_components.argtypes = [C.c_int32, C.c_int64, _P, _P, C.c_int64, _P, pp(C.c_int32)]
    L.sqh_pack_wire.argtypes = [pp(sqg_batch), C.c_int32, pp(pp(sqg_wire))]
    L.sqh_free_wire.argtypes = [pp(sqg_wire)]; L.sqh_free_wire.restype = None
    L.sqh_wire_bytes.argtypes = [pp(sqg_wire)]; L.sqh_wire_bytes.restype = C.c_int64
    L.sqg_load_chimeric.argtypes = [_P, pp(sqg_chimeric)]
    L.sqg_build_nodes.argtypes = [_P, pp(_P), pp(_P), pp(_P), pp(C.c_int64), pp(_P), pp(_P), pp(C.c_int32)]
    L.sqg_set_nodes.argtypes = [_P, _P, _P, _P, C.c_int64]
    L.sqg_build_edges.argtypes = [_P, pp(_P), pp(_P), pp(_P), pp(_P), pp(C.c_int64), pp(sqg_chimeric)]
    L.sqg_bp_coverage.argtypes = [_P, _P, _P, C.c_int64, _P]
    L.sqg_edges_device_table.argtypes = [_P, pp(_P), pp(_P), pp(C.c_int64)]
    L.sqg_merge_edge_tables.argtypes = [_P, _P, _P, C.c_int64, pp(_P), pp(_P), pp(_P), pp(_P), pp(C.c_int64)]
    L.sqg_phase_ms.argtypes = [_P, C.c_char_p]; L.sqg_phase_ms.restype = C.c_float
    L.sqg_launch_count.argtypes = [_P]; L.sqg_launch_count.restype = C.c_int64
    L.sqg_stat.argtypes = [_P, C.c_char_p]; L.sqg_stat.restype = C.c_int64
    L.sqg_classify_dump.argtypes = [_P, C.c_char_p, _P, C.c_int64, pp(C.c_int64)]
    L.sqg_plan_shards.argtypes = [pp(sqg_batch), pp(sqg_chimeric), pp(sqg_config), C.c_int32, C.c_int32, _P, pp(C.c_int32)]
    L.sqg_set_shard.argtypes = [_P, C.c_int32, C.c_int32]
    L.sqg_shard_seeds.argtypes = [_P, C.c_int32, pp(_P), pp(C.c_int64)]
    L.sqg_shard_build.argtypes = [_P, _P, C.c_int64, pp(_P), pp(_P), pp(_P), pp(C.c_int64), pp(_P), pp(_P), pp(C.c_int32)]
    L.sqg_shard_hint_state.argtypes = [_P, pp(C.c_int32), pp(C.c_int32)]
    L.sqg_shard_redo_edges.argtypes = [_P, C.c_int32]
    L.sqg_shard_cov_begin.argtypes = [_P, _P, _P, C.c_int64, pp(C.c_int64), pp(C.c_int64)]
    L.sqg_shard_cov_chain.argtypes = [_P, C.c_int64, pp(C.c_int64)]
    L.sqg_shard_cov_owned_t.argtypes = [_P, C.c_int64, C.c_int64, C.c_int64, _P]
    L.sqg_shard_cov_count.argtypes = [_P, C.c_int64, _P, _P]
    L.sqh_default_options.argtypes = [pp(sqh_options)]; L.sqh_default_options.restype = None
    L.sqh_open_case.argtypes = [C.c_char_p, C.c_char_p, pp(sqh_options), pp(_P), C.c_char_p, C.c_int]
    L.sqh_open_bam_case.argtypes = [C.c_char_p, C.c_char_p, pp(sqh_options), pp(_P), C.c_char_p, C.c_int]
    L.sqh_open_bam_chimeric.argtypes = [C.c_char_p, C.c_char_p, pp(sqh_options), pp(_P), C.c_char_p, C.c_int]
    L.sqh_case_chim_names.argtypes = [_P, pp(_P), pp(_P), pp(C.c_int64)]
    L.sqh_close_case.argtypes = [_P]; L.sqh_close_case.restype = None
    L.sqh_case_batch.argtypes = [_P]; L.sqh_case_batch.restype = pp(sqg_batch)
    L.sqh_case_chimeric.argtypes = [_P]; L.sqh_case_chimeric.restype = pp(sqg_chimeric)
    L.sqh_case_config.argtypes = [_P]; L.sqh_case_config.restype = pp(sqg_config)
    L.sqh_case_n_ref.argtypes = [_P]; L.sqh_case_n_ref.restype = C.c_int32
    L.sqh_case_ref_len.argtypes = [_P]; L.sqh_case_ref_len.restype = pp(C.c_int32)
    L.sqh_case_blocks.argtypes = [_P, C.c_int64, _P, C.c_int32, pp(C.c_int32), pp(C.c_int32)]
    L.sqh_case_blocks.restype = C.c_int32
    L.sqh_exact_breakpoint.argtypes = [_P, _P, _P, C.c_int64, pp(sqg_chimeric), C.c_int32, C.c_int32, pp(_P), pp(C.c_int64)]
    L.sqh_free.argtypes = [_P]; L.sqh_free.restype = None
    L.sqh_write_graph.argtypes = [C.c_char_p, _P, _P, _P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, _P, C.c_int64]
    L.sqh_write_bedpe.argtypes = [C.c_char_p, pp(C.c_char_p), C.c_int32, _P, _P, _P, C.c_int64, _P, _P, _P, _P, _P, C.c_int64, _P, _P, C.c_int64,
                                  _P, C.c_int64, _P, C.c_int64, C.c_double, C.c_int32, C.c_int32]
    _lib = L
    return L


def _np_from(ptr, n, dtype, owner=None) -> np.ndarray:
    """Array over library memory.  owner=None: a copy.  Else a VIEW (no copy) that keeps `owner` -- the object whose close()
    releases the memory -- alive for as long as the array (or anything sliced from it) lives."""
    n = int(n)
    if n == 0:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr if isinstance(ptr, int) else ptr.value)
    if owner is None:
        return np.frombuffer(buf, dtype=dtype, count=n).copy()
    buf._owner = owner
    return np.frombuffer(buf, dtype=dtype, count=n)


@dataclass
class Config:
    """The reference's Config globals that gate the path (src/Config.cpp:14-37)."""
    UsingSTAR: bool = True
    Phred_Type: int = 1
    Max_LowPhred_Len: int = 10
    Min_Phred: int = 4
    Min_MapQual: int = 255  # STAR default (Config.cpp:221-222)
    Concord_Dist_Pos: int = 50000
    Concord_Dist_Idx: int = 20
    ReadLen: int = 0

    def as_struct(self) -> sqg_config:
        return sqg_config(int(self.UsingSTAR), self.Max_LowPhred_Len, self.Min_MapQual, self.Concord_Dist_Pos, self.Concord_Dist_Idx, self.ReadLen)


class RecordBatch:
    """SoA record batch (host numpy arrays), see sqg_batch."""

    def __init__(self, arrays: dict):
        self.a = {k: np.ascontiguousarray(arrays[k], dtype=dt) for k, dt in BATCH_DTYPES.items()}
        self.n_rec = int(self.a["ref_id"].shape[0])
        self.n_blk = int(self.a["blk_ref_pos"].shape[0])
        assert self.a["blk_off"].shape[0] == self.n_rec + 1

    def as_struct(self) -> sqg_batch:
        s = sqg_batch()
        s.n_rec, s.n_blk = self.n_rec, self.n_blk
        for k in BATCH_DTYPES:
            setattr(s, k, self.a[k].ctypes.data)
        return s

    @staticmethod
    def from_struct(s: sqg_batch, owner=None) -> "RecordBatch":
        """owner: the object that owns the arrays of `s` (they are then viewed, not copied: a 100 M-pair batch is 9 GB)."""
        d = {}
        for k, dt in BATCH_DTYPES.items():
            n = s.n_blk if k.startswith("blk_") and k != "blk_off" else (s.n_rec + 1 if k == "blk_off" else s.n_rec)
            d[k] = _np_from(getattr(s, k), n, dt, owner)
        return RecordBatch(d)

    def slice(self, lo: int, hi: int) -> "RecordBatch":
        """Records [lo,hi) as an independent batch (range shard)."""
        b0, b1 = int(self.a["blk_off"][lo]), int(self.a["blk_off"][hi])
        d = {}
        for k in BATCH_DTYPES:
            if k == "blk_off":
                d[k] = (self.a[k][lo:hi + 1] - np.uint32(b0)).astype(np.uint32)
            elif k.startswith("blk_"):
                d[k] = self.a[k][b0:b1]
            else:
                d[k] = self.a[k][lo:hi]
        return RecordBatch(d)


class WireBatch:
    """Wire form of a RecordBatch (include/squid_b200.h: sqg_wire), packed by the host library (sqh_pack_wire)."""

    def __init__(self, batch: "RecordBatch", pinned: bool = False):
        L = lib()
        self._keep = batch
        bs = batch.as_struct()
        h = C.POINTER(sqg_wire)()
        rc = L.sqh_pack_wire(C.byref(bs), 1 if pinned else 0, C.byref(h))
        if rc != 0:
            raise SquidB200Error(rc, "sqh_pack_wire failed")
        self._h = h
        self.nbytes = int(L.sqh_wire_bytes(h))

    @property
    def struct(self) -> sqg_wire:
        return self._h.contents

    def arrays(self) -> dict:
        """numpy views of every wire array (tests decode them independently)."""
        w = self.struct
        nt = w.n_tiles
        spec = {"tile_ref_id": (nt, np.int32), "tile_pos": (nt, np.int32), "tile_blk_off": (nt + 1, np.uint32), "tile_rec_exc_off": (nt + 1, np.uint32),
                "tile_blk_exc_off": (nt + 1, np.uint32), "tile_wblk_off": (nt + 1, np.uint32), "dpos": (w.n_rec, np.uint16), "span": (w.n_rec, np.uint16), "dmate": (w.n_rec, np.int16),
                "flag": (w.n_rec, np.uint16), "total_len": (w.n_rec, np.uint16), "lowphred_run": (w.n_rec, np.uint8), "mapq": (w.n_rec, np.uint8),
                "aux_nblk": (w.n_rec, np.uint8), "blk_dref": (w.n_wblk, np.uint16), "blk_match_ref": (w.n_wblk, np.uint16), "blk_read_pos": (w.n_wblk, np.uint16),
                "blk_match_read": (w.n_wblk, np.uint16), "rec_exc": (w.n_rec_exc, WIRE_REC_EXC), "blk_exc": (w.n_blk_exc, WIRE_BLK_EXC)}
        return {k: _np_from(getattr(w, k) or 0, n, dt) for k, (n, dt) in spec.items()}

    def close(self):
        if self._h:
            lib().sqh_free_wire(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ChimericReads:
    """Chimrecord after the host loader, see sqg_chimeric.  Block arrays are trimmed in place by build_edges."""

    def __init__(self, arrays: dict):
        self.a = {k: np.ascontiguousarray(arrays[k], dtype=dt).copy() for k, dt in CHIM_DTYPES.items()}
        self.n_reads = int(self.a["n_first"].shape[0])
        self.n_blk = int(self.a["blk_ref_id"].shape[0])

    def as_struct(self) -> sqg_chimeric:
        s = sqg_chimeric()
        s.n_reads, s.n_blk = self.n_reads, self.n_blk
        for k in CHIM_DTYPES:
            setattr(s, k, self.a[k].ctypes.data)
        return s

    @staticmethod
    def from_struct(s: sqg_chimeric) -> "ChimericReads":
        d = {}
        for k, dt in CHIM_DTYPES.items():
            n = s.n_blk if k.startswith("blk_") else (s.n_reads + 1 if k == "read_off" else s.n_reads)
            d[k] = _np_from(getattr(s, k), n, dt)
        return ChimericReads(d)

    def block_table(self) -> np.ndarray:
        """(read, is_second, RefID, RefPos, ReadPos, MatchRef, MatchRead, IsReverse) rows, the oracle's dump layout."""
        a = self.a
        nb = np.diff(a["read_off"].astype(np.int64))
        read = np.repeat(np.arange(self.n_reads, dtype=np.int64), nb)
        k = np.arange(self.n_blk, dtype=np.int64) - np.repeat(a["read_off"][:-1].astype(np.int64), nb)
        second = (k >= np.repeat(a["n_first"].astype(np.int64), nb)).astype(np.int32)
        return np.stack([read.astype(np.int32), second, a["blk_ref_id"], a["blk_ref_pos"], a["blk_read_pos"], a["blk_match_ref"],
                         a["blk_match_read"], a["blk_is_reverse"].astype(np.int32)], axis=1).astype(np.int32)


class HostCase:
    """Host twin front end: SQMB files -> Chimrecord + packed concordant batch (sqh_open_case)."""

    def __init__(self, concordant_sqmb: str, chimeric_sqmb: str, bam: bool = False, header_only: bool = False, **opts):
        """bam=True: the two paths are coordinate-sorted BAM files (sqh_open_bam_case), else SQMB tables.  header_only=True (BAM
        only): the concordant file's header alone is read and the batch stays empty (sqh_open_bam_chimeric), for
        SegmentGraph.load_concordant_bam, which decodes that file on the device."""
        if header_only and not bam:
            raise ValueError("header_only needs bam=True")
        L = lib()
        o = sqh_options()
        L.sqh_default_options(C.byref(o))
        for k, v in opts.items():
            setattr(o, k, v)
        h = _P()
        err = C.create_string_buffer(512)
        opener = L.sqh_open_bam_chimeric if header_only else L.sqh_open_bam_case if bam else L.sqh_open_case
        rc = opener(concordant_sqmb.encode(), chimeric_sqmb.encode(), C.byref(o), C.byref(h), err, 512)
        if rc != 0:
            raise SquidB200Error(rc, err.value.decode())
        self._h = h
        self.batch = RecordBatch.from_struct(L.sqh_case_batch(h).contents, owner=self)  # views into the case (valid until close())
        self.chimeric = ChimericReads.from_struct(L.sqh_case_chimeric(h).contents)
        g = L.sqh_case_config(h).contents
        self.config = Config(True, o.phred33, g.max_lowphred_len, o.min_phred, g.min_mapq, g.concord_dist_pos, g.concord_dist_idx, g.read_len)
        n_ref = L.sqh_case_n_ref(h)
        self.ref_len = _np_from(C.cast(L.sqh_case_ref_len(h), _P), n_ref, np.int32)
        self.options = o

    def chim_names(self):
        """The ChimName list the concordant packer probes, as (blob bytes, int64 offsets[n + 1])."""
        blob, off, n = _P(), _P(), C.c_int64()
        rc = lib().sqh_case_chim_names(self._h, C.byref(blob), C.byref(off), C.byref(n))
        if rc != 0:
            raise SquidB200Error(rc, "sqh_case_chim_names failed")
        offs = _np_from(off, n.value + 1, np.int64)
        return (C.string_at(blob.value, int(offs[-1])) if offs[-1] else b""), offs

    def blocks(self, r: int):
        L = lib()
        out = np.zeros(64, np.int32)
        tl, lr = C.c_int32(), C.c_int32()
        n = L.sqh_case_blocks(self._h, r, out.ctypes.data, 16, C.byref(tl), C.byref(lr))
        return out[: 4 * n].reshape(-1, 4).copy(), tl.value, lr.value

    def close(self):
        if self._h:
            lib().sqh_close_case(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class Nodes:
    Chr: np.ndarray
    Position: np.ndarray
    Length: np.ndarray
    Support: np.ndarray
    AvgDepth: np.ndarray
    count3: np.ndarray = field(repr=False, default=None)
    sumlen3: np.ndarray = field(repr=False, default=None)


@dataclass
class Edges:
    Ind1: np.ndarray
    Ind2: np.ndarray
    Head1: np.ndarray
    Head2: np.ndarray
    Weight: np.ndarray

    def table(self) -> np.ndarray:
        return np.stack([self.Ind1, self.Ind2, self.Head1.astype(np.int32), self.Head2.astype(np.int32), self.Weight], axis=1).astype(np.int32)


class SegmentGraph:
    """Mirror of SegmentGraph_t for the segment-graph construction path, backed by the CUDA library.

        g = SegmentGraph(config, RefLength, device=0)
        g.BuildNode_STAR(Chimrecord, batch)      # SegmentGraph.cpp:192   -> g.vNodes
        g.BuildEdges()                           # SegmentGraph.cpp:1932  -> g.vEdges (Chimrecord trimmed in place)
        cov = g.BPCoverage(bp_chr, bp_pos)       # the BAM pass of ExactBPConcordantSupport, SegmentGraph.cpp:3124-3166
    """

    def __init__(self, config: Config, RefLength, device: int = 0):
        self.L = lib()
        self.config = config
        self.RefLength = np.ascontiguousarray(RefLength, dtype=np.int32)
        self._h = _P()
        cs = config.as_struct()
        rc = self.L.sqg_create(C.byref(self._h), C.byref(cs), self.RefLength.ctypes.data, int(self.RefLength.shape[0]), device)
        if rc != 0:
            msg = self.L.sqg_last_error(self._h).decode() if self._h else "sqg_create failed (no CUDA device?)"
            if self._h:
                self.L.sqg_destroy(self._h)
                self._h = None
            raise SquidB200Error(rc, msg)
        self.vNodes: Nodes | None = None
        self.vEdges: Edges | None = None
        self.Chimrecord: ChimericReads | None = None
        self._batch = None

    def _ck(self, rc: int):
        if rc != 0:
            raise SquidB200Error(rc, self.L.sqg_last_error(self._h).decode())

    def close(self):
        if self._h:
            self.L.sqg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- loading -----------------------------------------------------------------------------
    def load_concordant(self, batch: RecordBatch, first_record_index: int = 0):
        self._batch = batch  # keep the host arrays alive for the duration of the copy
        s = batch.as_struct()
        self._ck(self.L.sqg_load_concordant(self._h, C.byref(s), first_record_index))

    def load_concordant_wire(self, wire: "WireBatch", first_record_index: int = 0):
        self._wire = wire
        self._ck(self.L.sqg_load_concordant_wire(self._h, wire._h, int(first_record_index)))

    def load_concordant_bam(self, path: str, case: "HostCase", first_record_index: int = 0):
        """sqg_load_concordant_bam: the concordant BAM file inflated and decoded on the device into the resident batch -- the
        batch sqh_open_bam_case would pack from it.  `case` (HostCase(conc, chim, bam=True, header_only=True)) gives the decode
        options and ChimName."""
        blob, off = case.chim_names()
        self._names = (C.create_string_buffer(blob, max(1, len(blob))), np.ascontiguousarray(off, np.int64))
        opt = sqg_bam_decode(int(case.options.phred33), int(case.options.min_phred), int(off.shape[0] - 1), C.cast(self._names[0], C.c_void_p).value,
                             self._names[1].ctypes.data)
        self._batch = None
        self._ck(self.L.sqg_load_concordant_bam(self._h, path.encode(), C.byref(opt), int(first_record_index)))

    def download_concordant(self) -> "RecordBatch":
        """The resident batch copied back (check of the wire upload)."""
        n, nb = int(self.stat("n_rec")), int(self.stat("n_blk"))
        a = {"ref_id": np.empty(n, np.int32), "pos": np.empty(n, np.int32), "mate_ref_id": np.empty(n, np.int32), "mate_pos": np.empty(n, np.int32),
             "end_pos": np.empty(n, np.int32), "flag": np.empty(n, np.uint16), "total_len": np.empty(n, np.uint16), "lowphred_run": np.empty(n, np.uint16),
             "mapq": np.empty(n, np.uint8), "aux": np.empty(n, np.uint8), "blk_off": np.empty(n + 1, np.uint32), "blk_ref_pos": np.empty(nb, np.int32),
             "blk_match_ref": np.empty(nb, np.int32), "blk_read_pos": np.empty(nb, np.uint16), "blk_match_read": np.empty(nb, np.uint16)}
        out = RecordBatch(a)
        s = out.as_struct()
        self._ck(self.L.sqg_download_concordant(self._h, C.byref(s)))
        return out

    def attach_concordant_device(self, dev_struct: sqg_batch, keepalive=None, first_record_index: int = 0):
        self._batch = keepalive
        self._ck(self.L.sqg_attach_concordant_device(self._h, C.byref(dev_struct), first_record_index))

    def load_chimeric(self, chim: ChimericReads):
        self.Chimrecord = chim
        s = chim.as_struct()
        self._ck(self.L.sqg_load_chimeric(self._h, C.byref(s)))

    # -- the seam ----------------------------------------------------------------------------
    def BuildNode_STAR(self, Chimrecord: ChimericReads | None = None, batch: RecordBatch | None = None) -> Nodes:
        if batch is not None:
            self.load_concordant(batch)
        if Chimrecord is not None:
            self.load_chimeric(Chimrecord)
        chr_, pos, ln, c3, s3 = _P(), _P(), _P(), _P(), _P()
        n, other = C.c_int64(), C.c_int32()
        self._ck(self.L.sqg_build_nodes(self._h, C.byref(chr_), C.byref(pos), C.byref(ln), C.byref(n), C.byref(c3), C.byref(s3), C.byref(other)))
        N = n.value
        count3 = _np_from(c3, 3 * N, np.int32).reshape(3, N)
        sum3 = _np_from(s3, 3 * N, np.int32).reshape(3, N)
        length = _np_from(ln, N, np.int32)
        # Support / AvgDepth exactly as SegmentGraph.cpp:773-779, 785-801, 807-824: int sums, added as double, divided
        # only inside the `ReadsOther.size()!=0` branch
        support = count3[0] + count3[1] + (count3[2] if other.value else 0)
        depth = sum3[0].astype(np.float64) + sum3[1].astype(np.float64)
        if other.value:
            depth = depth + sum3[2].astype(np.float64)
            depth = 1.0 * depth / length
        self.vNodes = Nodes(_np_from(chr_, N, np.int32), _np_from(pos, N, np.int32), length, support.astype(np.int32), depth, count3, sum3)
        return self.vNodes

    # -- range shards of one stream (include/squid_b200.h "Exact range sharding"; driver: squid_b200/sharded.py) ---------
    def set_shard(self, index: int, count: int):
        self._ck(self.L.sqg_set_shard(self._h, index, count))

    def shard_seeds(self, prior_emission: bool) -> np.ndarray:
        """Stage 1: this shard's seed ops, rows (kind, chr, pos, len)."""
        ops, n = _P(), C.c_int64()
        self._ck(self.L.sqg_shard_seeds(self._h, int(prior_emission), C.byref(ops), C.byref(n)))
        return _np_from(ops, 4 * n.value, np.int32).reshape(-1, 4)

    def shard_build(self, ops_all: np.ndarray):
        """Stage 2: ops of all shards -> (Chr, Position, Length, count3[3,N], sumlen3[3,N], reads_other_nonempty) with this
        shard's partial depth numerators."""
        ops = np.ascontiguousarray(ops_all, np.int32).reshape(-1, 4)
        chr_, pos, ln, c3, s3 = _P(), _P(), _P(), _P(), _P()
        n, other = C.c_int64(), C.c_int32()
        self._ck(self.L.sqg_shard_build(self._h, ops.ctypes.data, int(ops.shape[0]), C.byref(chr_), C.byref(pos), C.byref(ln), C.byref(n),
                                        C.byref(c3), C.byref(s3), C.byref(other)))
        N = n.value
        return (_np_from(chr_, N, np.int32), _np_from(pos, N, np.int32), _np_from(ln, N, np.int32),
                _np_from(c3, 3 * N, np.int32).reshape(3, N), _np_from(s3, 3 * N, np.int32).reshape(3, N), int(other.value))

    def shard_hint_state(self):
        lead, out = C.c_int32(), C.c_int32()
        self._ck(self.L.sqg_shard_hint_state(self._h, C.byref(lead), C.byref(out)))
        return bool(lead.value), int(out.value)

    def shard_redo_edges(self, init_hint: int):
        self._ck(self.L.sqg_shard_redo_edges(self._h, int(init_hint)))

    def shard_cov_begin(self, bp_chr, bp_pos):
        self._bp = (np.ascontiguousarray(bp_chr, np.int32), np.ascontiguousarray(bp_pos, np.int32))
        nq, npass = C.c_int64(), C.c_int64()
        self._ck(self.L.sqg_shard_cov_begin(self._h, self._bp[0].ctypes.data, self._bp[1].ctypes.data, int(self._bp[0].shape[0]), C.byref(nq), C.byref(npass)))
        return int(nq.value), int(npass.value)

    def shard_cov_chain(self, k_in: int) -> int:
        k_out = C.c_int64()
        self._ck(self.L.sqg_shard_cov_chain(self._h, int(k_in), C.byref(k_out)))
        return int(k_out.value)

    def shard_cov_owned_t(self, rank_offset: int, k_in: int, k_out: int, t_global: np.ndarray):
        assert t_global.dtype == np.int64 and t_global.flags.c_contiguous
        self._ck(self.L.sqg_shard_cov_owned_t(self._h, int(rank_offset), int(k_in), int(k_out), t_global.ctypes.data))

    def shard_cov_count(self, rank_offset: int, t_global: np.ndarray) -> np.ndarray:
        t = np.ascontiguousarray(t_global, np.int64)
        out = np.zeros(t.shape[0], np.int32)
        self._ck(self.L.sqg_shard_cov_count(self._h, int(rank_offset), t.ctypes.data, out.ctypes.data))
        return out

    def set_nodes(self, Chr, Position, Length):
        c = np.ascontiguousarray(Chr, np.int32); p = np.ascontiguousarray(Position, np.int32); l = np.ascontiguousarray(Length, np.int32)
        self._ck(self.L.sqg_set_nodes(self._h, c.ctypes.data, p.ctypes.data, l.ctypes.data, int(c.shape[0])))

    def BuildEdges(self) -> Edges:
        i1, i2, hd, w = _P(), _P(), _P(), _P()
        n = C.c_int64()
        cs = self.Chimrecord.as_struct() if self.Chimrecord is not None else None
        self._ck(self.L.sqg_build_edges(self._h, C.byref(i1), C.byref(i2), C.byref(hd), C.byref(w), C.byref(n), C.byref(cs) if cs is not None else None))
        m = n.value
        heads = _np_from(hd, m, np.uint8)
        self.vEdges = Edges(_np_from(i1, m, np.int32), _np_from(i2, m, np.int32), (heads & 1).astype(bool), ((heads >> 1) & 1).astype(bool), _np_from(w, m, np.int32))
        return self.vEdges

    def BPCoverage(self, bp_chr, bp_pos) -> np.ndarray:
        c = np.ascontiguousarray(bp_chr, np.int32); p = np.ascontiguousarray(bp_pos, np.int32)
        out = np.zeros(c.shape[0], np.int32)
        self._ck(self.L.sqg_bp_coverage(self._h, c.ctypes.data, p.ctypes.data, int(c.shape[0]), out.ctypes.data))
        return out

    def ExactBPConcordantSupport(self, final_nodes: np.ndarray, final_edges: np.ndarray, ExactBP: dict) -> dict:
        """Twin of SegmentGraph.cpp:3083-3221.  final_nodes rows (Chr,Position,Length,...), final_edges rows
        (Ind1,Ind2,Head1,Head2,...), ExactBP {(Ind1,Ind2,Head1,Head2): [(bp1,bp2),...]} ->
        {(edge): [(cov1,cov2),...]}.  The BAM pass runs on the GPU; assembling BPs and mapping back is host glue."""
        fn = np.asarray(final_nodes, dtype=np.int64)
        bps = []
        for e in final_edges:
            k = tuple(int(v) for v in e[:4])
            pairs = ExactBP.get(k)
            if pairs:
                for b1, b2 in pairs:
                    bps.append((int(fn[k[0], 0]), int(b1))); bps.append((int(fn[k[1], 0]), int(b2)))
            else:
                bps.append((int(fn[k[0], 0]), int(fn[k[0], 1] + (0 if k[2] else fn[k[0], 2]))))
                bps.append((int(fn[k[1], 0]), int(fn[k[1], 1] + (0 if k[3] else fn[k[1], 2]))))
        bps.sort()
        arr = np.array(bps, dtype=np.int64).reshape(-1, 2)
        cov = self.BPCoverage(arr[:, 0], arr[:, 1]) if len(bps) else np.zeros(0, np.int32)
        key = arr[:, 0] * (1 << 32) + arr[:, 1]
        out = {}
        for e in final_edges:
            k = tuple(int(v) for v in e[:4])
            pairs = ExactBP.get(k)
            sup = []
            if pairs:
                for b1, b2 in pairs:
                    sup.append((int(cov[np.searchsorted(key, fn[k[0], 0] * (1 << 32) + b1)]), int(cov[np.searchsorted(key, fn[k[1], 0] * (1 << 32) + b2)])))
            else:
                p1 = fn[k[0], 1] + (0 if k[2] else fn[k[0], 2]); p2 = fn[k[1], 1] + (0 if k[3] else fn[k[1], 2])
                sup.append((int(cov[np.searchsorted(key, fn[k[0], 0] * (1 << 32) + p1)]), int(cov[np.searchsorted(key, fn[k[1], 0] * (1 << 32) + p2)])))
            out[k] = sup
        return out

    # -- instrumentation ---------------------------------------------------------------------
    def phase_ms(self, name: str) -> float:
        return float(self.L.sqg_phase_ms(self._h, name.encode()))

    def launch_count(self) -> int:
        return int(self.L.sqg_launch_count(self._h))

    def stat(self, name: str) -> int:
        return int(self.L.sqg_stat(self._h, name.encode()))

    CLASSIFY_DTYPES = {"cls": np.uint8, "first_len": np.uint16, "gap_rec": np.int32, "gap_key": np.uint64, "pc_rec": np.int32,
                       "dp_rec": np.int32, "okmax_excl": np.uint64, "ccmax": np.int32, "cov_nq": np.uint32, "cov_qmax": np.uint64,
                       "qstage_key": np.uint64, "qstage_end": np.int32}

    def classify_dump(self, name: str) -> np.ndarray:
        """One phase-1 array of the resident batch (sqg_classify_dump); call before BuildNode_STAR, which reuses the buffers."""
        n = C.c_int64()
        self._ck(self.L.sqg_classify_dump(self._h, name.encode(), None, 0, C.byref(n)))
        out = np.zeros(n.value, self.CLASSIFY_DTYPES[name])
        self._ck(self.L.sqg_classify_dump(self._h, name.encode(), out.ctypes.data, out.shape[0], C.byref(n)))
        return out


def ExactBreakpoint(final_nodes: np.ndarray, Chimrecord: "ChimericReads", Concord_Dist_Pos: int = 50000, Concord_Dist_Idx: int = 20) -> np.ndarray:
    """Twin of SegmentGraph_t::ExactBreakpoint + CountTop (SegmentGraph.cpp:3019-3081, 51-102), host side.  final_nodes rows
    (Chr, Position, Length, ...); Chimrecord as BuildEdges left it (trimmed in place again here).  Returns rows
    (Ind1, Ind2, Head1, Head2, bp1, bp2) in the order of the reference's map."""
    L = lib()
    fn = np.ascontiguousarray(np.asarray(final_nodes)[:, :3].T, np.int32)
    cs = Chimrecord.as_struct()
    rows, n = _P(), C.c_int64()
    rc = L.sqh_exact_breakpoint(fn[0].ctypes.data, fn[1].ctypes.data, fn[2].ctypes.data, int(fn.shape[1]), C.byref(cs), int(Concord_Dist_Pos), int(Concord_Dist_Idx),
                                C.byref(rows), C.byref(n))
    if rc != 0:
        raise SquidB200Error(rc, "sqh_exact_breakpoint failed")
    out = _np_from(rows, 6 * n.value, np.int32).reshape(-1, 6)
    L.sqh_free(rows)
    return out


def ConnectedComponent(n_nodes: int, Ind1, Ind2, device: int = 0) -> np.ndarray:
    """Twin of SegmentGraph_t::ConnectedComponent (SegmentGraph.cpp:2986-3003) on the device: Label per node, components numbered
    in the order of their smallest node."""
    a = np.ascontiguousarray(Ind1, np.int32); b = np.ascontiguousarray(Ind2, np.int32)
    assert a.shape == b.shape
    out = np.empty(int(n_nodes), np.int32)
    nc = C.c_int32()
    rc = lib().sqg_connected_components(int(device), int(n_nodes), a.ctypes.data, b.ctypes.data, int(a.shape[0]), out.ctypes.data, C.byref(nc))
    if rc != 0:
        raise SquidB200Error(rc, "sqg_connected_components failed")
    return out


def OutputGraph(path: str, nodes: np.ndarray, avg_depth: np.ndarray, label: np.ndarray, edges: np.ndarray):
    """Twin of SegmentGraph_t::OutputGraph (SegmentGraph.cpp:3223-3234): <prefix>_graph.txt.  nodes rows (Chr, Position, Length,
    Support), edges rows (Ind1, Ind2, Head1, Head2, Weight)."""
    L = lib()
    nd = np.ascontiguousarray(np.asarray(nodes)[:, :4].T, np.int32)
    ad = np.ascontiguousarray(avg_depth, np.float64); lb = np.ascontiguousarray(label, np.int32)
    ed = np.asarray(edges).reshape(-1, 5)
    e = [np.ascontiguousarray(ed[:, 0], np.int32), np.ascontiguousarray(ed[:, 1], np.int32), np.ascontiguousarray(ed[:, 2], np.uint8), np.ascontiguousarray(ed[:, 3], np.uint8),
         np.ascontiguousarray(ed[:, 4], np.int32)]
    rc = L.sqh_write_graph(path.encode(), nd[0].ctypes.data, nd[1].ctypes.data, nd[2].ctypes.data, nd[3].ctypes.data, ad.ctypes.data, lb.ctypes.data, int(nd.shape[1]),
                           e[0].ctypes.data, e[1].ctypes.data, e[2].ctypes.data, e[3].ctypes.data, e[4].ctypes.data, int(ed.shape[0]))
    if rc != 0:
        raise SquidB200Error(rc, "sqh_write_graph failed")


def WriteBEDPE(path: str, ref_names, nodes: np.ndarray, edges: np.ndarray, components, exactbp_rows: np.ndarray, support_rows: np.ndarray,
               DiscordantRatio: float = 8.0, Concord_Dist_Pos: int = 50000, Concord_Dist_Idx: int = 20):
    """Twin of DeMultiplyDisEdges + WriteBEDPE (SegmentGraph.cpp:3012-3017; WriteIO.cpp:45-124): <prefix>_sv.txt.  edges rows
    (Ind1, Ind2, Head1, Head2, Weight) in vEdges order with the weights still multiplied; components = list of lists of signed
    1-based node ids (the ordering stage's output)."""
    L = lib()
    nd = np.ascontiguousarray(np.asarray(nodes)[:, :3].T, np.int32)
    ed = np.asarray(edges).reshape(-1, 5)
    e = [np.ascontiguousarray(ed[:, 0], np.int32), np.ascontiguousarray(ed[:, 1], np.int32), np.ascontiguousarray(ed[:, 2], np.uint8), np.ascontiguousarray(ed[:, 3], np.uint8),
         np.ascontiguousarray(ed[:, 4], np.int32)]
    off = np.zeros(len(components) + 1, np.int64)
    for i, c in enumerate(components):
        off[i + 1] = off[i] + len(c)
    flat = np.ascontiguousarray(np.concatenate([np.asarray(c, np.int32) for c in components]) if len(components) else np.zeros(0, np.int32), np.int32)
    xb = np.ascontiguousarray(exactbp_rows, np.int32).reshape(-1, 6); sp = np.ascontiguousarray(support_rows, np.int32).reshape(-1, 6)
    names = (C.c_char_p * len(ref_names))(*[n.encode() for n in ref_names])
    rc = L.sqh_write_bedpe(path.encode(), names, len(ref_names), nd[0].ctypes.data, nd[1].ctypes.data, nd[2].ctypes.data, int(nd.shape[1]),
                           e[0].ctypes.data, e[1].ctypes.data, e[2].ctypes.data, e[3].ctypes.data, e[4].ctypes.data, int(ed.shape[0]),
                           off.ctypes.data, flat.ctypes.data, len(components), xb.ctypes.data, int(xb.shape[0]), sp.ctypes.data, int(sp.shape[0]),
                           float(DiscordantRatio), int(Concord_Dist_Pos), int(Concord_Dist_Idx))
    if rc != 0:
        raise SquidB200Error(rc, "sqh_write_bedpe failed (%d)" % rc)


def plan_shards(batch: RecordBatch, chim: ChimericReads, config: Config, n_ref: int, n_shards: int):
    """sqg_plan_shards: clean cuts of the sorted stream.  Returns [c_0 = 0, ..., c_m = n_rec] with m <= n_shards."""
    L = lib()
    bs, cs, cfg = batch.as_struct(), chim.as_struct(), config.as_struct()
    cuts = np.zeros(n_shards + 1, np.int64)
    m = C.c_int32()
    rc = L.sqg_plan_shards(C.byref(bs), C.byref(cs), C.byref(cfg), int(n_ref), int(n_shards), cuts.ctypes.data, C.byref(m))
    if rc != 0:
        raise SquidB200Error(rc, "sqg_plan_shards failed")
    return [int(x) for x in cuts[: m.value + 1]]
