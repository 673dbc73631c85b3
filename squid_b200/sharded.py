"""Exact range-sharded run of the segment-graph path over several contexts / GPUs (SURVEY.md §8e; C ABI: "Exact range
sharding" in include/squid_b200.h).  One sorted stream is cut at clean cuts (api.plan_shards), every shard runs the path on
its own records, and the small per-shard results are exchanged between the stages:

    stage                    exchanged                                   reference lines it reproduces
    seeds                    seed ops (kind, chr, pos, len)              SegmentGraph.cpp:296-701
    build                    depth numerators (sum), edge tables         :706-826, :1932-1959
    hints                    LocateRead's firstfrontindex per boundary   :1568, :1612-1614
    coverage                 rank counts, chain hand-over k, t, counts   :3124-3166

The combined result is bit-identical to SegmentGraph on the whole stream.  `comm` hides where the shards live: LocalComm
(every shard in this process, e.g. several contexts on one GPU -- used by the GPU tests) or DistComm (one shard per
torch.distributed rank: NCCL on the GPUs, gloo in the CPU tests of this logic).  The exchange is written once, in terms of
`comm.allgather(list of per-local-shard items) -> list of items of ALL shards in shard order`.
"""
from __future__ import annotations

import numpy as np

from . import shard as _shard
from .api import ChimericReads, Config, Edges, Nodes, SegmentGraph


class LocalComm:
    """All shards live in this process."""
    rank, world = 0, 1

    def allgather(self, items: list) -> list:
        return list(items)

    def allgather_arrays(self, arrays: list) -> list:
        """One flat array per LOCAL shard -> the flat arrays of ALL shards, shard order."""
        return [np.ascontiguousarray(a).ravel() for a in arrays]

    def allreduce(self, a: np.ndarray, op: str) -> np.ndarray:
        """Elementwise "sum" (two's-complement wrap-around, like the reference's int accumulators) or "max" over the
        PROCESSES; the caller has already combined its local shards."""
        return a


class DistComm(LocalComm):
    """One process per GPU (torch.distributed, backend nccl or gloo); every process holds the same number of consecutive
    shards.  Arrays travel as tensors (on the GPU with NCCL: all_gather_into_tensor / all_reduce over NVLink); `allgather`
    of arbitrary objects is kept for the rare large optional payloads (the trimmed chimeric blocks)."""

    def __init__(self, group=None, device=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.group = torch, dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        nccl = dist.get_backend(group) == "nccl"
        self.dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device()) if nccl else torch.device("cpu"))

    def allgather(self, items: list) -> list:
        out = [None] * self.world
        self.dist.all_gather_object(out, list(items), group=self.group)
        return [x for sub in out for x in sub]

    def _t(self, a: np.ndarray):
        view = {np.dtype(np.uint64): np.int64, np.dtype(np.uint32): np.int32, np.dtype(np.uint16): np.int16}.get(a.dtype)
        return self.torch.from_numpy(a.view(view) if view else a)

    def allgather_arrays(self, arrays: list) -> list:
        torch = self.torch
        flat = [np.ascontiguousarray(a).ravel() for a in arrays]
        dt = flat[0].dtype
        sizes = torch.tensor([f.shape[0] for f in flat], dtype=torch.int64, device=self.dev)
        all_sizes = torch.empty(self.world * len(flat), dtype=torch.int64, device=self.dev)
        self.dist.all_gather_into_tensor(all_sizes, sizes, group=self.group)
        all_sizes = all_sizes.cpu().numpy().reshape(self.world, len(flat))
        width = int(all_sizes.sum(axis=1).max())
        mine = np.concatenate(flat) if flat else np.zeros(0, dt)
        buf = torch.zeros(max(width, 1), dtype=self._t(mine[:0]).dtype, device=self.dev)
        if mine.shape[0]:
            buf[: mine.shape[0]] = self._t(mine).to(self.dev)
        out = torch.empty(self.world * buf.shape[0], dtype=buf.dtype, device=self.dev)
        self.dist.all_gather_into_tensor(out, buf, group=self.group)
        out = out.cpu().numpy().reshape(self.world, buf.shape[0])
        res = []
        for r in range(self.world):
            o = 0
            for n in all_sizes[r]:
                res.append(out[r, o:o + int(n)].view(dt).copy())
                o += int(n)
        return res

    def allreduce(self, a: np.ndarray, op: str) -> np.ndarray:
        t = self._t(np.ascontiguousarray(a)).to(self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM if op == "sum" else self.dist.ReduceOp.MAX, group=self.group)
        return t.cpu().numpy().view(a.dtype).reshape(a.shape)


def dev_view(ptr, n, dtype, dev):
    """torch view of library-owned device memory (no copy)."""
    import torch

    class _Arr:
        pass
    a = _Arr()
    a.__cuda_array_interface__ = {"shape": (int(n),), "typestr": {torch.int64: "<i8", torch.int32: "<i4"}[dtype], "data": (int(ptr), False), "version": 2, "strides": None}
    return torch.as_tensor(a, device=dev)


# ---- the exchange logic, free of any device call (tested on CPU with gloo) --------------------------------------------------
def first_wrong_prior(assumed, op_counts):
    """Shards run stage 1 assuming `assumed[s]` = "an earlier shard has emitted a seed op".  Returns (s, truth) for the first
    shard whose assumption is wrong given the op counts of the current runs, or None."""
    seen = False
    for s, n in enumerate(op_counts):
        if assumed[s] != seen:
            return s, seen
        seen = seen or n > 0
    return None


def incoming_hints(states):
    """states[s] = (lead_sensitive, out_hint).  firstfrontindex entering shard s = out_hint of the nearest earlier shard that
    located a read, 0 at the start of the stream (SegmentGraph.cpp:1568)."""
    inc, cur = [], 0
    for lead, out in states:
        inc.append(cur)
        if out >= 0:
            cur = out
    return inc


def chain_k_in_guess(n_pass):
    """k_in[s] guess = number of breakpoints passed by some record of an earlier shard (exact unless indBP lags across the
    boundary)."""
    g, m = [], 0
    for x in n_pass:
        g.append(m)
        m = max(m, x)
    return g


def merge_depth(parts):
    """parts = [(count3, sumlen3, other_nonempty)] per shard -> sums in the reference's `int` arithmetic (wrap-around)."""
    c = np.zeros_like(parts[0][0]); s = np.zeros_like(parts[0][1]); o = 0
    with np.errstate(over="ignore"):
        for pc, ps, po in parts:
            c = (c + pc).astype(np.int32); s = (s + ps).astype(np.int32); o |= int(po)
    return c, s, o


class ShardedSegmentGraph:
    """SegmentGraph over range shards.  `shard_ids` = the shards held by this process (all of them with LocalComm)."""

    def __init__(self, config: Config, RefLength, n_shards: int, shard_ids, comm=None, devices=None, force_hint_redo: bool = False):
        self.comm = comm or LocalComm()
        self.force_hint_redo = force_hint_redo  # test hook: every shard repeats its edge pass with its true incoming hint
        self.config, self.RefLength, self.n_shards = config, np.ascontiguousarray(RefLength, np.int32), int(n_shards)
        self.ids = list(shard_ids)
        devices = devices if devices is not None else [0] * len(self.ids)
        self.g = [SegmentGraph(config, self.RefLength, device=d) for d in devices]
        for g, sid in zip(self.g, self.ids):
            g.set_shard(sid, self.n_shards)
        self.vNodes = None
        self.vEdges = None
        self.Chimrecord = None
        self.rounds = {"seeds": 0, "hints": 0, "chain": 0}
        self.detail_ms = {}  # host wall clock per sub-stage (exchanges included), accumulated over the calls
        self._t = None

    def _lap(self, name=None):
        import time
        now = time.perf_counter()
        if name is not None and self._t is not None:
            self.detail_ms[name] = self.detail_ms.get(name, 0.0) + 1e3 * (now - self._t)
        self._t = now

    def close(self):
        for g in self.g:
            g.close()

    def load(self, batches, chim_factory):
        """batches[i] = RecordBatch of local shard i; chim_factory() -> a fresh ChimericReads (every shard gets all reads)."""
        for g, b in zip(self.g, batches):
            g.load_concordant(b)
            g.load_chimeric(chim_factory())

    def load_bam(self, path: str, case):
        """Every local shard context decodes the whole concordant BAM on its device (load_concordant_bam), loads all chimeric
        reads, plans the cuts on the resident batch (plan_shards) and keeps its own record range (keep_records).  No records
        travel between the ranks: each plans the same cuts from the same file, and one all-gather checks that they did.
        `case` = HostCase(conc, chim, bam=True, header_only=True).  Returns the cuts; raises ValueError when the stream has
        fewer clean cuts than shards."""
        mine = []
        for g in self.g:
            g.load_concordant_bam(path, case)
            g.load_chimeric(ChimericReads(case.chimeric.a))
            mine.append(g.plan_shards(self.n_shards))
        every = self.comm.allgather(mine)
        if any(c != every[0] for c in every):
            raise RuntimeError("shard contexts planned different cuts: %s" % every)
        cuts = every[0]
        if len(cuts) - 1 < self.n_shards:
            raise ValueError("the stream has %d clean shards, not %d: cuts %s" % (len(cuts) - 1, self.n_shards, cuts))
        for g, sid in zip(self.g, self.ids):
            g.keep_records(cuts[sid], cuts[sid + 1])
        return cuts

    # -- BuildNode_STAR ------------------------------------------------------------------------------------------------
    def BuildNode_STAR(self) -> Nodes:
        N = self.n_shards
        assumed = [s > 0 for s in range(N)]
        self._lap()
        ops = [g.shard_seeds(assumed[sid]) for g, sid in zip(self.g, self.ids)]
        self._lap("nodes: shard_seeds")
        while True:
            self.rounds["seeds"] += 1
            all_ops = [o.reshape(-1, 4) for o in self.comm.allgather_arrays(ops)]
            wrong = first_wrong_prior(assumed, [int(o.shape[0]) for o in all_ops])
            if wrong is None:
                break
            s, truth = wrong
            assumed[s] = truth
            if s in self.ids:
                i = self.ids.index(s)
                ops[i] = self.g[i].shard_seeds(truth)
        cat = np.concatenate(all_ops, axis=0) if all_ops else np.zeros((0, 4), np.int32)
        self._lap("nodes: seed-op exchange")
        parts, node = [], None
        for g in self.g:
            c, p, l, c3, s3, other = g.shard_build(cat)
            node = (c, p, l)
            parts.append((c3, s3, other))
        self._lap("nodes: shard_build")
        count3, sum3, other = merge_depth(parts)  # the local shards; then across the processes, in one int32 vector
        tot = self.comm.allreduce(np.concatenate([count3.ravel(), sum3.ravel(), np.array([other], np.int32)]).astype(np.int32), "sum")
        nn = count3.size
        count3, sum3, other = tot[:nn].reshape(count3.shape), tot[nn:2 * nn].reshape(sum3.shape), int(tot[2 * nn] != 0)
        self._lap("nodes: depth all-reduce")
        self._fix_hints()
        self._lap("nodes: hint exchange")
        length = node[2]
        support = count3[0] + count3[1] + (count3[2] if other else 0)  # as api.SegmentGraph.BuildNode_STAR
        depth = sum3[0].astype(np.float64) + sum3[1].astype(np.float64)
        if other:
            depth = depth + sum3[2].astype(np.float64)
            depth = 1.0 * depth / length
        self.vNodes = Nodes(node[0], node[1], length, support.astype(np.int32), depth, count3, sum3)
        return self.vNodes

    def _fix_hints(self):
        used = [0] * self.n_shards
        while True:
            self.rounds["hints"] += 1
            st = self.comm.allgather_arrays([np.array(g.shard_hint_state(), np.int32) for g in self.g])
            states = [(bool(x[0]), int(x[1])) for x in st]
            inc = incoming_hints(states)
            redo = [s for s in range(self.n_shards) if (states[s][0] or self.force_hint_redo) and used[s] != inc[s]]
            if not redo:
                return
            for s in redo:
                used[s] = inc[s]
                if s in self.ids:
                    self.g[self.ids.index(s)].shard_redo_edges(inc[s])

    # -- BuildEdges ----------------------------------------------------------------------------------------------------
    def _merge_edges_on_device(self):
        """One shard per process over NCCL: the per-shard (key, weight) tables never leave HBM -- one all_gather of
        [count | keys | weights] per rank, then sort + reduce-by-key on the device (sqg_merge_edge_tables)."""
        import ctypes as C
        comm, g = self.comm, self.g[0]
        torch, dist, dev = comm.torch, comm.dist, comm.dev
        dk, dw, n = C.c_void_p(), C.c_void_p(), C.c_int64()
        g._ck(g.L.sqg_edges_device_table(g._h, C.byref(dk), C.byref(dw), C.byref(n)))
        m = n.value
        mx_t = torch.tensor([m], dtype=torch.int64, device=dev)
        dist.all_reduce(mx_t, op=dist.ReduceOp.MAX, group=comm.group)
        mx = int(mx_t.item())
        buf = torch.zeros(1 + 2 * mx, dtype=torch.int64, device=dev)
        buf[0] = m
        if m:
            buf[1:1 + m] = dev_view(dk.value, m, torch.int64, dev)
            buf[1 + mx:1 + mx + m] = dev_view(dw.value, m, torch.int32, dev).to(torch.int64)
        allb = torch.empty(comm.world * (1 + 2 * mx), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allb, buf, group=comm.group)
        allb = allb.view(comm.world, 1 + 2 * mx)
        cnts = allb[:, 0].tolist()
        allk = torch.cat([allb[r, 1:1 + int(cnts[r])] for r in range(comm.world)])
        allw = torch.cat([allb[r, 1 + mx:1 + mx + int(cnts[r])] for r in range(comm.world)]).to(torch.int32)
        torch.cuda.current_stream().synchronize()  # the library works on its own stream
        i1, i2, hd, w, ne = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64()
        g._ck(g.L.sqg_merge_edge_tables(g._h, allk.data_ptr(), allw.data_ptr(), int(allk.shape[0]), C.byref(i1), C.byref(i2), C.byref(hd), C.byref(w), C.byref(ne)))
        k = ne.value
        from .api import _np_from
        heads = _np_from(hd, k, np.uint8)
        return Edges(_np_from(i1, k, np.int32), _np_from(i2, k, np.int32), (heads & 1).astype(bool), ((heads >> 1) & 1).astype(bool), _np_from(w, k, np.int32))

    def BuildEdges(self, gather_chimeric: bool = True) -> Edges:
        """gather_chimeric=False: the trimmed chimeric blocks stay with the process that holds shard 0."""
        if isinstance(self.comm, DistComm) and self.comm.dev.type == "cuda" and len(self.g) == 1:
            self._lap()
            self.g[0].BuildEdges()  # this shard's table (and, on shard 0, the in-place trim of the chimeric blocks)
            chim = self.g[0].Chimrecord if self.ids[0] == 0 else None
            self._lap("edges: local tables")
            self.vEdges = self._merge_edges_on_device()
            self._lap("edges: all-gather + merge on the device")
            if gather_chimeric and self.comm.world > 1:
                got = self.comm.allgather([chim.a if chim is not None else None])
                ca = next((a for a in got if a is not None), None)
                chim = ChimericReads(ca) if ca is not None else None
            self.Chimrecord = chim
            return self.vEdges
        keys, ws, chim = [], [], None
        self._lap()
        for g, sid in zip(self.g, self.ids):
            e = g.BuildEdges()
            keys.append(_shard.pack_edge_keys(e.Ind1, e.Ind2, e.Head1, e.Head2)); ws.append(e.Weight)
            if sid == 0:
                chim = g.Chimrecord  # trimmed in place by shard 0 (it owns the chimeric reads' LocateRead pass)
        self._lap("edges: local tables")
        all_k, all_w = self.comm.allgather_arrays(keys), self.comm.allgather_arrays(ws)
        self._lap("edges: all-gather")
        mk, mw = _shard.merge_edge_tables(list(zip(all_k, all_w)))
        i1, i2, h1, h2 = _shard.unpack_edge_keys(mk)
        self.vEdges = Edges(i1, i2, h1, h2, mw)
        self._lap("edges: merge")
        if gather_chimeric and self.comm.world > 1:
            got = self.comm.allgather([chim.a if (chim is not None and sid == 0) else None for sid in self.ids])
            ca = next((a for a in got if a is not None), None)
            chim = ChimericReads(ca) if ca is not None else None
        self.Chimrecord = chim
        return self.vEdges

    # -- ExactBPConcordantSupport's BAM pass -----------------------------------------------------------------------------
    def BPCoverage(self, bp_chr, bp_pos) -> np.ndarray:
        K = int(np.asarray(bp_chr).shape[0])
        if K == 0:
            return np.zeros(0, np.int32)
        self._lap()
        begun = [np.array(g.shard_cov_begin(bp_chr, bp_pos), np.int64) for g in self.g]
        self._lap("coverage: begin")
        info = self.comm.allgather_arrays(begun)
        self._lap("coverage: begin exchange")
        nq = [int(x[0]) for x in info]
        off = np.concatenate([[0], np.cumsum(nq)]).astype(np.int64)
        k_in = chain_k_in_guess([int(x[1]) for x in info])
        k_in[0] = 0
        k_out = {sid: g.shard_cov_chain(k_in[sid]) for g, sid in zip(self.g, self.ids)}
        self._lap("coverage: chain")
        while True:
            self.rounds["chain"] += 1
            outs = [int(x[0]) for x in self.comm.allgather_arrays([np.array([k_out[sid]], np.int64) for sid in self.ids])]
            redo = [s for s in range(1, self.n_shards) if k_in[s] != outs[s - 1]]
            if not redo:
                break
            s = redo[0]  # the hand-over is sequential: settle the first broken link, later ones may change with it
            k_in[s] = outs[s - 1]
            if s in self.ids:
                k_out[s] = self.g[self.ids.index(s)].shard_cov_chain(k_in[s])
        self._lap("coverage: chain exchange")
        t = np.full(K, -1, np.int64)
        for g, sid in zip(self.g, self.ids):
            g.shard_cov_owned_t(int(off[sid]), k_in[sid], k_out[sid], t)
        self._lap("coverage: owned t")
        t = self.comm.allreduce(t, "max")  # every process filled the entries its shards own
        t[t < 0] = int(off[-1])  # never passed: every qualifying record is tested against the breakpoint
        self._lap("coverage: t all-reduce")
        cov = np.zeros(K, np.int32)
        for g, sid in zip(self.g, self.ids):
            cov += g.shard_cov_count(int(off[sid]), t)
        self._lap("coverage: count")
        out = self.comm.allreduce(cov, "sum")
        self._lap("coverage: count all-reduce")
        return out
