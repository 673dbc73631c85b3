#!/usr/bin/env python
"""Benchmark of the B200 segment-graph construction path (BASELINE.json metric: read pairs/s through
segment-graph build, with % of HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: BuildNode_STAR + BuildEdges + breakpoint coverage on
synthetic sorted alignment records of the configs[1] shape (GRCh38 layout, ~0.5 % discordant, SURVEY App. C block mix K = 1.35).
  value : whole-job pairs/s with the record batch already resident in HBM when the timed region starts
  e2e   : the same through the C ABI with HOST (pinned) buffers: H2D of the batch inside the timed region
  roofline : the kernel with the longest live CUDA-event time in the step: algorithmic bytes (SURVEY.md §8d / DESIGN.md §3) / that
             time / measured HBM peak; every timed kernel is listed under roofline.kernels, the whole path under roofline.whole_path
  parity   : CRC32 of every output of the step against the reference build's on the same stream (tests/golden/bench_crc.json);
             a mismatch makes the run exit 3
  cpu_baseline : the reference's own BuildNode_STAR/BuildEdges/ExactBPConcordantSupport (oracle/_ref, single thread)
                 on a bounded sample of the same generator
N > 1: weak scaling over N independent streams, one per rank (a cohort of N samples; every rank generates its own copy of the
same stream so that the work per GPU is fixed -- SQUID_BENCH_DISTINCT_STREAMS=1 gives every rank another seed): every rank runs
the whole path on its own stream; independent samples have nothing to exchange, so there is no data-path collective (round 1 merged the
per-rank edge tables anyway: 10 ms of an 8-GPU step spent on a table that means nothing across samples).  The same
run also times ONE stream (rank 0's) cut into N exact genomic-range shards -- bit-identical results for every N, checked against
the pinned CRCs -- and reports it as `one_stream` (strong scaling, DESIGN.md §9).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DEFAULT_PAIRS = int(os.environ.get("SQUID_BENCH_PAIRS", 100_000_000))
DISC_FRAC = 0.005
CPU_SAMPLE_PAIRS = int(os.environ.get("SQUID_BENCH_CPU_PAIRS", 2_000_000))   # one reference run on it: ~4 s on one core
REF_ARM_PAIRS = int(os.environ.get("SQUID_BENCH_REF_PAIRS", 4_000_000))      # --impl reference: ~8 s per step, the largest sample that keeps 25 steps within a few minutes
# SURVEY.md App. C: 100-bp reads, ~70 % unspliced / ~30 % spliced, K = 1.35 aligned blocks per record.  The splicing comes from
# the transcript model (reads laid on exon chains), so K is set through the exon length range; pairs with an aligned block
# under 4 bp are dropped by the generator (STAR's default minimum splice overhangs are 3-5 bp).
BENCH_EXON_LEN = (60, 460)
BENCH_MIN_BLOCK = 4
CRC_FILE = os.path.join(ROOT, "tests", "golden", "bench_crc.json")


def make_workload(pairs: int, seed: int, device: str):
    from squid_b200 import synth_gpu
    return synth_gpu.make_bench_batch(pairs, seed=seed, device=device, exon_len=BENCH_EXON_LEN, min_block=BENCH_MIN_BLOCK)


def workload_id(pairs: int, seed: int) -> str:
    return "grch38 pairs=%d seed=%d disc=%g exon_len=%d-%d min_block=%d genes=20000" % (pairs, seed, DISC_FRAC, BENCH_EXON_LEN[0], BENCH_EXON_LEN[1], BENCH_MIN_BLOCK)


def output_crcs(nodes, edges, chim_blocks, cov) -> dict:
    """CRC32 of every output of one step, in the layout of the reference harness's dumps."""
    import zlib
    c = lambda a: zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xffffffff
    nd = np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32)
    return {"nodes": c(nd), "avgdepth": c(np.asarray(nodes.AvgDepth, np.float64)), "edges": c(edges.table()), "chim_after_edges": c(np.asarray(chim_blocks, np.int32)),
            "coverage": c(np.asarray(cov, np.int32)), "n_nodes": int(nd.shape[0]), "n_edges": int(edges.Ind1.shape[0]), "n_bp": int(np.asarray(cov).shape[0])}


DUMP_BYTES_PER_ARRAY = 12 << 20  # five arrays: at most 60 MB in all


def dump_outputs(outdir: str, nodes, edges, chim_blocks, cov) -> None:
    """Writes the outputs of one step as float64 .npy files (exact for their int32 values), in the layout of output_crcs().
    An array larger than DUMP_BYTES_PER_ARRAY is replaced by a fixed sample of its rows (seed 0, original order), which
    depends on the row count only, so two builds that agree on the count dump the same rows."""
    os.makedirs(outdir, exist_ok=True)
    arrays = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1), "avgdepth": np.asarray(nodes.AvgDepth),
              "edges": edges.table(), "chim_after_edges": np.asarray(chim_blocks), "coverage": np.asarray(cov)}
    for name, a in arrays.items():
        a = np.asarray(a, np.float64)
        if a.nbytes > DUMP_BYTES_PER_ARRAY:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_BYTES_PER_ARRAY // a[:1].nbytes, replace=False))]
        np.save(os.path.join(outdir, name + ".npy"), a)


def pinned_crcs(pairs: int, seed: int):
    """Reference CRCs of this exact workload, if it has been pinned (tests/tools/pin_bench_crc.py ran the reference on it)."""
    try:
        for rec in json.load(open(CRC_FILE)):
            if rec["workload"] == workload_id(pairs, seed):
                return rec
    except Exception:
        pass
    return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index, self.t0, self.t1 = [], None, index, None, None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")] + [time.time()])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        # nvidia-smi takes a while to start, so it is started before the warm-up steps; only the samples that arrived between
        # mark_begin() and mark_end() -- the timed region -- are used (all samples under load if that window caught none)
        window = "timed region"
        if self.t0 is not None and self.t1 is not None:
            inside = [r for r in self.rows if self.t0 <= r[-1] <= self.t1]
            if inside:
                self.rows = inside
            else:
                window = "warm-up + timed steps (no sample fell inside the timed region)"
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: take one synchronous sample
            try:
                q = "clocks.sm,clocks.max.sm"
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
                a, b = [float(x) for x in o.strip().split(",")[:2]]
                sm, mx = [a], [b]
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "window": window}


def bps_from_graph(nodes, edges, min_weight=5):
    """Stand-in for the out-of-scope host stages between BuildEdges and ExactBPConcordantSupport: every edge of weight
    >= -w contributes its two segment-end breakpoints (SegmentGraph.cpp:3100-3107), sorted as at :3109."""
    keep = edges.Weight >= min_weight
    i1, i2 = edges.Ind1[keep], edges.Ind2[keep]
    p1 = nodes.Position[i1] + np.where(edges.Head1[keep], 0, nodes.Length[i1])
    p2 = nodes.Position[i2] + np.where(edges.Head2[keep], 0, nodes.Length[i2])
    c = np.concatenate([nodes.Chr[i1], nodes.Chr[i2]]).astype(np.int64)
    p = np.concatenate([p1, p2]).astype(np.int64)
    key = np.sort((c << 32) | p)  # (chr, pos) ascending; positions are non-negative
    return (key >> 32).astype(np.int32), (key & 0xffffffff).astype(np.int32)


def reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path (oracle/_ref = its unmodified sources), single thread,
    on a bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import pyref
    from squid_b200 import sqmb, synth
    pyref.build()
    P = REF_ARM_PAIRS
    with tempfile.TemporaryDirectory() as d:
        conc, chim, info = synth.make_case(P, ref_len=synth.GRCH38_LEN, seed=100, disc_frac=DISC_FRAC, n_genes=20000, adversarial=False, exon_len=BENCH_EXON_LEN, min_block=BENCH_MIN_BLOCK)
        sqmb.write_sqmb(d + "/conc.sqmb", conc); sqmb.write_sqmb(d + "/chim.sqmb", chim)
        n_pairs = conc.n / 2.0
        times = []
        for i in range(args.warmup + args.steps):
            r = pyref.run(d + "/conc.sqmb", d + "/chim.sqmb", d + "/out")
            t = r["timings"]
            if i >= args.warmup:
                times.append(t["build_nodes_s"] + t["build_edges_s"] + t["bp_coverage_s"])
    sec = float(np.mean(times))
    val = n_pairs / sec
    cpu = {"value": val, "unit": "read pairs/s", "cores": 1, "kind": "reference",
           "sample": "%d read pairs, GRCh38 layout, %.1f%% discordant; BuildNode_STAR+BuildEdges+ExactBPConcordantSupport of the reference's own sources (oracle/_ref), in-memory BAM shim" % (int(n_pairs), 100 * DISC_FRAC)}
    print(json.dumps({"impl": "reference", "metric": "read pairs/s through segment-graph build", "value": val, "unit": "read pairs/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "int32", "data": "synthetic", "config": {"workload": "synthetic GRCh38-layout read pairs, ~0.5% discordant, K = 1.35 blocks/record (bounded sample of configs[1]: the largest that keeps the run within a few minutes on one core)", "pairs_per_step": int(n_pairs)},
                      "cpu_baseline": cpu, "e2e": {"value": val, "unit": "read pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_leg(device: int = 0):
    """The reference on a bounded sample, and -- on the SAME input files -- this repo's whole flow starting where the reference
    starts: open the two alignment tables, decode every record (ReadRec_t twin), pack, ChimName probes, upload, BuildNode_STAR,
    BuildEdges, ExactBreakpoint, ExactBPConcordantSupport.  `same_input` is the like-for-like comparison (equal work, equal
    pair count); the outputs of the two are compared as well."""
    from oracle import pyref
    from squid_b200 import sqmb, synth
    try:
        pyref.build()
        if not pyref.available():
            return None
        P = CPU_SAMPLE_PAIRS
        with tempfile.TemporaryDirectory() as d:
            conc, chim, info = synth.make_case(P, ref_len=synth.GRCH38_LEN, seed=100, disc_frac=DISC_FRAC, n_genes=20000, adversarial=False, exon_len=BENCH_EXON_LEN, min_block=BENCH_MIN_BLOCK)
            sqmb.write_sqmb(d + "/conc.sqmb", conc); sqmb.write_sqmb(d + "/chim.sqmb", chim)
            r = pyref.run(d + "/conc.sqmb", d + "/chim.sqmb", d + "/out")
            same = None
            try:
                same = same_input_leg(d + "/conc.sqmb", d + "/chim.sqmb", r, conc.n / 2.0, device)
            except Exception as e:
                same = {"failed": str(e)}
        t = r["timings"]
        sec = t["build_nodes_s"] + t["build_edges_s"] + t["bp_coverage_s"]
        if same and "seconds" in same:
            same["reference_seconds"] = sec
            same["ratio"] = sec / same["seconds"]
        return {"value": (conc.n / 2.0) / sec, "unit": "read pairs/s", "cores": 1, "kind": "reference",
                "sample": "%d read pairs of the same generator; reference's own sources (oracle/_ref), single thread, BGZF excluded; phases s: nodes %.2f edges %.2f coverage %.2f" % (conc.n // 2, t["build_nodes_s"], t["build_edges_s"], t["bp_coverage_s"]),
                "same_input": same}
    except Exception as e:  # the baseline is informative; never fail the bench on it
        return {"value": None, "unit": "read pairs/s", "cores": 1, "kind": "reference", "sample": "failed: %s" % e}


def same_input_leg(cp, hp, ref, n_pairs, device):
    from oracle import pyref
    from squid_b200 import api
    best = None
    for it in range(5):  # the first pass pays the allocations of a fresh context
        t0 = time.perf_counter()
        case = api.HostCase(cp, hp)
        t1 = time.perf_counter()
        g = api.SegmentGraph(case.config, case.ref_len, device=device)
        nodes = g.BuildNode_STAR(case.chimeric, case.batch)
        edges = g.BuildEdges()
        t2 = time.perf_counter()
        # the host stages between BuildEdges and the breakpoint pass are out of scope: their result (final graph) is the reference's
        ebp = api.ExactBreakpoint(ref["final_nodes"], case.chimeric, case.config.Concord_Dist_Pos, case.config.Concord_Dist_Idx)
        sup = g.ExactBPConcordantSupport(ref["final_nodes"], ref["final_edges"], _rows_to_map(ebp))
        t3 = time.perf_counter()
        cur = {"open_decode_pack_s": t1 - t0, "graph_s": t2 - t1, "breakpoints_s": t3 - t2, "seconds": t3 - t0}
        if best is None or cur["seconds"] < best["seconds"]:
            best = cur
        got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth, "edges": edges.table()}
        ok = all(np.array_equal(ref[k], got[k]) for k in ("nodes", "avgdepth", "edges")) and sup == pyref.support_map(ref)
        g.close(); case.close()
        if not ok:
            break
    best.update({"pairs": int(n_pairs), "value": n_pairs / best["seconds"], "unit": "read pairs/s", "outputs_equal_reference": bool(ok), "host_threads": os.cpu_count(),
                 "what": "same two input tables as the reference run; timed from opening them to the support map: host decode/pack on all cores + upload + CUDA path (best of 5)"})
    return best


def _rows_to_map(rows6):
    m = {}
    for r in np.asarray(rows6).reshape(-1, 6):
        m.setdefault((int(r[0]), int(r[1]), int(r[2]), int(r[3])), []).append((int(r[4]), int(r[5])))
    return m


def stream_case(pairs: int, seed: int):
    """Chimeric reads + config of the stream (pairs, seed) through the host loader, without generating its concordant records."""
    from squid_b200 import api, sqmb, synth
    rng = np.random.Generator(np.random.PCG64(seed))
    tx = synth.Transcriptome(rng, np.asarray(synth.GRCH38_LEN, dtype=np.int64), 20000, exon_len=BENCH_EXON_LEN)
    prob = tx.g_expr / tx.g_expr.sum()
    chim_tab, _ = synth.make_chimeric(tx, prob, pairs, seed, DISC_FRAC, adversarial=False)
    with tempfile.TemporaryDirectory() as d:
        sqmb.write_sqmb(d + "/chim.sqmb", chim_tab)
        sqmb.write_sqmb(d + "/conc.sqmb", sqmb.empty(synth.GRCH38_LEN, 0))
        case = api.HostCase(d + "/conc.sqmb", d + "/chim.sqmb")
    return case, case.chimeric


def one_stream_leg(args, rank, world, local, dev, batch, chim0, case, steps, warmup):
    """N > 1, north_star's split: ONE sorted stream -- rank 0's stream, the very stream the single-GPU run measures -- cut at
    clean cuts into N exact genomic-range shards (sqg_plan_shards), one per GPU; seed ops, depth numerators, edge tables,
    LocateRead hints and the coverage chain cross the ranks over NCCL (squid_b200/sharded.py).  The combined outputs are
    bit-identical to the single-GPU run, so they are held against the same pinned reference CRCs.  Strong scaling."""
    import torch
    import torch.distributed as dist
    from squid_b200 import api, sharded, synth_gpu
    comm = sharded.DistComm()
    shm = "/dev/shm/sq_bench_%s" % os.environ.get("MASTER_PORT", "0")
    t_plan = 0.0
    if rank == 0:
        os.makedirs(shm, exist_ok=True)
        host = {k: v.cpu().numpy() for k, v in batch.items()}
        hb = api.RecordBatch({k: (v.view(np.uint16) if v.dtype == np.int16 else v.view(np.uint32) if k == "blk_off" else v) for k, v in host.items()})
        t0 = time.perf_counter()
        cuts = api.plan_shards(hb, chim0, case.config, len(case.ref_len), world)
        t_plan = time.perf_counter() - t0
        ok = len(cuts) - 1 == world
        if ok:
            for r in range(world):
                for k, v in hb.slice(cuts[r], cuts[r + 1]).a.items():
                    np.save("%s/%d_%s.npy" % (shm, r, k), v)
        json.dump({"cuts": cuts, "ok": ok}, open(shm + "/cuts.json", "w"))
        del hb, host
    dist.barrier()
    meta = json.load(open(shm + "/cuts.json"))
    if not meta["ok"]:
        return {"unavailable": "the planner found %d clean shards for %d ranks" % (len(meta["cuts"]) - 1, world)}
    cuts = meta["cuts"]
    mine = {k: np.load("%s/%d_%s.npy" % (shm, rank, k)) for k in api.BATCH_DTYPES}
    dbatch = {k: torch.from_numpy(v.view(np.int16) if v.dtype == np.uint16 else v.view(np.int32) if v.dtype == np.uint32 else v).to(dev) for k, v in mine.items()}
    del mine
    dist.barrier()
    if rank == 0:
        for f in os.listdir(shm):
            os.unlink(os.path.join(shm, f))
        os.rmdir(shm)
    dstruct = synth_gpu.batch_struct(dbatch)
    sg = sharded.ShardedSegmentGraph(case.config, case.ref_len, world, [rank], comm=comm, devices=[local])
    g = sg.g[0]
    st = {}

    def step():
        pool = st.setdefault("pool", [])
        chim = pool.pop() if pool else api.ChimericReads(chim0.a)
        st["chim"] = chim
        g.attach_concordant_device(dstruct, keepalive=dbatch, first_record_index=cuts[rank])
        g.load_chimeric(chim)
        t0 = time.perf_counter()
        nodes = sg.BuildNode_STAR()
        t1 = time.perf_counter()
        edges = sg.BuildEdges(gather_chimeric=False)
        t2 = time.perf_counter()
        if "bps" not in st:
            st["bps"] = bps_from_graph(nodes, edges)
        bc, bp = st["bps"]
        cov = sg.BPCoverage(bc, bp)
        t3 = time.perf_counter()
        tl = st.setdefault("tl", {})
        for k, v in (("BuildNode_STAR", t1 - t0), ("BuildEdges", t2 - t1), ("BPCoverage", t3 - t2)):
            tl[k] = tl.get(k, 0.0) + 1e3 * v
        return nodes, edges, cov

    def barrier():
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    st["pool"] = [api.ChimericReads(chim0.a) for _ in range(steps)]
    st["tl"] = {}
    sg.rounds = {"seeds": 0, "hints": 0, "chain": 0}
    sg.detail_ms = {}
    barrier()
    t = time.perf_counter()
    for _ in range(steps):
        nodes, edges, cov = step()
    barrier()
    sec = (time.perf_counter() - t) / steps
    tt = torch.tensor([sec], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    sec = float(tt.item())
    per_rank = comm.allgather([{"rank": rank, "records": int(cuts[rank + 1] - cuts[rank]), "host_timeline_ms": {k: round(v / steps, 2) for k, v in st["tl"].items()},
                                "detail_ms": {k: round(v / steps, 2) for k, v in sg.detail_ms.items()}}])
    out = None
    if rank == 0:
        R = cuts[-1]
        got = output_crcs(nodes, edges, st["chim"].block_table(), cov)
        out = {"mode": "ONE stream of %d read pairs in %d exact genomic-range shards (sqg_plan_shards), NCCL exchanges between the stages" % (R // 2, world),
               "scaling": "strong", "value": (R // 2) / sec, "unit": "read pairs/s", "ms_per_step": 1e3 * sec, "planner_s": round(t_plan, 3), "cuts": cuts,
               "exchange_rounds_per_step": {k: v / steps for k, v in sg.rounds.items()}, "per_rank": per_rank, "crc32": got}
    sg.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=DEFAULT_PAIRS, help="read pairs per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (resident batch) as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from squid_b200 import api, build, sqmb, synth, synth_gpu

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    build.build(verbose=False)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    real_stdout = None
    if world > 1:
        # NCCL prints its version banner on stdout: keep stdout clean for the one JSON line
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)

    P = args.pairs
    # ---- workload: generated on the device, sorted; chimeric reads through the host loader --------------------
    t0 = time.time()
    # Weak scaling = the SAME work on every GPU: each rank generates its own copy of the stream of seed0 (the configuration the
    # single-GPU line is quoted on).  Streams of different seeds differ by up to 25 % in cost (a fusion hub inside a highly expressed
    # gene makes the seed machine and the coverage count heavier), and the step time of the job is the maximum over the ranks: with
    # seed0 + rank the 8-GPU line measured which rank had drawn the heaviest sample, not the machine.
    seed0 = int(os.environ.get("SQUID_BENCH_SEED", 100))
    seed_r = seed0 + rank if os.environ.get("SQUID_BENCH_DISTINCT_STREAMS") else seed0
    batch, tx, prob = make_workload(P, seed_r, str(dev))
    chim_tab, fusions = synth.make_chimeric(tx, prob, P, seed_r, DISC_FRAC, adversarial=False)
    with tempfile.TemporaryDirectory() as d:
        sqmb.write_sqmb(d + "/chim.sqmb", chim_tab)
        sqmb.write_sqmb(d + "/conc.sqmb", sqmb.empty(synth.GRCH38_LEN, 0))
        case = api.HostCase(d + "/conc.sqmb", d + "/chim.sqmb")
    cfg = case.config
    chim0 = case.chimeric
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    R = int(batch["ref_id"].shape[0]); NB = int(batch["blk_ref_pos"].shape[0])
    P_req, P = P, R // 2  # the generator drops pairs with <4-bp blocks: count what is really there
    n_bytes = synth_gpu.batch_bytes(batch)
    dstruct = synth_gpu.batch_struct(batch)
    # Host copies for the end-to-end legs.  One GPU: the batch in page-locked memory in both forms (wire = the headline, SoA = the
    # resident layout shipped as it is).  N GPUs on one host: only the wire form is page-locked (N x 14 GB of pinned memory is more
    # than a host should be asked for); it is packed from a pageable copy that is dropped afterwards, and e2e_soa is not measured.
    want_soa = world == 1
    host_kind = "pinned"
    host = None
    if want_soa:
        try:
            host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in batch.items()}
        except RuntimeError as e:
            print("[rank %d] pinning the host batch failed (%s): e2e_soa is measured from pageable memory" % (rank, str(e).splitlines()[0]), file=sys.stderr, flush=True)
            host_kind = "wire pinned; SoA pageable (pinning failed)"
    if host is None:
        host = {k: torch.empty(v.shape, dtype=v.dtype) for k, v in batch.items()}
    for k in batch:
        host[k].copy_(batch[k])
    torch.cuda.synchronize()
    hstruct = synth_gpu.batch_struct(host)
    t_pack = time.perf_counter()
    host_rb = api.RecordBatch({k: v.numpy().view(api.BATCH_DTYPES[k]) for k, v in host.items()})  # views: no copy
    try:
        wire = api.WireBatch(host_rb, pinned=True)
    except api.SquidB200Error as e:
        print("[rank %d] page-locking the wire batch failed (%s): e2e is measured from pageable memory" % (rank, e), file=sys.stderr, flush=True)
        wire = api.WireBatch(host_rb, pinned=False)
        host_kind = "pageable (pinning failed)"
    t_pack = time.perf_counter() - t_pack
    wire._keep = None
    if not want_soa:
        del host_rb, host, hstruct
        host = hstruct = None

    g = api.SegmentGraph(cfg, case.ref_len, device=local)
    state = {}

    def step(mode: str):  # where the batch comes from: "resident" (HBM), "wire" (host, compact wire form), "soa" (host, resident layout)
        tl = state.setdefault("timeline", {})
        t_ = [time.perf_counter()]

        def lap(name):
            t1 = time.perf_counter()
            tl[name] = tl.get(name, 0.0) + 1e3 * (t1 - t_[0])
            t_[0] = t1
        # sqg_build_edges trims the chimeric blocks in place (LocateRead, :1229-1248): restore the four mutable arrays
        # -- a caller that runs the path once never pays for that, so every step gets its own pristine copy, made before the
        # timed region (chim_pool is refilled by timed() before each measurement)
        pool = state.setdefault("chim_pool", [])
        chim = pool.pop() if pool else api.ChimericReads(chim0.a)
        state["chim"] = chim
        lap("chim_input")
        if mode == "resident":
            g.attach_concordant_device(dstruct, keepalive=batch)
        elif mode == "wire":
            g.load_concordant_wire(wire)
        else:
            import ctypes as C0
            g._ck(g.L.sqg_load_concordant(g._h, C0.byref(hstruct), 0))
        lap("load_concordant")
        g.load_chimeric(chim)
        lap("load_chimeric")
        nodes = g.BuildNode_STAR()
        lap("BuildNode_STAR")
        edges = g.BuildEdges()
        lap("BuildEdges")
        # The host stages between BuildEdges and ExactBPConcordantSupport (filters, ordering, ExactBreakpoint) are out of scope;
        # their stand-in only has to produce the sorted breakpoint list, which is the same every step: computed in the warm-up
        # steps, reused (and its cost reported separately) in the timed ones.
        if "bps" not in state or not state.get("timed"):
            t_b = time.perf_counter()
            state["bps"] = bps_from_graph(nodes, edges)
            state["bps_standin_ms"] = 1e3 * (time.perf_counter() - t_b)
        bc, bp = state["bps"]
        lap("breakpoints (cached host stand-in)")
        cov = g.BPCoverage(bc, bp)
        lap("BPCoverage")
        state["stats"] = {k: g.stat(k) for k in ("groups", "islands", "heavy_islands", "giant_islands", "gap_records", "partial_records", "displaced_records", "lmax", "sensitive_reads", "raw_edges", "cov_chain_fallback", "cov_chain_chunks", "edges_single_path", "edges_generic_path", "slow_records", "qualifying_records", "seed_window_records", "short_other_blocks", "unstable_depth_blocks", "device_sort_status")}
        state["last"] = (nodes, edges, cov)
        state.update(n_nodes=int(nodes.Chr.shape[0]), n_edges=int(edges.Ind1.shape[0]), n_bp=int(bc.shape[0]), cov_sum=int(cov.sum()),
                     d2h=int(nodes.Chr.nbytes * 3 + nodes.count3.nbytes * 2 + edges.Ind1.nbytes * 3 + edges.Ind1.shape[0] + cov.nbytes))
        return nodes, edges, cov

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(mode: str, steps: int, warmup: int):
        sampler = ClockSampler(local)
        sampler.start()
        for _ in range(warmup):
            step(mode)
        state["chim_pool"] = [api.ChimericReads(chim0.a) for _ in range(steps)]  # pristine inputs of the timed steps
        barrier()
        state["timeline"] = {}
        state["timed"] = True
        l0 = g.launch_count()
        sampler.mark_begin()
        t = time.perf_counter()
        phases = {}
        for _ in range(steps):
            step(mode)
            for ph in ("h2d", "prepass", "classify", "seed", "tile", "depth_edges", "edge_sort", "coverage", "k_classify", "k_seed_islands", "k_assign", "k_assign_depth", "k_assign_edges", "k_edges_generic", "k_cov_compact", "k_cov_count"):
                v = g.phase_ms(ph)
                if v >= 0:
                    phases[ph] = phases.get(ph, 0.0) + v / steps
        barrier()
        sec = (time.perf_counter() - t) / steps
        sampler.mark_end()
        clocks = sampler.stop()
        if world > 1:
            tt = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sec = float(tt.item())
        state["timeline_ms"] = {k: v / steps for k, v in state["timeline"].items()}
        state["timed"] = False
        if rank == 0:
            nodes_l, edges_l, cov_l = state["last"]
            state.setdefault("crcs", {})[mode] = output_crcs(nodes_l, edges_l, state["chim"].block_table(), cov_l)
        return sec, phases, clocks, (g.launch_count() - l0) // steps

    sec, phases, clocks, launches = timed("resident", args.steps, args.warmup)
    timeline = dict(state["timeline_ms"])
    if args.dump_outputs and rank == 0:
        nodes_l, edges_l, cov_l = state["last"]
        dump_outputs(args.dump_outputs, nodes_l, edges_l, state["chim"].block_table(), cov_l)
    if world > 1:
        print("[rank %d] resident step %.1f ms; host timeline %s" % (rank, 1e3 * sec, {k: round(v, 1) for k, v in timeline.items()}), file=sys.stderr, flush=True)
    # end to end from host memory: the wire form (13 + 8 B, what a front end hands over; packed once, outside the timed region, its
    # cost reported as pack_wire_s) is the headline; the resident 32 + 12 B layout shipped as it is stays as `e2e_soa`
    sec_e2e, phases_e2e, _, _ = timed("wire", max(1, min(args.steps, 5)), 2)
    sec_soa, phases_soa = None, None
    if want_soa:
        sec_soa, phases_soa, _, _ = timed("soa", max(1, min(args.steps, 2)), 1)

    # ---- N > 1: the same stream as the single-GPU run, range-sharded over the N GPUs (strong scaling, north_star's split) ----
    one_stream = None
    if world > 1:
        if rank != 0:
            del batch
            torch.cuda.empty_cache()
        case0, chim00 = (case, chim0) if (rank == 0 or seed_r == seed0) else stream_case(P_req, seed0)  # every rank holds ALL chimeric reads of the one stream
        one_stream = one_stream_leg(args, rank, world, local, dev, batch if rank == 0 else None, chim00, case0, max(1, min(args.steps, 5)), 2)

    # ---- roofline ------------------------------------------------------------------------------------------------------
    # Every timed kernel with its algorithmic bytes per launch (SURVEY.md §8d / DESIGN.md §3): the stream kernels read the whole
    # batch (32 B per record + 12 B per aligned block); phase 3's pairs leave the classification kernel per tile (12 B written per
    # qualifying record on top of its read of the batch) and are gathered (12 B
    # read + 12 B written per qualifying record), then counted (12 B per qualifying record); the generic
    # edge kernel the records it is handed (32 B + 12 B per block of each).  The seed machine's input is the window of concordant
    # records in front of each discordant group (7 B each: pos, first-block length, class), counted by the kernel itself; it
    # walks them with dependent loads (break by break), so its fraction says "latency-bound", not "wasteful".
    K = NB / R
    st_ = state.get("stats", {})
    n_slow = max(0, st_.get("slow_records", 0)); nq = max(0, st_.get("qualifying_records", 0))
    alg = {"k_classify": 32 * R + 12 * NB + 12 * nq, "k_assign_depth": 32 * R + 12 * NB, "k_assign_edges": 32 * R + 12 * NB, "k_cov_compact": 24 * nq,
           "k_edges_generic": int(n_slow * (32 + 12 * max(2.0, K))), "k_cov_count": 12 * nq, "k_seed_islands": 7 * max(0, st_.get("seed_window_records", 0))}
    # DRAM bytes per record of each kernel from this round's `ncu --set full` capture (profiles/r2_traffic.json, written by
    # tests/tools/ncu_summary.py from the committed capture; dram__bytes_read.sum + dram__bytes_write.sum over the records of that run)
    traffic_pr = {}
    try:
        traffic_pr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["dram_bytes_per_record"]
    except Exception:
        pass
    peak, peak_src = measured_peak_gbs()
    timed = {k: v for k, v in phases.items() if k in alg}
    top = max(timed, key=timed.get) if timed else None
    per_kernel = {}
    for k, v in timed.items():
        gb = alg[k] / (v * 1e-3) / 1e9 if alg[k] else None
        per_kernel[k] = {"ms": v, "alg_bytes": alg[k], "GBps": gb, "frac": gb / peak if gb else None,
                         "dram_traffic_bytes": traffic_pr[k] * R if k in traffic_pr else None}
    b_alg_pair = (2 * (32 * R + 12 * NB) + 24 * R) / P
    # phases are disjoint intervals of the main stream; the coverage compaction runs beside the island machine on its own stream
    total_gpu_ms = sum(v for k, v in phases.items() if not k.startswith("k_") and k not in ("prepass", "h2d"))
    whole = (b_alg_pair * P / sec) / 1e9
    roof = None
    if top:
        pk = per_kernel[top]
        roof = {"bound": "hbm", "kernel": top, "achieved": pk["GBps"], "peak": peak, "unit": "GB/s", "frac": pk["frac"], "traffic": pk["dram_traffic_bytes"],
                "peak_source": peak_src, "alg_bytes_per_launch": pk["alg_bytes"], "ms": pk["ms"],
                "note": "the kernel with the longest live CUDA-event time in the step (all timed kernels are in `kernels`); traffic = DRAM bytes per record of this round's ncu capture x records of this run",
                "whole_path": {"alg_bytes_per_pair": b_alg_pair, "achieved": whole, "frac": whole / peak, "ms_per_step": 1e3 * sec,
                               "what": "B_alg = 2 (32 R + 12 B) + 24 R over the whole step, wall clock (SURVEY.md 8d)"},
                "kernels": per_kernel}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_leg(local)
    # ---- parity at full size: the outputs of the last timed step against the reference's, pinned once for this exact workload
    #      (tests/tools/pin_bench_crc.py: the reference's own sources ran on these records; tests/golden/bench_crc.json)
    parity = None
    if rank == 0:
        crcs = state.get("crcs", {})
        got = crcs.get("resident")
        pin = pinned_crcs(P_req, seed0)
        if pin is None:
            parity = {"checked": False, "why": "this workload has not been pinned (tests/tools/pin_bench_crc.py)", "crc32": got}
        else:
            bad = [(k if m == "resident" else m + ":" + k) for m, c in crcs.items() for k, v in pin["reference_crc32"].items() if c.get(k) != v]
            parity = {"checked": True, "ok": not bad, "against": "reference build (oracle/_ref) on the same %d records; coverage: CPU restatement" % pin["records"], "mismatch": bad,
                      "input_paths_checked": sorted(crcs)}
            if bad:
                print(json.dumps({"error": "outputs differ from the pinned reference CRCs", "mismatch": bad, "got": got, "want": pin["reference_crc32"]}), file=sys.stderr, flush=True)
    if rank == 0:
        out = {
            "metric": "read pairs/s through segment-graph build", "value": world * P / sec, "unit": "read pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": {"workload": "synthetic GRCh38-layout sorted alignment records, %d read pairs per GPU, ~0.5%% discordant (configs[1])" % P,
                       "pairs_per_gpu": P, "pairs_requested": P_req, "records": R, "blocks_per_record": K, "chimeric_reads": int(chim0.n_reads), "parallelism": ("one GPU" if world == 1 else "weak scaling: one independent stream per GPU x%d -- every rank generates and processes its own copy of the same 100 M-pair stream, so the work per GPU is fixed --, no data-path collective (independent samples have nothing to exchange); `one_stream` = rank 0's stream in %d exact genomic-range shards with the NCCL exchanges of the sharded protocol (strong scaling)" % (world, world)),
                       "block_mix": "SURVEY App. C: K = %.3f aligned blocks per record (exon lengths %d-%d)" % (K, BENCH_EXON_LEN[0], BENCH_EXON_LEN[1]),
                       "l2": "inputs (%.1f GB) larger than L2" % (n_bytes / 1e9), "segments": state.get("n_nodes"), "edges": state.get("n_edges"), "breakpoints": state.get("n_bp"),
                       "breakpoint_source": "host stand-in for the out-of-scope stages between BuildEdges and ExactBPConcordantSupport, computed in the warm-up steps"},
            "e2e": {"value": world * P / sec_e2e, "unit": "read pairs/s", "h2d_bytes_per_step": wire.nbytes + sum(v.nbytes for v in chim0.a.values()), "d2h_bytes_per_step": state.get("d2h", 0), "ms_per_step": 1e3 * sec_e2e, "host_memory": host_kind,
                    "input": "sqg_wire (include/squid_b200.h): delta-coded records, 13 B + 8 B per explicit block (%d of %d blocks are implied by their record: plain unclipped reads), %d record and %d block exceptions; uploaded in chunks, widened on the device while the next chunks are on the bus" % (wire.struct.n_blk - wire.struct.n_wblk, wire.struct.n_blk, wire.struct.n_rec_exc, wire.struct.n_blk_exc),
                    "pack_wire_s_outside_timed_region": t_pack, "pack_threads": os.cpu_count()},
            "e2e_soa": ({"value": world * P / sec_soa, "unit": "read pairs/s", "h2d_bytes_per_step": n_bytes + sum(v.nbytes for v in chim0.a.values()), "ms_per_step": 1e3 * sec_soa,
                         "input": "sqg_batch (the resident 32 B + 12 B layout) copied as it is", "phases_ms": phases_soa} if sec_soa else None),
            "roofline": roof,
            "whole_path": {"alg_bytes_per_pair": b_alg_pair, "gpu_ms_in_phases": total_gpu_ms,
                           "frac_of_hbm_roofline_wall": (b_alg_pair * P / sec) / 1e9 / peak, "frac_of_hbm_roofline_phases": (b_alg_pair * P / (total_gpu_ms * 1e-3)) / 1e9 / peak if total_gpu_ms else None},
            "phases_ms": phases, "host_timeline_ms": timeline, "bps_standin_ms_outside_timed_region": state.get("bps_standin_ms"), "phases_ms_e2e": phases_e2e, "stats": state.get("stats"),
            "cpu_baseline": cpu, "clocks": clocks, "gpu_launches": int(launches), "gen_s": t_gen, "parity": parity,
        }
        if one_stream is not None:
            pin = pinned_crcs(P_req, seed0)
            if pin is not None and "crc32" in one_stream:
                bad = [k for k, v in pin["reference_crc32"].items() if one_stream["crc32"].get(k) != v]
                one_stream["parity"] = {"checked": True, "ok": not bad, "mismatch": bad, "against": "the pinned reference CRCs of the single-GPU workload"}
                if bad:
                    parity = dict(parity or {}, checked=True, ok=False, mismatch=(parity or {}).get("mismatch", []) + ["one_stream:" + k for k in bad])
                    out["parity"] = parity
            out["one_stream"] = one_stream
        if real_stdout is not None:
            sys.stdout.flush()
            os.dup2(real_stdout, 1)
        print(json.dumps(out), flush=True)
    g.close()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and parity and parity.get("checked") and not parity.get("ok"):
        raise SystemExit(3)  # a fast step with the wrong answer is not a result


if __name__ == "__main__":
    main()
