"""One shard per torch.distributed rank / GPU over NCCL, from a concordant BAM decoded on the device: the seeded case of
tests/tools/dist_sharded.py written as BAM files, and every rank runs ShardedSegmentGraph.load_bam -- decodes the whole file on
its GPU, plans the cuts on the resident batch, checks with one all-gather that every rank planned the same cuts, keeps its own
record range.  No host batch is built.  Launch:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29613 tests/tools/dist_sharded_bam.py [n_pairs]
Every rank must end with the reference's segments, Support, AvgDepth, edges, trimmed chimeric blocks and breakpoint support.
Rank 0 prints one line with every rank's verdict."""
import os
import sys
import tempfile
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyref  # noqa: E402  (test infrastructure: the checker)
from squid_b200 import api, bamio, sharded, synth  # noqa: E402
from tests import common  # noqa: E402


def main():
    n_pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 400000
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    d = tempfile.mkdtemp(prefix="sq_dist_bam_%d_" % rank)
    cp, hp, conc, chim, _ = common.write_case(d, n_pairs, 1020, 0.05, synth.GRCH38_LEN, fusion_support=10)
    cb, hb = os.path.join(d, "conc.bam"), os.path.join(d, "chim.bam")
    bamio.write_bam(cb, conc); bamio.write_bam(hb, chim)
    case = api.HostCase(cb, hb, bam=True, header_only=True)
    sg = sharded.ShardedSegmentGraph(case.config, case.ref_len, world, [rank], comm=sharded.DistComm(), devices=[local])
    dist.barrier()
    t0 = time.perf_counter()
    cuts = sg.load_bam(cb, case)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    nodes = sg.BuildNode_STAR()
    edges = sg.BuildEdges()
    torch.cuda.synchronize(); dist.barrier()
    t2 = time.perf_counter()
    got = {"nodes": np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1).astype(np.int32), "avgdepth": nodes.AvgDepth,
           "edges": edges.table(), "chim_after_edges": sg.Chimrecord.block_table()}
    ref = None
    if rank == 0:
        pyref.build()
        oracle = pyref  # the reference build where it is present, else the CPU restatement (as the parity tests do)
        if not pyref.available():
            pyref.build_restate()
            oracle = pyref.Restated
        ref = oracle.run(cp, hp, os.path.join(d, "ref"))
    objs = [ref]
    dist.broadcast_object_list(objs, src=0)
    ref = objs[0]
    common.assert_same(ref, got)
    sup = api.SegmentGraph.ExactBPConcordantSupport(sg, ref["final_nodes"], ref["final_edges"], pyref.exactbp_map(ref))
    assert sup == pyref.support_map(ref)
    oks = [None] * world
    dist.all_gather_object(oks, "bit-exact")
    if rank == 0:
        print({"world": world, "records": cuts[-1], "cuts": cuts, "load_bam_s": round(t1 - t0, 4), "segments": int(nodes.Chr.shape[0]),
               "edges": int(edges.Weight.shape[0]), "verdicts": oks, "rounds": sg.rounds, "build_nodes_edges_s": round(t2 - t1, 4),
               "backend": dist.get_backend()}, flush=True)
    sg.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
