"""Times phase 2 of the bench workload (`depth_edges` and its kernels k_assign_tiles<depth>, k_assign_tiles<edges> and
k_edges_generic) with several builds of the library in one process, in alternating order, and checks that they compute
the same segments, edges and trimmed chimeric blocks.  Written to compare position indexes of the segment table; it takes
any builds, e.g. this tree's library against one built from an earlier commit.

    python tests/tools/seg_index_time.py --lib new=squid_b200/libsquid_b200.so --lib old=/path/to/libsquid_b200.so \
        [--pairs N] [--rounds R] [--out FILE]

Prints (and writes to FILE) one JSON object: the GPU and its power limit, and per build the phase times of every round
(live CUDA-event times of the library, ms) with their medians.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

PHASES = ("depth_edges", "k_assign_depth", "k_assign_edges", "k_edges_generic", "classify", "seed", "coverage")


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, metavar="NAME=PATH", help="a build of libsquid_b200.so (repeatable)")
    ap.add_argument("--pairs", type=int, default=100_000_000)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=100)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    import bench
    from squid_b200 import api, sqmb, synth, synth_gpu

    if not torch.cuda.is_available():
        raise SystemExit("seg_index_time.py needs a CUDA device")
    libs = [tuple(x.split("=", 1)) for x in args.lib]
    batch, tx, prob = bench.make_workload(args.pairs, args.seed, "cuda:0")
    chim_tab, _ = synth.make_chimeric(tx, prob, args.pairs, args.seed, bench.DISC_FRAC, adversarial=False)
    with tempfile.TemporaryDirectory() as d:
        sqmb.write_sqmb(d + "/chim.sqmb", chim_tab)
        sqmb.write_sqmb(d + "/conc.sqmb", sqmb.empty(synth.GRCH38_LEN, 0))
        case = api.HostCase(d + "/conc.sqmb", d + "/chim.sqmb")
    chim0 = case.chimeric
    dstruct = synth_gpu.batch_struct(batch)
    torch.cuda.synchronize()

    graphs = {}
    for name, path in libs:  # every SegmentGraph keeps the library it was created with
        api._lib = None
        api.LIB_PATH = os.path.abspath(path)
        graphs[name] = api.SegmentGraph(case.config, case.ref_len, device=0)

    def step(g):
        chim = api.ChimericReads(chim0.a)
        torch.cuda.synchronize()
        t = time.perf_counter()
        g.attach_concordant_device(dstruct, keepalive=batch)
        g.load_chimeric(chim)
        nodes = g.BuildNode_STAR()
        edges = g.BuildEdges()
        torch.cuda.synchronize()
        wall = 1e3 * (time.perf_counter() - t)
        ph = {p: g.phase_ms(p) for p in PHASES}
        ph["build_wall"] = wall
        return ph, bench.output_crcs(nodes, edges, chim.block_table(), np.zeros(0, np.int32))

    for name, _ in libs:
        for _ in range(args.warmup):
            step(graphs[name])
    times = {name: [] for name, _ in libs}
    crcs = {}
    for r in range(args.rounds):
        order = libs if r % 2 == 0 else libs[::-1]
        for name, _ in order:
            ph, crc = step(graphs[name])
            times[name].append(ph)
            crcs.setdefault(name, crc)
            if crc != crcs[name]:
                raise SystemExit("%s: outputs changed between rounds" % name)
    ref = crcs[libs[0][0]]
    res = {"gpu": gpu_info(), "pairs": int(batch["ref_id"].shape[0]) // 2, "rounds": args.rounds, "same_outputs": all(c == ref for c in crcs.values()),
           "crcs": crcs, "median_ms": {n: {p: round(statistics.median(t[p] for t in ts), 3) for p in ts[0]} for n, ts in times.items()},
           "rounds_ms": {n: [{p: round(v, 3) for p, v in t.items()} for t in ts] for n, ts in times.items()}}
    for g in graphs.values():
        g.close()
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")
    if not res["same_outputs"]:
        raise SystemExit("the builds compute different outputs")


if __name__ == "__main__":
    main()
