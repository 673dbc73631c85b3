"""From a concordant BAM file to one range shard ready on the device, per rank: the device path against the host path.

    python tests/tools/bam_sharded_time.py --pairs 10000000 --out profiles/bam_sharded_time.json

The stream is sorted and holds --pairs pairs: one synthetic case (synth.make_case, --base-pairs pairs on one chromosome) is
written once by bamio's per-record writer, then copy k of its records is placed on chromosome k of a header of as many
chromosomes (refID fields patched), and the whole is BGZF-compressed (zlib level 6, members every 0xFF00 bytes, all cores).
For N shards and every rank r < N, best of --reps, device synchronised:
  device: sqh_open_bam_chimeric + sqg_load_concordant_bam + sqg_load_chimeric + sqg_plan_shards_resident (classifies the whole
          stream first) + sqg_keep_records(cuts[r], cuts[r + 1])
  host:   sqh_open_bam_case (inflate + decode + pack on all cores) + sqg_plan_shards + sqg_load_concordant of the rank's slice
Every rank of a real run does this on its own GPU at the same time; here the ranks run one after the other on one GPU, so the
host path's numbers are those of a host whose cores serve one rank.  The kept batch is compared with the host slice.  Needs a
CUDA device; the card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import concurrent.futures
import json
import os
import struct
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from squid_b200 import api, bamio, synth  # noqa: E402
from tests import bam_device_cases as cases  # noqa: E402
from tests.tools.bam_device_time import gpu_info  # noqa: E402

CHR_LEN = 60_000_000


def header(n_chr: int) -> bytes:
    text = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:chr%d\tLN:%d\n" % (i, CHR_LEN) for i in range(n_chr))
    out = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", n_chr)
    for i in range(n_chr):
        nm = b"chr%d\0" % i
        out += struct.pack("<i", len(nm)) + nm + struct.pack("<i", CHR_LEN)
    return out


def on_chromosome(recs: list, k: int) -> bytes:
    """The records (all on chromosome 0 or unplaced) moved to chromosome k: refID and next_refID 0 -> k."""
    body = np.frombuffer(b"".join(recs), np.uint8).copy()
    starts = np.concatenate([[0], np.cumsum([len(r) for r in recs])[:-1]]).astype(np.int64)
    kb = np.frombuffer(struct.pack("<i", k), np.uint8)
    for field in (4, 24):
        at = starts + field
        val = body[at[:, None] + np.arange(4)].copy().view("<i4").ravel()
        sel = at[val == 0]
        body[sel[:, None] + np.arange(4)] = kb
    return body.tobytes()


def write_stream(d: str, base_pairs: int, copies: int):
    conc, chim, _ = synth.make_case(base_pairs, ref_len=[CHR_LEN], seed=11, disc_frac=0.02)
    hdr = header(copies)
    recs = bamio.bam_parts(conc)[1:]
    raw = hdr + b"".join(on_chromosome(recs, k) for k in range(copies))
    edges = list(range(0, len(raw), 0xFF00)) + [len(raw)]
    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 8) as ex:
        members = list(ex.map(lambda ab: cases.member(raw[ab[0]:ab[1]], 6), zip(edges[:-1], edges[1:])))
    cb, hb = os.path.join(d, "conc.bam"), os.path.join(d, "chim.bam")
    with open(cb, "wb") as f:
        for m in members:
            f.write(m)
        f.write(bamio._BGZF_EOF)
    craw = hdr + b"".join(bamio.bam_parts(chim)[1:])
    open(hb, "wb").write(bamio.bgzf_compress(craw, 0xFF00))
    return cb, hb, len(raw)


def device_rank(cb, hb, n_shards, rank, torch):
    t = {}
    t0 = time.perf_counter()
    case = api.HostCase(cb, hb, bam=True, header_only=True)
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant_bam(cb, case)
    g.load_chimeric(api.ChimericReads(case.chimeric.a))
    torch.cuda.synchronize(); t1 = time.perf_counter()
    cuts = g.plan_shards(n_shards)
    t2 = time.perf_counter()
    g.keep_records(cuts[rank], cuts[rank + 1])
    torch.cuda.synchronize(); t3 = time.perf_counter()
    t.update(total_s=t3 - t0, open_decode_s=t1 - t0, classify_plan_s=t2 - t1, keep_s=t3 - t2,
             plan_ms=g.phase_ms("plan"), classify_ms=g.phase_ms("classify"))
    return t, cuts, g, case


def host_rank(cb, hb, n_shards, rank, torch):
    t0 = time.perf_counter()
    case = api.HostCase(cb, hb, bam=True)
    t1 = time.perf_counter()
    cuts = api.plan_shards(case.batch, case.chimeric, case.config, len(case.ref_len), n_shards)
    t2 = time.perf_counter()
    g = api.SegmentGraph(case.config, case.ref_len)
    g.load_concordant(case.batch.slice(cuts[rank], cuts[rank + 1]))
    g.load_chimeric(api.ChimericReads(case.chimeric.a))
    torch.cuda.synchronize(); t3 = time.perf_counter()
    return dict(total_s=t3 - t0, open_decode_s=t1 - t0, plan_s=t2 - t1, upload_s=t3 - t2), cuts, g, case


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--base-pairs", type=int, default=250_000)
    ap.add_argument("--shards", default="1,2")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="bam_sharded_time.json")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    res = {"gpu": gpu_info(), "pairs": a.pairs, "base_pairs": a.base_pairs, "reps": a.reps, "runs": []}
    with tempfile.TemporaryDirectory() as d:
        copies = max(1, -(-a.pairs // a.base_pairs))
        t0 = time.perf_counter()
        cb, hb, inflated = write_stream(d, a.base_pairs, copies)
        res.update(copies=copies, inflated_bytes=inflated, compressed_bytes=os.path.getsize(cb), write_s=round(time.perf_counter() - t0, 1))
        for ns in [int(x) for x in a.shards.split(",")]:
            for rank in range(ns):
                dev, host = [], []
                for rep in range(a.reps):
                    td, dcuts, gd, dcase = device_rank(cb, hb, ns, rank, torch)
                    th, hcuts, gh, hcase = host_rank(cb, hb, ns, rank, torch)
                    dev.append(td); host.append(th)
                    if rep == a.reps - 1:
                        want = hcase.batch.slice(hcuts[rank], hcuts[rank + 1])
                        got = gd.download_concordant()
                        equal = dcuts == hcuts and all(np.array_equal(want.a[k], got.a[k]) for k in api.BATCH_DTYPES)
                    gd.close(); gh.close(); dcase.close(); hcase.close()
                best = lambda rows: min(rows, key=lambda r: r["total_s"])
                row = {"n_shards": ns, "rank": rank, "cuts": dcuts, "records": dcuts[-1], "shard_records": dcuts[rank + 1] - dcuts[rank],
                       "device": {k: round(v, 4) for k, v in best(dev).items()}, "host": {k: round(v, 4) for k, v in best(host).items()},
                       "device_total_all_s": [round(r["total_s"], 4) for r in dev], "host_total_all_s": [round(r["total_s"], 4) for r in host],
                       "same_cuts_and_records": bool(equal)}
                res["runs"].append(row)
                print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
