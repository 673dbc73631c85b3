"""Host BAM front end + upload against the device BAM decode, on one concordant stream of >= 10 M pairs written in two layouts.

    python tests/tools/bam_device_time.py --pairs 10000000 --out profiles/bam_device_time.json

The stream is one synthetic case (synth.make_case, --base-pairs pairs) whose records are repeated behind one header until it holds
--pairs pairs: bamio's per-record writer runs once on the base case, the repetition and the BGZF compression (zlib level 6, all
cores) are bulk operations.  Layouts: "htslib" (members end at record boundaries, at most 0xFF00 bytes) and "straddle" (members
cut every 0xFF00 bytes wherever that falls).  Per layout, best of --reps:
  host:   sqh_open_bam_case (inflate + boundaries + decode + pack on all cores) + sqg_load_concordant, device synchronised
  device: sqh_open_bam_chimeric (chimeric file + concordant header) + sqg_load_concordant_bam, device synchronised
plus the device phases of the last device run, the inflated GB/s of its inflate phase, and whether the two batches are equal.
Needs a CUDA device; the card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from squid_b200 import api, bamio, synth  # noqa: E402
from tests import bam_device_cases as cases  # noqa: E402


def write_layouts(conc, copies: int, d: str, level: int = 6) -> dict:
    parts = bamio.bam_parts(conc)
    hdr, recs = parts[0], parts[1:]
    body = b"".join(recs)
    lens = np.array([len(r) for r in recs], np.int64)
    raw = hdr + body * copies
    # htslib: the header alone, then greedy members of whole records (a record is never split: all are far below 0xFF00 bytes)
    rec_lens = np.tile(lens, copies)
    cuts_h = [len(hdr)]
    start = len(hdr)
    ends = len(hdr) + np.cumsum(rec_lens)
    i = 0
    n = rec_lens.shape[0]
    while i < n:  # jump with searchsorted: the last record end that fits into the member
        j = int(np.searchsorted(ends, start + 0xFF00, side="right")) - 1
        j = max(j, i)
        start = int(ends[j]); cuts_h.append(start); i = j + 1
    edges = {"htslib": [0] + cuts_h, "straddle": list(range(0, len(raw), 0xFF00)) + [len(raw)]}
    out = {}
    workers = os.cpu_count() or 8
    for name, e in edges.items():
        e = sorted(set(e))
        with concurrent.futures.ThreadPoolExecutor(workers) as ex:
            members = list(ex.map(lambda ab: cases.member(raw[ab[0]:ab[1]], level), zip(e[:-1], e[1:])))
        p = os.path.join(d, "conc_%s.bam" % name)
        with open(p, "wb") as f:
            for m in members:
                f.write(m)
            f.write(bamio._BGZF_EOF)
        out[name] = p
    return out, len(raw)


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--base-pairs", type=int, default=250_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="bam_device_time.json")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    res = {"gpu": gpu_info(), "pairs": a.pairs, "base_pairs": a.base_pairs, "reps": a.reps, "layouts": {}}
    with tempfile.TemporaryDirectory() as d:
        conc, chim, _ = synth.make_case(a.base_pairs, ref_len=synth.CHR17_LEN, seed=11, disc_frac=0.02)
        copies = max(1, -(-a.pairs // a.base_pairs))
        t0 = time.perf_counter()
        paths, inflated = write_layouts(conc, copies, d)
        hb = os.path.join(d, "chim.bam")
        bamio.write_bam(hb, chim)
        res.update(copies=copies, inflated_bytes=inflated, write_s=round(time.perf_counter() - t0, 1))
        for name, cb in paths.items():
            row = {"compressed_bytes": os.path.getsize(cb)}
            host_s, dev_s = [], []
            host_batch = None
            for rep in range(a.reps):
                t = time.perf_counter()
                case = api.HostCase(cb, hb, bam=True)
                g = api.SegmentGraph(case.config, case.ref_len)
                g.load_concordant(case.batch)
                torch.cuda.synchronize()
                host_s.append(time.perf_counter() - t)
                if rep == a.reps - 1:
                    host_batch = case
                else:
                    case.close()
                g.close()
                t = time.perf_counter()
                dcase = api.HostCase(cb, hb, bam=True, header_only=True)
                gd = api.SegmentGraph(dcase.config, dcase.ref_len)
                gd.load_concordant_bam(cb, dcase)
                torch.cuda.synchronize()
                dev_s.append(time.perf_counter() - t)
                if rep < a.reps - 1:
                    gd.close(); dcase.close()
            phases = {p: round(gd.phase_ms(p), 3) for p in ("bam_h2d", "bam_inflate", "bam_records", "bam_decode")}
            got = gd.download_concordant()
            equal = all(np.array_equal(host_batch.batch.a[k], got.a[k]) for k in api.BATCH_DTYPES)
            row.update(n_rec=int(got.n_rec), host_open_upload_s=round(min(host_s), 4), device_open_load_s=round(min(dev_s), 4),
                       host_all_s=[round(x, 4) for x in host_s], device_all_s=[round(x, 4) for x in dev_s], device_phases_ms=phases,
                       inflate_GBps=round(inflated / (phases["bam_inflate"] * 1e-3) / 1e9, 2) if phases["bam_inflate"] > 0 else None,
                       members=gd.stat("bam_members"), windows=gd.stat("bam_windows"), repair_rounds=gd.stat("bam_repair_rounds"), batch_equal=bool(equal))
            res["layouts"][name] = row
            print(json.dumps({name: row}), flush=True)
            gd.close(); host_batch.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
