"""Streams for the shard planner on the resident batch (sqg_plan_shards_resident): the cases tests/test_cpu_plan_resident.py steps
on the CPU and tests/test_gpu_plan_resident.py runs on the device, each compared with the host planner (sqg_plan_shards)."""
import os
import subprocess

import numpy as np

from squid_b200 import api, synth
from tests import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
LOOK_BACK = 1 << 20  # host/plan.cpp: records the walk back from a cut looks at

# the four case shapes of tests/test_gpu_sharded.py at a quarter of their size or less: n_pairs, seed, disc_frac, ref_len, kwargs
SHAPES = {
    "chr17": (5000, 17, 0.02, None, {}),
    "fourchr": (8000, 31, 0.005, [3000000, 2000000, 500000, 16569], {"n_genes": 20}),
    "grch38": (20000, 1003, 0.02, "grch38", {}),
    "grch38_fusions": (20000, 2024, 0.05, "grch38", {"fusion_support": 10}),
}
# non-default -mq / -pl / -pm (HostCase options) and the reference's flags for them
OPTS = dict(min_mapq=3, max_lowphred_len=25, min_phred=10)
OPTS_ARGS = ["-mq", "3", "-pl", "25", "-pm", "10"]


def write_shape(d, name, **kw):
    n, seed, disc, rl, extra = SHAPES[name]
    return common.write_case(str(d), n, seed, disc, synth.GRCH38_LEN if rl == "grch38" else rl, **dict(extra, **kw))


def golden_cases():
    """The golden STAR cases (conc.sqmb + chim.sqmb)."""
    return sorted(c for c in os.listdir(GOLD) if os.path.exists(os.path.join(GOLD, c, "conc.sqmb")))


def with_records(batch: api.RecordBatch, at: int, src: int, count: int, mapq=None) -> api.RecordBatch:
    """`batch` with `count` copies of record `src` (its blocks included) inserted in front of record `at`; mapq=None keeps them
    exact duplicates (gated, not kept), else they carry that mapq (filtered).  src = at - 1 keeps the stream sorted."""
    a = batch.a
    off = a["blk_off"].astype(np.int64)
    rec = np.concatenate([np.arange(at), np.full(count, src), np.arange(at, batch.n_rec)])
    d = {}
    for k in api.BATCH_DTYPES:
        if k == "blk_off" or k.startswith("blk_"):
            continue
        d[k] = a[k][rec].copy()
    if mapq is not None:
        d["mapq"][at:at + count] = mapq
    nb = off[1:] - off[:-1]
    new_nb = nb[rec]
    d["blk_off"] = np.concatenate([[0], np.cumsum(new_nb)]).astype(np.uint32)
    blk = np.concatenate([np.arange(off[at]), np.tile(np.arange(off[src], off[src + 1]), count), np.arange(off[at], off[-1])]).astype(np.int64)
    for k in ("blk_ref_pos", "blk_match_ref", "blk_read_pos", "blk_match_read"):
        d[k] = a[k][blk].copy()
    return api.RecordBatch(d)


def no_gap_batch(batch: api.RecordBatch) -> api.RecordBatch:
    """Every alignment reaches past every later one: no record is at a coverage gap, so there is no clean cut."""
    b = batch.slice(0, batch.n_rec)
    b.a["end_pos"][:] = np.int32(2**30)
    return b


def unmapped_tail(batch: api.RecordBatch, frac: float) -> api.RecordBatch:
    """The last `frac` of the records turned into unmapped reads without a position (ref_id -1, flag 0x4), as a sorted BAM ends."""
    b = batch.slice(0, batch.n_rec)
    t = int(b.n_rec * (1 - frac))
    b.a["ref_id"][t:] = -1
    b.a["flag"][t:] |= np.uint16(4)
    return b


def host_cuts(batch, case, max_shards=8):
    return {ns: api.plan_shards(batch, case.chimeric, case.config, len(case.ref_len), ns) for ns in range(1, max_shards + 1)}


def build_emul_plan(out_dir) -> str:
    """Compiles tests/emul/emul_plan.cpp into `out_dir` (not into the repository tree, which may be read-only)."""
    os.makedirs(str(out_dir), exist_ok=True)
    out = os.path.join(str(out_dir), "emul_plan")
    srcs = ["tests/emul/emul_plan.cpp", "squid_b200/csrc/host/prepass.cpp"]
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-fopenmp", "-I", "include", "-I", "squid_b200/csrc", "-o", out] + srcs + ["-lpthread"],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def emul_cuts(emul, d, batch, case, max_shards=8, no_groups=False):
    """The planner rules of sq_plan.cuh stepped on the CPU over `batch` and the chimeric reads of `case` (no_groups: as if there
    were no discordant group, i.e. without condition C)."""
    os.makedirs(str(d), exist_ok=True)
    for k in api.BATCH_DTYPES:
        batch.a[k].tofile(os.path.join(str(d), "batch_%s.bin" % k))
    for k in api.CHIM_DTYPES:
        case.chimeric.a[k].tofile(os.path.join(str(d), "chim_%s.bin" % k))
    c = case.config
    np.array([c.Min_MapQual, c.Max_LowPhred_Len, c.Concord_Dist_Pos, c.Concord_Dist_Idx, c.ReadLen, len(case.ref_len)], np.int32).tofile(os.path.join(str(d), "config.bin"))
    env = dict(os.environ, SQ_EMUL_PLAN_NO_GROUPS="1") if no_groups else None
    r = subprocess.run([emul, str(d), str(max_shards)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    return {ns: [int(x) for x in lines[ns - 1].split()] for ns in range(1, max_shards + 1)}
