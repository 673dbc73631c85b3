"""One fuzz seed of tests/tools/fuzz_sharded.py, single context against the reference build (which outputs differ, where)."""
import os
import random
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyref  # noqa: E402
from squid_b200 import api, synth  # noqa: E402
from tests import common  # noqa: E402

seed = int(sys.argv[1])
rnd = random.Random(seed * 104729)
n = rnd.choice([5000, 20000, 60000, 150000])
d = rnd.choice([0.005, 0.02, 0.05, 0.1])
ref = rnd.choice([synth.CHR17_LEN, [30000000, 20000000, 5000000, 16569], synth.GRCH38_LEN, [3000000, 2000000, 500000, 16569]])
kw = {"n_genes": rnd.choice([None, 30, 300, 2000]), "fusion_support": rnd.choice([5, 10, 20, 100])}
if rnd.random() < 0.25:
    kw.update(exon_len=(20, 170), intron_len=(60, 400))
print("case", n, d, ref, kw)
with tempfile.TemporaryDirectory() as td:
    cp, hp, *_ = common.write_case(td, n, seed, d, ref, **kw)
    refd = pyref.run(cp, hp, os.path.join(td, "ref"))
    for rep in range(3):
        got = common.run_cuda(cp, hp)
        g = got["graph"]
        bad = []
        for k in ("nodes", "avgdepth", "edges", "chim_after_edges"):
            a, b = refd[k], got[k]
            if a.shape != b.shape:
                bad.append("%s shape %s vs %s" % (k, a.shape, b.shape))
            elif not np.array_equal(a, b):
                rows = np.flatnonzero((a != b).reshape(a.shape[0], -1).any(axis=1))
                bad.append("%s %d rows, first %s ref %s got %s" % (k, rows.size, rows[:2], a[rows[:2]].tolist(), b[rows[:2]].tolist()))
        print("rep", rep, "device_sort_status", g.stat("device_sort_status"), "sensitive", g.stat("sensitive_reads"), "OK" if not bad else bad, flush=True)
