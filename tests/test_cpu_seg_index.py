"""The segment table's position index (sq_common.cuh: per-chromosome headers and 16-byte bin entries behind seg_at, and the
plain chr_first / bin_seg form the CPU stepping harness builds) against its definition: for tables that tile the genome in
every awkward way, every position of every chromosome and the positions just past both ends give the segment std::upper_bound
gives, with that segment's Position and End, at every bin width."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("seg_index") / "seg_index_check")
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-I", "include", "-I", "squid_b200/csrc", "-o", out, "tests/emul/seg_index_check.cpp"],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def tiling(ref_len, cuts, start=0):
    """Segments of one chromosome from `start` to ref_len, cut at the sorted positions `cuts` (inside (start, ref_len))."""
    b = [start] + sorted(set(int(x) for x in cuts if start < x < ref_len)) + [ref_len]
    return [(b[i], b[i + 1] - b[i]) for i in range(len(b) - 1)]


def family(name, seed):
    """(ref_len per chromosome, segments per chromosome as (pos, len) lists; an empty list: a chromosome without segments)"""
    rng = np.random.default_rng(seed)
    if name == "one_bp":  # 1-bp segments everywhere
        lens = [300, 1, 2, 700]
        return lens, [tiling(L, range(1, L)) for L in lens]
    if name == "dense_bin":  # hundreds of segments inside one 512-bp bin, long ones around them
        L = 5000
        cuts = list(range(1030, 1500, 2)) + list(rng.integers(1500, 1536, 20)) + [300, 2600, 4000]
        return [L, 900], [tiling(L, cuts), tiling(900, [450])]
    if name == "one_per_chr":
        lens = [int(x) for x in rng.integers(1, 3000, 6)]
        return lens, [[(0, L)] for L in lens]
    if name == "on_grid":  # every boundary on the grid of every bin width checked
        L = 8192
        return [L, 4096], [tiling(L, range(512, L, 512)), tiling(4096, range(16, 4096, 16))]
    if name == "short_chr":  # chromosomes shorter than one bin
        lens = [3, 17, 100, 511, 512, 513]
        return lens, [tiling(L, rng.integers(1, max(2, L), min(L, 5))) for L in lens]
    if name == "empty_chr":  # chromosomes without segments between and at both ends of the table
        lens = [600, 2000, 1500, 40, 900]
        segs = [[], tiling(2000, rng.integers(1, 2000, 30)), [], tiling(40, [7, 8]), []]
        return lens, segs
    if name == "late_start":  # a first segment that starts right of 0: positions before it clamp to it
        lens = [3000, 1200]
        return lens, [tiling(3000, rng.integers(600, 3000, 25), start=517), tiling(1200, [5, 6, 1100], start=3)]
    if name == "random":
        lens = [int(x) for x in rng.integers(1, 40000, 5)]
        segs = []
        for L in lens:
            k = int(rng.integers(0, min(L, 400)))
            dense = rng.integers(0, L, k // 2)
            burst = int(rng.integers(0, L))
            segs.append(tiling(L, list(dense) + list(range(burst, min(L, burst + k), int(rng.integers(1, 4))))))
        return lens, segs
    raise ValueError(name)


FAMILIES = ["one_bp", "dense_bin", "one_per_chr", "on_grid", "short_chr", "empty_chr", "late_start", "random"]


@pytest.mark.parametrize("form", ["packed", "plain"])
@pytest.mark.parametrize("bin_shift", [0, 1, 4, 9, 12])
@pytest.mark.parametrize("name,seed", [(f, 0) for f in FAMILIES] + [("random", s) for s in (1, 2, 3)])
def test_lookups_match_upper_bound(checker, name, seed, bin_shift, form, tmp_path):
    lens, segs = family(name, seed)
    rows = [(c, p, l) for c, ss in enumerate(segs) for p, l in ss]
    path = tmp_path / "table.bin"
    with open(path, "wb") as f:
        np.array([len(lens)] + lens, dtype=np.int32).tofile(f)
        np.array(rows, dtype=np.int32).reshape(-1, 3).tofile(f)
    r = subprocess.run([checker, str(path), str(bin_shift), form], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert int(r.stdout) == sum((ss[-1][0] + ss[-1][1] if ss else L) + 7 for L, ss in zip(lens, segs))
