"""The shard planner of the resident batch (sq_plan.cuh: the per-record candidate rule and the greedy over the candidates) stepped
on the CPU by tests/emul/emul_plan.cpp, against the host planner (sqg_plan_shards, host/plan.cpp) on the same stream, for 1 to 8
shards: the case shapes of the sharded GPU tests, the golden cases, an unmapped tail, a stream without a clean cut, dense
discordant groups and runs of filtered or duplicate records longer than the planner's look-back window."""
import numpy as np
import pytest

from tests import plan_cases as pc


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return pc.build_emul_plan(tmp_path_factory.mktemp("emul_plan"))


def _same(emul, d, batch, case):
    want = pc.host_cuts(batch, case)
    got = pc.emul_cuts(emul, d, batch, case)
    assert got == want
    return want


@pytest.mark.parametrize("shape,opts", [(s, {}) for s in pc.SHAPES] + [("chr17", pc.OPTS)])
def test_case_shapes(shape, opts, emul, tmp_path, built_lib):
    from squid_b200 import api
    cp, hp, *_ = pc.write_shape(tmp_path, shape)
    case = api.HostCase(cp, hp, **opts)
    cuts = _same(emul, tmp_path / "emu", case.batch, case)
    assert max(len(c) for c in cuts.values()) >= 4, "no shard count found two cuts: the case tests little"


@pytest.mark.parametrize("name", pc.golden_cases())
def test_golden_cases(name, emul, tmp_path, built_lib):
    import os
    from squid_b200 import api
    case = api.HostCase(os.path.join(pc.GOLD, name, "conc.sqmb"), os.path.join(pc.GOLD, name, "chim.sqmb"))
    _same(emul, tmp_path / "emu", case.batch, case)


def test_unmapped_tail(emul, tmp_path, built_lib):
    """A third of the stream is unmapped: the planner stops at its first record and the shards that would lie in it are not made."""
    from squid_b200 import api
    cp, hp, *_ = pc.write_shape(tmp_path, "fourchr")
    case = api.HostCase(cp, hp)
    b = pc.unmapped_tail(case.batch, 0.34)
    cuts = _same(emul, tmp_path / "emu", b, case)
    first_unmapped = int(np.argmax(b.a["ref_id"] < 0))
    assert len(cuts[8]) < 9 and all(c <= first_unmapped for c in cuts[8][:-1]) and len(cuts[2]) == 3


def test_no_clean_cut(emul, tmp_path, built_lib):
    from squid_b200 import api
    cp, hp, *_ = pc.common.write_case(str(tmp_path), 3000, 3, 0.05)
    case = api.HostCase(cp, hp)
    b = pc.no_gap_batch(case.batch)
    cuts = _same(emul, tmp_path / "emu", b, case)
    assert all(c == [0, b.n_rec] for c in cuts.values())


def test_dense_groups_decide(emul, tmp_path, built_lib):
    """Many discordant groups: condition C rejects coverage gaps that A, B and D accept, and the cuts move."""
    from squid_b200 import api
    cp, hp, *_ = pc.common.write_case(str(tmp_path), 8000, 303, 0.3, [3000000, 2000000], n_genes=40, fusion_support=8)
    case = api.HostCase(cp, hp)
    _same(emul, tmp_path / "emu", case.batch, case)
    without_c = pc.emul_cuts(emul, tmp_path / "emu_no_groups", case.batch, case, no_groups=True)
    assert without_c != pc.host_cuts(case.batch, case)


@pytest.mark.parametrize("mapq", [None, 0], ids=["duplicates", "filtered"])
def test_look_back_window_decides(mapq, emul, tmp_path, built_lib):
    """A run of records that are not kept, inserted right behind the last gate-passing record before a clean cut c: the cut moves with the
    run while the walk back from it stays inside plan.cpp's window, and is no cut at all once the run is as long as the window."""
    from squid_b200 import api
    cp, hp, *_ = pc.write_shape(tmp_path, "chr17")
    case = api.HostCase(cp, hp)
    c0 = pc.host_cuts(case.batch, case, 2)[2][1]
    a = case.batch.a
    gate = ((a["aux"] & 11) == 0) & (a["mapq"] >= case.config.Min_MapQual) & ((a["flag"] & 0x404) == 0) & (a["ref_id"] >= 0)
    k1 = int(np.flatnonzero(gate[:c0])[-1])  # the last gate-passing record before c0: copies of it right behind it are duplicates
    for run, moves in ((pc.LOOK_BACK - 2000, True), (pc.LOOK_BACK, False)):
        b = pc.with_records(case.batch, k1 + 1, k1, run, mapq)
        cuts = _same(emul, tmp_path / ("emu_%d" % run), b, case)
        assert ((c0 + run) in cuts[2]) == moves, (run, cuts[2])
