"""The device twin of the chimeric pre-pass sort (squid_b200/csrc/sq_gpusort.cuh) against std::sort on the host: the same
permutation, payload included, for keys with many ties (what decides which equal (RefID,RefPos) block the reference sees
first, SURVEY.md App. A-11), sorted, reversed and organ-pipe inputs, across the leaf / multi-level size boundaries."""
import ctypes as C

import pytest

pytestmark = pytest.mark.gpu


def _run(n, seed, rng, pattern):
    from squid_b200 import api
    L = api.lib()
    L.sqg_selftest_gpu_sort.argtypes = [C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_float)]
    ms = C.c_float(-1)
    return L.sqg_selftest_gpu_sort(0, n, seed, rng, pattern, C.byref(ms)), ms.value


@pytest.mark.parametrize("n", [2, 3, 16, 17, 100, 1024, 1025, 2049, 5000, 40000, 300000, 1200000])
def test_random_keys_with_ties(built_lib, n):
    for seed, rng in ((1, 0), (2, 3), (3, 50), (4, max(2, n // 7)), (5, 1 << 40)):  # range 0: every key equal
        v, ms = _run(n, seed, rng, 0)
        assert v == 1, "n=%d range=%d: verdict %d" % (n, rng, v)


@pytest.mark.parametrize("pattern", [1, 2, 3])
def test_structured_inputs(built_lib, pattern):
    for n in (1000, 1025, 70000, 900000):
        v, ms = _run(n, 7, 0, pattern)
        # organ-pipe inputs can exhaust std::sort's depth budget: the device then declines (2) and the CPU twin takes over
        assert v == 1 or (pattern == 3 and v == 2), "pattern %d n=%d: verdict %d" % (pattern, n, v)


def test_prepass_uses_the_device_sort(tmp_path, built_lib, ref_oracle):
    """End to end on a small input: the pre-pass sort runs on the device, same segments / edges as the reference build."""
    from tests import common
    cp, hp, *_ = common.write_case(str(tmp_path), 60000, 1031, 0.05, fusion_support=10)
    ref = ref_oracle.run(cp, hp, str(tmp_path / "ref"))
    got = common.run_cuda(cp, hp)
    assert got["graph"].stat("device_sort_status") == 0
    common.assert_same(ref, got)
