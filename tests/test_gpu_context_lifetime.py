"""What a device context and a device call leave behind: sqg_connected_components keeps no memory from call to call, a closed
SegmentGraph gives back every buffer it allocated, and a chimeric input without reads or without blocks runs the device pre-pass
and is refused without harm to the context."""
import os

import numpy as np
import pytest

from squid_b200 import api, sqmb, synth
from tests import common

pytestmark = pytest.mark.gpu

GROWTH_LIMIT = 64 << 20


def _device_bytes_used() -> int:
    """This process's device memory: its NVML entry where NVML lists it (other tenants share the GPU), else what the whole device
    has in use (PID namespaces can hide the process from NVML)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            pid, used = os.getpid(), None
            for i in range(pynvml.nvmlDeviceGetCount()):
                for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                    if p.pid == pid and p.usedGpuMemory is not None:
                        used = (used or 0) + int(p.usedGpuMemory)
            if used is not None:
                return used
        finally:
            pynvml.nvmlShutdown()
    except Exception:
        pass
    import torch
    free, total = torch.cuda.mem_get_info(0)
    return int(total - free)


def _growth(step, cycles=5) -> int:
    step()  # warm-up: module load, CUB and driver pools
    before = _device_bytes_used()
    for _ in range(cycles):
        step()
    return _device_bytes_used() - before


def test_connected_components_keeps_no_memory(built_lib):
    n, m = 4_000_000, 12_000_000
    rng = np.random.default_rng(41)
    a = rng.integers(0, n, m).astype(np.int32); b = rng.integers(0, n, m).astype(np.int32)
    growth = _growth(lambda: api.ConnectedComponent(n, a, b))
    print("connected components: growth over 5 calls %.1f MiB" % (growth / 2**20))
    assert growth < GROWTH_LIMIT, "5 calls kept %.1f MiB of device memory" % (growth / 2**20)


def test_closed_context_gives_memory_back(tmp_path, built_lib):
    cp, hp, *_ = common.write_case(str(tmp_path), 1_000_000, seed=59, disc_frac=0.02)
    case = api.HostCase(cp, hp)
    bps = common.chr_start_bps(case.ref_len)

    def cycle():
        g = api.SegmentGraph(case.config, case.ref_len, device=0)
        w = api.WireBatch(case.batch)
        g.load_concordant_wire(w)
        g.load_chimeric(api.ChimericReads(case.chimeric.a))  # (a copy: BuildEdges trims the block arrays in place)
        g.BuildNode_STAR()
        g.BuildEdges()
        g.BPCoverage(bps[:, 0], bps[:, 1])
        g.close()
        w.close()

    growth = _growth(cycle)
    print("closed contexts: growth over 5 cycles %.1f MiB" % (growth / 2**20))
    assert growth < GROWTH_LIMIT, "5 closed contexts kept %.1f MiB of device memory" % (growth / 2**20)


def _refused_after_device_prepass(g, chim, batch):
    """BuildNode_STAR on chimeric reads that push no discordant block: the pre-pass runs on the device and leaves no blocks and no
    groups, and the call is refused where the reference is undefined (SegmentGraph.cpp:757 on an empty vector)."""
    with pytest.raises(api.SquidB200Error) as e:
        g.BuildNode_STAR(chim, batch)
    assert e.value.code == -5 and "no discordant block" in str(e.value)
    assert g.stat("disc_blocks") == 0 and g.stat("groups") == 0
    assert g.stat("device_sort_status") == 0


def test_empty_chimeric_input_on_the_device(tmp_path, built_lib, ref_oracle):
    conc, chim, _ = synth.make_case(40000, ref_len=synth.CHR17_LEN, seed=61, disc_frac=0.02)
    cp, hp, full = str(tmp_path / "conc.sqmb"), str(tmp_path / "chim_empty.sqmb"), str(tmp_path / "chim.sqmb")
    sqmb.write_sqmb(cp, conc); sqmb.write_sqmb(hp, chim.take(np.zeros(0, np.int64))); sqmb.write_sqmb(full, chim)
    case, empty = api.HostCase(cp, full), api.HostCase(cp, hp)
    assert empty.chimeric.n_reads == 0
    g = api.SegmentGraph(case.config, case.ref_len, device=0)
    # no reads at all
    _refused_after_device_prepass(g, empty.chimeric, empty.batch)
    # reads without blocks: they push nothing in BuildNode_STAR part A
    rng = np.random.default_rng(62)
    r = 1000
    arrays = {k: np.zeros(r + 1 if k == "read_off" else 0 if k.startswith("blk_") else r, dt) for k, dt in api.CHIM_DTYPES.items()}
    arrays["first_total_len"][:] = rng.integers(50, 151, r); arrays["second_total_len"][:] = rng.integers(50, 151, r)
    arrays["first_lowphred"][:] = rng.integers(0, 2, r); arrays["second_lowphred"][:] = rng.integers(0, 2, r)
    arrays["multi_filter"][:] = rng.integers(0, 2, r)
    _refused_after_device_prepass(g, api.ChimericReads(arrays), empty.batch)
    # the context goes on with the reads of the case: the reference's results
    ref = ref_oracle.run(cp, full, str(tmp_path / "ref"))
    nodes = g.BuildNode_STAR(case.chimeric, case.batch)
    edges = g.BuildEdges()
    g.close()
    assert np.array_equal(np.stack([nodes.Chr, nodes.Position, nodes.Length, nodes.Support], axis=1), ref["nodes"])
    assert np.array_equal(nodes.AvgDepth, ref["avgdepth"])
    assert np.array_equal(edges.table(), ref["edges"])
