"""The CIGAR and record rules (sq_cigar.cuh, sq_bam.cuh) on random CIGARs over all nine ops (bam_device_cases.random_cigar_table):
against the reference restatement through the chimeric loader, and through every front end of the concordant batch -- the SQMB
packer, the host BAM front end and the CPU stepping of the device decode -- under several -pt / -pm / -pl settings."""
import os

import numpy as np
import pytest

from oracle import pyref
from squid_b200 import api, bamio, sqmb
from tests import bam_device_cases as cases
from tests import test_cpu_bam_device as dev

SETTINGS = [dict(phred33=1, min_phred=4, max_lowphred_len=10), dict(phred33=1, min_phred=20, max_lowphred_len=3),
            dict(phred33=0, min_phred=10, max_lowphred_len=25), dict(phred33=1, min_phred=50, max_lowphred_len=10),
            dict(phred33=0, min_phred=70, max_lowphred_len=0)]


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    d = tmp_path_factory.mktemp("cigar_rules")
    t = cases.random_cigar_table(2024)
    sp, bp = str(d / "t.sqmb"), str(d / "t.bam")
    sqmb.write_sqmb(sp, t)
    bamio.write_bam(bp, t)
    return t, sp, bp


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return cases.build_emul_bam(tmp_path_factory.mktemp("emul_bam"))


def test_family_reaches_every_op(table):
    t, _, _ = table
    ops = set((t.cigar & 15).tolist())
    assert ops == set(range(9)) and t.n >= 2000 and (t.seq_off < 0).any() and (t.seq_off >= 0).any()


@pytest.mark.parametrize("opts", SETTINGS)
def test_chimeric_loader_matches_restatement(table, tmp_path, built_lib, opts):
    """Blocks, TotalLen and the low-quality flags of every read, as the restatement (which shares no code with the library) loads them."""
    _, sp, _ = table
    hc = api.HostCase(sp, sp, **opts)
    ref = pyref.run_restate(sp, sp, str(tmp_path / "ref"), opts=pyref.restate_opts(["-pt", opts["phred33"], "-pm", opts["min_phred"], "-pl", opts["max_lowphred_len"]]),
                            stop_after=1)
    assert np.array_equal(hc.chimeric.block_table(), ref["chim_loaded"])
    meta = ref["chim_loaded_meta"]
    assert np.array_equal(hc.chimeric.a["first_total_len"], meta[:, 0]) and np.array_equal(hc.chimeric.a["second_total_len"], meta[:, 1])
    for col, key in ((2, "first_lowphred"), (3, "second_lowphred")):
        known = meta[:, col] >= 0  # the reference leaves *LowPhred of an unseen mate uninitialised
        assert np.array_equal(hc.chimeric.a[key][known], meta[known, col])


@pytest.mark.parametrize("opts", SETTINGS)
@pytest.mark.parametrize("layout", ["htslib", "straddle_997"])
def test_bam_front_ends_match_sqmb_packer(table, tmp_path, built_lib, emul, layout, opts):
    """The SQMB packer, the host BAM front end and the stepped device decode (20 kB windows) give one batch."""
    t, sp, bp = table
    cb = str(tmp_path / "conc.bam")
    open(cb, "wb").write(cases.layouts(t)[layout])
    want = api.HostCase(sp, sp, **opts).batch
    host = api.HostCase(cb, bp, bam=True, **opts).batch
    for k in api.BATCH_DTYPES:
        assert np.array_equal(want.a[k], host.a[k]), k
    info, got = dev._decode(emul, cb, api.HostCase(cb, bp, bam=True, header_only=True, **opts), str(tmp_path), 20000)
    assert got is not None, info
    dev._assert_batch(want, got)
    assert info["windows"] >= 2
