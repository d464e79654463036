"""CPU: the oracle restatement on REAL racon windows (tests/golden/lambda_windows.npz: the reference's own
lambda-phage test data through the unmodified racon CPU pipeline) and on cudapoa's 67 deep sample windows."""
import numpy as np
import pytest

from common import contig_edit_distance, cudapoa_fixture, identity_order, lambda_fixture, lambda_reference
from oracle_lib import processing_order


@pytest.mark.parametrize("case,golden", [("fastq_500", 1312), ("fasta_500", 1566), ("fastq_1000", 1289)])
def test_oracle_reproduces_racon_on_real_windows(oracle, ref, case, golden):
    """Every window's consensus and status equal racon's CPU path; the stitched contig reproduces the
    reference's golden edit distance (test/racon_test.cpp:106-107, 128-129, 194-195)."""
    b, cons, polished, p = lambda_fixture(case)
    assert p["edit_distance"] == golden
    from racon_gpu_b200 import api
    order = api.processing_order(b)
    assert (order == processing_order(b, ref.layer_order)).all()  # the product's layer order is racon's std::sort call
    oc, _, opol = oracle.polish(b, order, p["m"], p["x"], p["g"], tgs=p["tgs"], trim=p["trim"], threads=8, stride=8192)
    assert oc == cons
    assert (opol == polished).all()
    assert contig_edit_distance(oracle, oc, lambda_reference()) == golden
    # real windows are what the synthetic ones are not: partial spans, qualities, uneven depth
    nseq = np.diff(b.win_seq_off)
    L = np.diff(b.seq_off)[b.win_seq_off[:-1]]
    part = ((b.begins > 0.01 * np.repeat(L, nseq)) | (b.ends < np.repeat(L, nseq) * 0.99 - 1))
    part[b.win_seq_off[:-1]] = False
    assert part.sum() > 50 and nseq.max() > 2 * np.median(nseq) * 0.6


def test_oracle_on_cudapoa_sample_windows(oracle):
    """67 windows, depth 105-170: consensus and coverage of the unmodified reference (spoa as window.cpp calls it)."""
    b, cons, cov = cudapoa_fixture()
    assert b.n_windows == 67 and np.diff(b.win_seq_off).max() >= 160
    oc, ocov, _ = oracle.polish(b, identity_order(b), 3, -5, -4, tgs=False, trim=False, threads=8, stride=8192)
    assert oc == cons
    assert all((a == c).all() for a, c in zip(ocov, cov))


@pytest.mark.parametrize("case", ["fastq_500", "fasta_500"])
def test_engine_emulation_on_real_windows(oracle, case):
    """The engine's own graph phases (host lane-emulation build) on real windows: full band bit-exact (consensus and
    coverage), static band 256 within the stated tolerance (>= 99 % identical, edit distance <= 2)."""
    from emu_lib import Emu
    from racon_gpu_b200 import api
    from racon_gpu_b200.windows import edit_distance
    b, _, _, p = lambda_fixture(case)
    order = api.processing_order(b)
    oc, ocov, _ = oracle.polish(b, order, p["m"], p["x"], p["g"], tgs=False, trim=False, threads=8, stride=8192)
    ec, ecov, est, _ = Emu().polish(b, order, p["m"], p["x"], p["g"], max_nodes=3072, max_edges=6 * 3072, stride=8192)
    assert (est == 0).all() and ec == oc
    assert all((a == c).all() for a, c in zip(ecov, ocov))
    bc, _, bst, _ = Emu().polish(b, order, p["m"], p["x"], p["g"], max_nodes=4092, max_edges=6 * 4092, band=256, stride=8192)
    d = [edit_distance(a, c) for a, c in zip(bc, oc)]
    assert (bst == 0).all() and sum(x == 0 for x in d) >= 0.99 * len(d) and max(d) <= 2
