"""GPU (-m gpu): REAL racon windows through the C ABI against the consensus racon's CPU path computed for them
(tests/golden/lambda_windows.npz, generator tests/golden/make_lambda_golden.py + oracle/racon_dump.cpp) and the 67
deep cudapoa sample windows (tests/golden/cudapoa_windows.npz)."""
import numpy as np
import pytest

from common import (contig_edit_distance, cudapoa_fixture, identity_order, lambda_fixture, lambda_reference)
from racon_gpu_b200 import api
from racon_gpu_b200.windows import edit_distance

pytestmark = pytest.mark.gpu
MEM = 6 << 30


@pytest.mark.parametrize("case,golden", [("fastq_500", 1312), ("fasta_500", 1566)])
@pytest.mark.parametrize("via_adapter", [False, True])
def test_lambda_windows_full_band_equal_racon_cpu(oracle, case, golden, via_adapter):
    """test/racon_test.cpp:88-130 on the GPU: every window bit-identical to racon's CPU consensus (partial-span
    layers, real qualities, uneven depth), same per-window status, and the stitched contig reproduces the CPU golden
    edit distance (1312 / 1566) -- the reference's own GPU path gives 1385 / 1607 (test/racon_test.cpp:311-312, 333-334)."""
    b, cons, polished, p = lambda_fixture(case)
    got_c, got_l, got_p, status, _ = api.polish_windows(b, p["m"], p["x"], p["g"], banded=False, tgs=p["tgs"], trim=p["trim"],
                                                        mem_per_batch=MEM, stride=4096, via_adapter=via_adapter)
    got = api.consensus_list(got_c, got_l)
    assert (status == 0).all()
    assert (got_p == polished).all()
    assert got == cons
    assert contig_edit_distance(oracle, got, lambda_reference()) == golden


@pytest.mark.parametrize("case,golden", [("fastq_500", 1312), ("fasta_500", 1566)])
def test_lambda_windows_static_band_within_tolerance(oracle, case, golden):
    """Banded mode on real windows: stated tolerance vs racon's unbanded CPU consensus (>= 99 % of the windows
    identical, per-window edit distance <= 2); the contig's distance to the reference moves by at most that much."""
    b, cons, polished, p = lambda_fixture(case)
    got_c, got_l, got_p, status, _ = api.polish_windows(b, p["m"], p["x"], p["g"], banded=True, tgs=p["tgs"], trim=p["trim"],
                                                        mem_per_batch=MEM, stride=4096)
    got = api.consensus_list(got_c, got_l)
    d = [edit_distance(a, c) for a, c in zip(got, cons)]
    assert (status == 0).all() and (got_p == polished).all()
    assert sum(x == 0 for x in d) >= 0.99 * len(d) and max(d) <= 2
    assert abs(contig_edit_distance(oracle, got, lambda_reference()) - golden) <= sum(d)


def test_lambda_windows_layer_order_from_the_reference(oracle, ref):
    """The oracle is fed the layer order of the UNMODIFIED reference's std::sort call (its stored answers), not the
    product's: untrimmed consensus and coverage of every real window must still agree."""
    from oracle_lib import processing_order
    b, _, _, p = lambda_fixture("fastq_500")
    order = processing_order(b, ref.layer_order)
    oc, ocov, _ = oracle.polish(b, order, p["m"], p["x"], p["g"], tgs=False, trim=False, threads=16, stride=8192)
    pb = api.PoaBatch(max_gpu_mem=MEM, gap=p["g"], mismatch=p["x"], match=p["m"])
    n, added = pb.add_windows(b)
    assert n == b.n_windows and (np.asarray(added) == np.diff(b.win_seq_off) - 1).all()
    pb.generate_poa()
    gc, gcov, st = pb.get_consensus()
    pb.close()
    assert (st == 0).all() and gc == oc
    assert all((a == c).all() for a, c in zip(gcov, ocov))


def test_cudapoa_sample_windows(oracle):
    """vendor/GenomeWorks/cudapoa/data/sample-windows.txt: 67 windows, depth 105-170.  Full band: consensus and
    coverage of the unmodified reference's spoa path; static band within the stated tolerance."""
    b, cons, cov = cudapoa_fixture()
    wins = [b.window(w)[0] for w in range(b.n_windows)]
    for banded in (False, True):
        pb = api.PoaBatch(max_gpu_mem=MEM, banded=banded)
        for seqs in wins:  # file order IS the processing order here (cudapoa's add_poa_group contract)
            st, per = pb.add_poa_group([(s, None) for s in seqs])
            assert st == 0 and all(x == 0 for x in per)
        assert pb.get_total_poas() == 67
        pb.generate_poa()
        gc, gcov, st = pb.get_consensus()
        pb.close()
        assert (st == 0).all()
        if not banded:
            assert gc == cons
            assert all((a == c).all() for a, c in zip(gcov, cov))
        else:
            d = [edit_distance(a, c) for a, c in zip(gc, cons)]
            assert sum(x == 0 for x in d) >= 0.99 * len(d) and max(d) <= 2
