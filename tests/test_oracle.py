"""CPU: the oracle (oracle/poa_oracle.c) against the reference's golden vectors and the reference itself."""
import numpy as np
import pytest

from common import G, M, X, identity_order, ref_fixture, spoa_golden, spoa_window
from oracle_lib import processing_order
from racon_gpu_b200 import api
from racon_gpu_b200.windows import synth_windows


@pytest.mark.parametrize("use_quality,key", [(False, "GlobalConsensus"), (True, "GlobalConsensusWithQualities")])
def test_oracle_matches_spoa_known_answers(oracle, use_quality, key):
    """vendor/spoa/test/spoa_test.cpp:220-238 / :283-301 (NW 5/-4/-8 on sample.fastq)."""
    gold = spoa_golden()
    b = spoa_window(use_quality)
    sc = gold["scoring"]
    cons, _, pol = oracle.polish(b, identity_order(b), sc["m"], sc["x"], sc["g"], tgs=False, trim=False)
    assert cons[0].decode() == gold[key]
    assert pol[0]


@pytest.mark.parametrize("name", ["A", "C", "Q", "B"])
def test_oracle_matches_reference_fixtures(oracle, name):
    """Committed outputs of the unmodified reference (racon::Window + spoa AVX2), both trim modes."""
    b, ref_untrimmed, ref_trimmed = ref_fixture(name)
    order = api.processing_order(b)
    c0, _, _ = oracle.polish(b, order, M, X, G, tgs=False, trim=False, threads=8)
    c1, _, _ = oracle.polish(b, order, M, X, G, tgs=True, trim=True, threads=8)
    assert c0 == ref_untrimmed
    assert c1 == ref_trimmed


def test_oracle_matches_live_reference(oracle, ref):
    """Fresh seeds against the unmodified reference (its stored answers)."""
    for (n, L, D, e, q, seed) in [(24, 500, 32, 0.15, False, 1), (24, 300, 12, 0.2, True, 2), (6, 1000, 40, 0.1, False, 3)]:
        b = synth_windows(n, L, D, e, seed=seed, with_quality=q)
        order = processing_order(b, ref.layer_order)
        oc, ocov, _ = oracle.polish(b, order, M, X, G, tgs=True, trim=True, threads=8)
        rc, _ = ref.polish(b, M, X, G, tgs=True, trim=True, threads=8, window_length=L)
        assert oc == rc
    # coverage and topological order against spoa itself (window.cpp keeps coverages private)
    b = synth_windows(4, 300, 16, 0.15, seed=9)
    order = processing_order(b, ref.layer_order)
    oc, ocov, _ = oracle.polish(b, order, M, X, G, tgs=False, trim=False)
    for w in range(b.n_windows):
        seqs, wts, _, _ = b.window(w)
        s0 = int(b.win_seq_off[w])
        od = order[s0:s0 + len(seqs)]
        c, cov, _ = ref.spoa_window([seqs[i] for i in od], [wts[i] for i in od], M, X, G)
        assert c == oc[w] and (cov == ocov[w]).all()


def test_partial_span_layers_use_the_subgraph_path(oracle, ref):
    """window.cpp:92-103: layers that do not span the window are aligned to a subgraph."""
    from common import partial_span_windows
    pb = partial_span_windows()
    order = processing_order(pb, ref.layer_order)
    oc, _, _ = oracle.polish(pb, order, M, X, G, tgs=True, trim=True, threads=8)
    rc, _ = ref.polish(pb, M, X, G, tgs=True, trim=True, threads=8, window_length=400)
    assert oc == rc


def test_fewer_than_three_sequences_returns_backbone(oracle):
    from racon_gpu_b200.windows import WindowBatch
    b = WindowBatch.from_lists([[(b"ACGTACGT", None, 0, 0), (b"ACGTTCGT", None, 0, 7)]])
    cons, _, pol = oracle.polish(b, identity_order(b), M, X, G)
    assert cons[0] == b"ACGTACGT" and not pol[0]
