"""Multiple sequence alignment output (SURVEY.md 8(f)-4: Batch::get_msa, generateMSAKernel).

Parity target = spoa::Graph::generate_multiple_sequence_alignment (vendor/spoa/src/graph.cpp:373-427), which is what the
reference's own test holds cudapoa's MSA against (vendor/GenomeWorks/cudapoa/tests/Test_CudapoaGenerateMSA2.cu:117-128).
CPU here: the oracle's restatement against committed digests of the unmodified reference (tests/golden/ref_msa.npz)
and its stored rows (tests/golden/ref_answers.npz), and the engine's emulation against the oracle.  GPU:
tests/test_gpu_msa.py."""
import os
import sys

import numpy as np
import pytest

from common import G, GOLDEN, M, X
from oracle_lib import oracle_window_msa

sys.path.insert(0, GOLDEN)
from make_msa_golden import digest, msa_groups  # noqa: E402


@pytest.fixture(scope="module")
def groups():
    return msa_groups()


def test_oracle_msa_matches_the_committed_reference_digests(oracle, groups):
    z = np.load(os.path.join(GOLDEN, "ref_msa.npz"))
    assert set(z.files) == set(groups)
    for name, (seqs, wts, (m, x, g)) in groups.items():
        n_rows, msa_len, sha = z[name].tobytes().decode().split()
        rows = oracle_window_msa(oracle, seqs, wts, None, None, m, x, g)
        assert (len(rows), len(rows[0])) == (int(n_rows), int(msa_len)), name
        assert digest(rows) == sha, name
        # Test_CudapoaGenerateMSA2.cu:120-126: a row without its gaps is the input sequence
        assert [r.replace(b"-", b"") for r in rows] == [bytes(s) for s in seqs]


def test_oracle_msa_matches_live_reference(oracle, ref, groups):
    for name, (seqs, wts, (m, x, g)) in list(groups.items())[:12]:
        assert oracle_window_msa(oracle, seqs, wts, None, None, m, x, g) == ref.window_msa(seqs, wts, m, x, g), name


def _oracle_msas(oracle, b, order, m, x, g, spans=True):
    from oracle_lib import window_sequences
    out = []
    for w in range(b.n_windows):
        seqs, wts, bg, en = window_sequences(b, order, w)
        out.append(oracle_window_msa(oracle, seqs, wts, bg if spans else None, en if spans else None, m, x, g))
    return out


def _emu_vs_oracle(oracle, b, m, x, g, **kw):
    from emu_lib import Emu
    from racon_gpu_b200 import api
    order = api.processing_order(b)
    emu = Emu()
    _, _, st, _ = emu.polish(b, order, m, x, g, msa_cap=256 << 20, **kw)
    want = _oracle_msas(oracle, b, order, m, x, g)
    assert (st == 0).all()
    for w in range(b.n_windows):
        assert emu.last_msa[w] == want[w], f"window {w}"
    return emu


def test_emulated_engine_msa_equals_oracle_on_synthetic_windows(oracle):
    from racon_gpu_b200.windows import synth_windows
    _emu_vs_oracle(oracle, synth_windows(12, 500, 32, 0.15, seed=41), M, X, G)
    _emu_vs_oracle(oracle, synth_windows(8, 300, 14, 0.2, seed=42, with_quality=True), M, X, G)


def test_emulated_engine_msa_with_partial_span_layers_and_other_scorings(oracle):
    from common import awkward_windows, partial_span_windows
    _emu_vs_oracle(oracle, partial_span_windows(), M, X, G)
    for (m, x, g) in [(5, -4, -8), (1, -1, -1)]:
        _emu_vs_oracle(oracle, awkward_windows(m, x, g, n=24), m, x, g)


def test_emulated_engine_msa_on_real_racon_windows(oracle):
    """Real lambda-phage windows (two thirds of their layers are partial spans, FASTQ qualities)."""
    from common import lambda_fixture
    b, _, _, prm = lambda_fixture("fastq_500")
    from racon_gpu_b200.windows import WindowBatch
    keep = [w for w in range(b.n_windows) if b.win_seq_off[w + 1] - b.win_seq_off[w] >= 3][:24]
    sub = WindowBatch.from_lists([[(s, wt, bg, en) for s, wt, bg, en in zip(*b.window(w))] for w in keep])
    _emu_vs_oracle(oracle, sub, prm["m"], prm["x"], prm["g"], max_len=2047, max_nodes=8192)


def test_msa_longer_than_max_consensus_size_is_reported_like_cudapoa(oracle):
    """cudapoa_generate_msa.cuh:203-208 / Test_CudapoaGenerateMSA2.cu:132-170 (CudapoaMSAFailure)."""
    from emu_lib import Emu
    from racon_gpu_b200 import api
    from racon_gpu_b200.windows import synth_windows
    b = synth_windows(2, 200, 24, 0.3, seed=43)
    emu = Emu()
    _, _, st, _ = emu.polish(b, api.processing_order(b), M, X, G, msa_cap=1 << 20, stride=256)
    assert all(m == 2 for m in emu.last_msa)  # exceeded_maximum_sequence_size
