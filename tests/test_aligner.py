"""CPU: the overlap alignment path (SURVEY.md 8(f)-4, CUDABatchAligner / src/overlap.cpp:205-224).

Parity target = the CIGAR racon's CPU path gets from edlib (NW, path).  Here: the oracle's restatement
(oracle/aln_oracle.c) against the committed digests of the unmodified edlib on REAL overlaps
(tests/golden/lambda_overlaps.npz), against its stored answers (tests/golden/ref_answers.npz) on random pairs around
every threshold of edlib's recursion, and the engine's lane emulation against the oracle.  GPU:
tests/test_gpu_aligner.py."""
import hashlib

import numpy as np
import pytest

from common import overlap_fixture, random_pairs
from oracle_lib import ops_to_cigar, oracle_align

SHAPES = [(1, 0.5), (2, 0.5), (5, 0.3), (63, 0.2), (64, 0.2), (65, 0.2), (129, 0.25), (200, 0.15), (700, 0.15),
          (1500, 0.1), (1800, 0.15), (1850, 0.15), (2000, 0.15), (2600, 0.2), (4000, 0.12), (5000, 0.3)]


def test_restatement_matches_edlib_digests_on_real_overlaps(oracle):
    fx = overlap_fixture()
    assert len(fx) == 181
    order = np.argsort([len(f["q"]) * len(f["t"]) for f in fx])
    for i in list(order[:70]) + list(order[-2:]):  # the 70 smallest (1.4 - 4 kb) and the two largest (11 kb)
        f = fx[i]
        ops, score = oracle_align(oracle, f["q"], f["t"])
        assert score == f["score"] and ops.shape[0] == f["n_ops"]
        assert hashlib.sha256(ops_to_cigar(oracle, ops)).hexdigest() == f["cigar_sha"], i


def test_restatement_matches_live_edlib(oracle, ref):
    pairs = []
    for rep in range(6):
        pairs += random_pairs(100 + rep, [s for s in SHAPES if s[0] < 300 or rep < 2])
    rng = np.random.default_rng(7)
    for n, m in [(100, 3000), (3000, 100), (1, 5000), (5000, 1), (2500, 2500), (700, 9000), (9000, 700)]:
        pairs.append((rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n).tobytes(),
                      rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=m).tobytes()))
    for q, t in pairs:
        a, sa = oracle_align(oracle, q, t)
        b, sb, cigar = ref.align(q, t)
        assert sa == sb and a.shape == b.shape and (a == b).all()
        assert ops_to_cigar(oracle, a) == cigar


@pytest.fixture(scope="module")
def emu():
    from emu_lib import EmuAligner
    return EmuAligner()


def test_emulated_aligner_equals_oracle_on_random_pairs(oracle, emu):
    """Wavefront bit-vector passes, split rule, leaf records and traceback of the engine (lane emulation)."""
    pairs = []
    for rep in range(3):
        pairs += random_pairs(300 + rep, [s for s in SHAPES if s[0] < 300 or rep < 1])
    rng = np.random.default_rng(11)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    # unrelated sequences and extreme shapes: tall leaves span several 32-block stripes, 1-row / 1-column problems
    for n, m in [(100, 3000), (3000, 100), (1, 5000), (5000, 1), (2500, 2500), (300, 9000), (9000, 300), (4200, 130)]:
        pairs.append((rng.choice(acgt, size=n).tobytes(), rng.choice(acgt, size=m).tobytes()))
    # characters outside ACGT equal only themselves (edlib builds its alphabet from the bytes it sees)
    q, t = random_pairs(17, [(900, 0.1)])[0]
    qa, ta = bytearray(q), bytearray(t)
    for k in range(0, len(qa), 37):
        qa[k] = ord("N")
    for k in range(5, len(ta), 41):
        ta[k] = ord("N") if k % 2 else ord("R")
    pairs.append((bytes(qa), bytes(ta)))
    depths = set()
    for q, t in pairs:
        a, sa = oracle_align(oracle, q, t)
        b, sb, depth, leaves = emu.align(q, t)
        assert sa == sb and a.shape == b.shape and (a == b).all(), (len(q), len(t))
        assert emu.cigar == ops_to_cigar(oracle, a)  # run starts (aln_runs) -> CIGAR like edlibAlignmentToCigar
        depths.add(depth)
    assert 0 in depths and max(depths) >= 2  # direct tracebacks and Hirschberg recursions both occurred


def test_emulated_aligner_on_real_overlaps(oracle, emu):
    fx = overlap_fixture()
    order = np.argsort([len(f["q"]) * len(f["t"]) for f in fx])
    for i in list(order[:12]) + [order[90], order[-1]]:
        f = fx[i]
        ops, score, depth, leaves = emu.align(f["q"], f["t"])
        assert score == f["score"] and ops.shape[0] == f["n_ops"]
        assert hashlib.sha256(ops_to_cigar(oracle, ops)).hexdigest() == f["cigar_sha"], i


def test_emulated_aligner_on_long_reads_against_live_edlib(ref, emu):
    """40 kb reads: five Hirschberg levels, all three shape classes (short / tall / huge), leaves of many stripes; only
    the real edlib is fast enough to be the checker here."""
    pairs = random_pairs(902, [(42000, 0.12)])
    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs.append((rng.choice(acgt, size=30000).tobytes(), rng.choice(acgt, size=12000).tobytes()))
    pairs.append((rng.choice(acgt, size=900).tobytes(), rng.choice(acgt, size=50000).tobytes()))
    for q, t in pairs:
        ops, score, cigar = ref.align(q, t)
        a, sa, depth, leaves = emu.align(q, t)
        assert sa == score and a.shape == ops.shape and (a == ops).all() and emu.cigar == cigar
    assert depth >= 3


def test_breaking_points_restatement_and_engine(oracle, ref, emu):
    """src/overlap.cpp:226-290: the oracle's restatement against the UNMODIFIED racon (its stored answers) on random
    overlaps with random coordinates / strands / window lengths, the committed real breaking points (window length 500),
    and the engine's run-based version (lane emulation) against both."""
    from oracle_lib import oracle_breaking_points
    rng = np.random.default_rng(3)
    for rep in range(60):
        n, e = int(rng.integers(1, 3000)), float(rng.uniform(0.02, 0.4))
        q, t = random_pairs(2000 + rep, [(n, e)])[0]
        w = int(rng.choice([1, 7, 50, 100, 500, 1000, 5000]))
        t_begin = int(rng.integers(0, 2500))
        strand, q_len = int(rng.integers(0, 2)), len(q) + int(rng.integers(0, 300))
        q_begin = int(rng.integers(0, q_len - len(q) + 1))
        q_first = q_len - (q_begin + len(q)) if strand else q_begin
        ops, score = oracle_align(oracle, q, t)
        want = oracle_breaking_points(oracle, ops, q_first, t_begin, t_begin + len(t), w)
        got = ref.breaking_points(ops_to_cigar(oracle, ops), q_len, q_begin, q_begin + len(q), strand,
                                  t_begin + len(t) + 5, t_begin, t_begin + len(t), w)
        assert got.shape == want.shape and (got == want).all(), rep
        emu.align(q, t, q_first, t_begin, w)
        assert emu.breaking_points.shape == want.shape and (emu.breaking_points == want).all(), (rep, n, w)
    fx = overlap_fixture()
    order = np.argsort([len(f["q"]) * len(f["t"]) for f in fx])
    for i in list(order[:10]) + [order[100], order[-1]]:
        f = fx[i]
        ops, score = oracle_align(oracle, f["q"], f["t"])
        want = oracle_breaking_points(oracle, ops, f["q_first"], f["t_begin"], f["t_begin"] + len(f["t"]), 500)
        assert want.shape == f["bp"].shape and (want == f["bp"]).all(), i
        emu.align(f["q"], f["t"], f["q_first"], f["t_begin"], 500)
        assert (emu.breaking_points == f["bp"]).all(), i


def test_banded_passes_with_guessed_and_exact_bounds(oracle, ref, emu):
    """Bands: children of a split know their optimum exactly (every test above already runs them banded); the top
    sub-problem gets a GUESS from the host and is redone without a band when its optimum turns out larger.  Too small,
    exact, tight and generous guesses all give edlib's alignment."""
    pairs = random_pairs(77, [(2600, 0.2), (4000, 0.12), (5000, 0.3), (2300, 0.02)])
    rng = np.random.default_rng(12)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs.append((rng.choice(acgt, size=4100).tobytes(), rng.choice(acgt, size=2900).tobytes()))  # unrelated: a huge distance
    pairs.append((rng.choice(acgt, size=300).tobytes(), rng.choice(acgt, size=9000).tobytes()))
    for q, t in pairs:
        ops, score = oracle_align(oracle, q, t)
        for guess in (0, score // 2, score - 1, score, score + 1, 2 * score + 64, 10 ** 6):
            a, sa, depth, leaves = emu.align(q, t, guess=guess)
            assert sa == score and a.shape == ops.shape and (a == ops).all(), (len(q), len(t), guess)
    # long reads: narrow strips of a large matrix, several stripes handing over anchors
    for (q, t), frac in zip(random_pairs(903, [(42000, 0.12), (30000, 0.03)]), (0.25, 0.05)):
        ops, score, cigar = ref.align(q, t)
        for guess in (int(frac * len(t)), score, score - 1):
            a, sa, depth, leaves = emu.align(q, t, guess=guess)
            assert sa == score and (a == ops).all() and emu.cigar == cigar, (len(q), guess)
