"""GPU: the overlap aligner through its C ABI (include/b200aln.h) against racon's CPU path.

Parity bar: bit-exact -- same edit distance, same operations (hence the same CIGAR) as edlib returns for
edlibAlign(q, t, {-1, EDLIB_MODE_NW, EDLIB_TASK_PATH}) (src/overlap.cpp:205-224): the oracle's restatement on seeded
random pairs around every threshold of edlib's recursion, the committed digests of the UNMODIFIED edlib on the 181
real lambda-phage overlaps of the reference's test data, and its stored answers on long reads."""
import hashlib

import numpy as np
import pytest

from common import overlap_fixture, random_pairs
from oracle_lib import ops_to_cigar, oracle_align

pytestmark = pytest.mark.gpu

SHAPES = [(1, 0.5), (2, 0.5), (5, 0.3), (63, 0.2), (64, 0.2), (65, 0.2), (129, 0.25), (200, 0.15), (700, 0.15),
          (1500, 0.1), (1800, 0.15), (1850, 0.15), (2000, 0.15), (2600, 0.2), (4000, 0.12), (5000, 0.3)]
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def _pairs():
    pairs = []
    for rep in range(3):
        pairs += random_pairs(500 + rep, SHAPES)
    rng = np.random.default_rng(23)
    # unrelated sequences and extreme shapes: several 32-block stripes, one-row / one-column problems, deep recursions
    for n, m in [(100, 3000), (3000, 100), (1, 5000), (5000, 1), (2500, 2500), (300, 9000), (9000, 300), (4200, 130),
                 (7000, 7500)]:
        pairs.append((rng.choice(ACGT, size=n).tobytes(), rng.choice(ACGT, size=m).tobytes()))
    pairs += random_pairs(31, [(9500, 0.15)])  # >= 8192 rows and 32 M cells: the "huge" shape (always a team of warps)
    q, t = random_pairs(29, [(1200, 0.1)])[0]  # bytes outside ACGT equal only themselves (edlib's alphabet)
    qa, ta = bytearray(q), bytearray(t)
    for k in range(0, len(qa), 37):
        qa[k] = ord("N")
    for k in range(5, len(ta), 41):
        ta[k] = ord("N") if k % 2 else ord("R")
    pairs.append((bytes(qa), bytes(ta)))
    return pairs


@pytest.fixture(scope="module")
def aligner():
    from racon_gpu_b200.aligner import CUDABatchAligner
    a = CUDABatchAligner(device_id=0, max_gpu_memory=8 << 30)
    yield a
    a.close()


def test_random_pairs_equal_the_oracle(oracle, aligner):
    pairs = _pairs()
    aligner.reset()
    for q, t in pairs:
        assert aligner.add_overlap(q, t)
    aligner.align_all()
    got = aligner.generate_cigar_strings()
    info = aligner.info()
    assert info["levels"] >= 2 and info["n_leaves"] >= len(pairs)
    # per level at most one launch of warp teams and one of single warps; then the leaves, then the CIGARs
    assert info["levels"] + 2 <= info["kernel_launches"] <= 2 * info["levels"] + 2
    assert info["team_launches"] >= 1  # a thin level's tall sub-problems went to teams of warps
    for k, (q, t) in enumerate(pairs):
        ops, score = oracle_align(oracle, q, t)
        cigar, ed = got[k]
        assert ed == score, (k, len(q), len(t))
        mine = aligner.ops(k)
        assert mine.shape == ops.shape and (mine == ops).all(), (k, len(q), len(t))
        assert cigar == ops_to_cigar(oracle, ops)
    aligner.reset()


def test_real_lambda_overlaps_equal_unmodified_edlib(aligner):
    """All 181 overlaps of /root/reference/test/data/sample_overlaps.paf.gz, cut like src/overlap.cpp:186-199."""
    fx = overlap_fixture()
    aligner.reset()
    for f in fx:
        assert aligner.add_overlap(f["q"], f["t"])
    aligner.align_all()
    got = aligner.generate_cigar_strings()
    assert len(got) == len(fx) == 181
    for k, f in enumerate(fx):
        cigar, ed = got[k]
        assert ed == f["score"], k
        assert hashlib.sha256(cigar).hexdigest() == f["cigar_sha"], k
        assert aligner.ops(k).shape[0] == f["n_ops"]
    aligner.reset()


@pytest.mark.parametrize("permille", [0, 30, 150, 320, 600, -1])
def test_top_level_band_guesses_never_change_the_result(permille):
    """The top sub-problem of every alignment runs in a band the host GUESSES (b200aln_batch_set_band_guess) and the
    kernels verify: far too small (every alignment is redone whole), about right, generous, learnt from the batch's
    previous align_all (-1: the second round guesses) -- always edlib's CIGARs, for one-warp and team launches alike."""
    from racon_gpu_b200.aligner import CUDABatchAligner, pack_pairs
    fx = overlap_fixture()
    q, qo, t, to = pack_pairs([(f["q"], f["t"]) for f in fx])
    al = CUDABatchAligner(device_id=0, max_gpu_memory=8 << 30)
    al.set_band_guess(permille)
    for rnd in range(2):
        assert al.add_overlaps(q, qo, t, to) == len(fx)
        al.align_all()
        text, off, ln, ed = al.cigars()
        for k, f in enumerate(fx):
            assert ed[k] == f["score"], (rnd, k)
            assert hashlib.sha256(text[off[k]:off[k] + ln[k]]).hexdigest() == f["cigar_sha"], (rnd, k)
        al.reset()
    al.close()


def test_saturated_level_with_huge_overlaps_on_the_side_stream():
    """Enough tall sub-problems to fill the device one warp each (so the level is not 'thin'), among them overlaps of
    >= 8192 rows: those go to teams of warps on the side stream while the one-warp grid does the rest.  Every CIGAR is
    still edlib's."""
    from racon_gpu_b200.aligner import CUDABatchAligner, pack_pairs
    fx = overlap_fixture()
    rep = 16
    assert sum(1 for f in fx if len(f["q"]) >= 8192) >= 2
    q, qo, t, to = pack_pairs([(f["q"], f["t"]) for f in fx] * rep)
    al = CUDABatchAligner(device_id=0, max_gpu_memory=24 << 30)
    assert al.add_overlaps(q, qo, t, to) == len(fx) * rep
    al.align_all()
    text, off, ln, ed = al.cigars()
    info = al.info()
    al.close()
    assert info["team_launches"] >= 1 and info["kernel_launches"] > info["team_launches"] + 2
    for k in range(len(fx) * rep):
        f = fx[k % len(fx)]
        assert ed[k] == f["score"], k
        assert hashlib.sha256(text[off[k]:off[k] + ln[k]]).hexdigest() == f["cigar_sha"], k


@pytest.mark.parametrize("devices,batches", [((0,), 2), ((0, 0), 1), ((0,), 3)])
def test_aligner_pool_threads_and_devices(devices, batches):
    """b200aln_aligner_*: several batches per device / several devices, one host thread per batch (the structure of
    cudapolisher.cpp:74-214).  A small per-batch budget forces every thread through several fill/align/reset rounds."""
    from racon_gpu_b200.aligner import AlignerPool, pack_pairs
    fx = overlap_fixture()
    rep = 3
    q, qo, t, to = pack_pairs([(f["q"], f["t"]) for f in fx] * rep)
    pool = AlignerPool(devices=devices, batches_per_device=batches, max_gpu_memory_per_batch=3 << 30)
    for _ in range(2):  # a pool is reusable
        ed, buf, off, ln, info = pool.align(q, qo, t, to)
        for k in range(len(fx) * rep):
            f = fx[k % len(fx)]
            assert ed[k] == f["score"], k
            assert hashlib.sha256(buf[off[k]:off[k] + ln[k]].tobytes()).hexdigest() == f["cigar_sha"], k
            assert buf[off[k] + ln[k]] == 0
    assert info["cells"] > 0 and info["kernel_launches"] >= 6
    pool.close()


@pytest.mark.parametrize("skip_cigars", [False, True])
def test_breaking_points_of_real_overlaps_equal_racons(skip_cigars):
    """Overlap::find_breaking_points_from_cigar (src/overlap.cpp:226-290) on the device: all 181 real overlaps, window
    length 500, against what the UNMODIFIED racon derives from edlib's CIGAR (tests/golden/lambda_overlaps.npz: bp)."""
    from racon_gpu_b200.aligner import CUDABatchAligner, pack_pairs
    fx = overlap_fixture()
    q, qo, t, to = pack_pairs([(f["q"], f["t"]) for f in fx])
    al = CUDABatchAligner(device_id=0, max_gpu_memory=8 << 30)
    al.set_window_length(500, skip_cigars=skip_cigars)
    assert al.add_overlaps(q, qo, t, to, 0, np.asarray([f["q_first"] for f in fx]), np.asarray([f["t_begin"] for f in fx])) == len(fx)
    al.align_all()
    bps = al.breaking_points()
    for k, f in enumerate(fx):
        assert bps[k].shape == f["bp"].shape and (bps[k] == f["bp"]).all(), k
    if skip_cigars:
        with pytest.raises(RuntimeError):
            al.cigars()
        assert al.info()["d2h_bytes"] < 200_000  # 5116 points x 8 B + 48 B per overlap: no CIGAR bytes came back
    else:
        text, off, ln, ed = al.cigars()
        for k, f in enumerate(fx):
            assert hashlib.sha256(text[off[k]:off[k] + ln[k]]).hexdigest() == f["cigar_sha"], k
    al.close()


def test_breaking_points_random_coordinates_and_window_lengths(oracle):
    from oracle_lib import oracle_breaking_points
    from racon_gpu_b200.aligner import CUDABatchAligner
    rng = np.random.default_rng(9)
    for w in (1, 7, 100, 500, 5000):
        al = CUDABatchAligner(device_id=0, max_gpu_memory=2 << 30)
        al.set_window_length(w)
        cases = []
        for rep in range(24):
            n, e = int(rng.integers(1, 4000)), float(rng.uniform(0.02, 0.4))
            q, t = random_pairs(3000 + 100 * w + rep, [(n, e)])[0]
            q_first, t_begin = int(rng.integers(0, 5000)), int(rng.integers(0, 50000))
            st = al.lib.b200aln_batch_add_overlap(al.h, q, len(q), t, len(t), q_first, t_begin)
            assert st == 0
            cases.append((q, t, q_first, t_begin))
        al.align_all()
        bps = al.breaking_points()
        for k, (q, t, q_first, t_begin) in enumerate(cases):
            ops, score = oracle_align(oracle, q, t)
            want = oracle_breaking_points(oracle, ops, q_first, t_begin, t_begin + len(t), w)
            assert bps[k].shape == want.shape and (bps[k] == want).all(), (w, k)
        al.close()


def test_full_batch_is_back_pressure_not_an_error(oracle):
    """Aligner::add_alignment -> exceeded_max_alignments => addOverlap returns false (cudaaligner.cpp:64-67); the
    caller aligns, resets and goes on (cudapolisher.cpp:139-174).  Results do not depend on the batching."""
    from racon_gpu_b200.aligner import CUDABatchAligner, pack_pairs, align_pairs
    pairs = random_pairs(77, [(3000, 0.12)] * 40 + [(800, 0.2)] * 40)
    small = CUDABatchAligner(device_id=0, max_gpu_memory=4 << 20)  # two slots + about forty of these pairs
    out, rounds, k = [], 0, 0
    while k < len(pairs):
        while k < len(pairs) and small.add_overlap(*pairs[k]):
            k += 1
        assert small.has_overlaps()
        small.align_all()
        out += small.generate_cigar_strings()
        small.reset()
        rounds += 1
    small.close()
    assert rounds >= 2 and len(out) == len(pairs)
    # columnar add + in-place CIGAR table (b200aln_batch_add_alignments / _get_cigars), same answers
    q, qo, t, to = pack_pairs(pairs)
    bulk = CUDABatchAligner(device_id=0, max_gpu_memory=1 << 30)
    assert bulk.add_overlaps(q, qo, t, to) == len(pairs)
    bulk.align_all()
    text, off, ln, ed2 = bulk.cigars()
    assert [(text[off[i]:off[i] + ln[i]], int(ed2[i])) for i in range(len(pairs))] == out
    bulk.close()
    # the view form: no staging copy, upload straight from the caller's (here page-locked) buffers
    from racon_gpu_b200.aligner import pinned
    viewb = CUDABatchAligner(device_id=0, max_gpu_memory=1 << 30)
    with pinned(q, t):
        assert viewb.add_overlaps(q, qo, t, to, view=True) == len(pairs)
        viewb.align_all()
    text, off, ln, ed2 = viewb.cigars()
    assert [(text[off[i]:off[i] + ln[i]], int(ed2[i])) for i in range(len(pairs))] == out
    viewb.close()
    ed, cigars, coff, info = align_pairs(*pack_pairs(pairs), device_id=0, max_gpu_memory=2 << 30)
    for i, (q, t) in enumerate(pairs):
        ops, score = oracle_align(oracle, q, t)
        want = ops_to_cigar(oracle, ops)
        assert out[i] == (want, score)
        assert ed[i] == score and cigars[coff[i]:coff[i + 1] - 1].tobytes() == want
    assert info["cells"] > 0 and info["kernel_ms"] > 0


def unmodified_edlib_pairs():
    pairs = random_pairs(901, [(6000, 0.14), (2500, 0.3), (1900, 0.05), (64, 0.3)])
    # long reads: slots re-made for the longer sequences, five and more Hirschberg levels, huge sub-problems on teams at
    # several levels, leaves of many stripes (tall, narrow) -- only the real edlib is fast enough to check these
    pairs += random_pairs(902, [(42000, 0.12), (70000, 0.08)])
    rng = np.random.default_rng(5)
    pairs.append((rng.choice(ACGT, size=30000).tobytes(), rng.choice(ACGT, size=12000).tobytes()))  # unrelated, tall
    pairs.append((rng.choice(ACGT, size=900).tobytes(), rng.choice(ACGT, size=50000).tobytes()))    # unrelated, wide
    return pairs


def test_live_against_the_unmodified_edlib(ref, aligner):
    pairs = unmodified_edlib_pairs()
    aligner.reset()
    for q, t in pairs:
        assert aligner.add_overlap(q, t)
    aligner.align_all()
    got = aligner.generate_cigar_strings()
    for k, (q, t) in enumerate(pairs):
        ops, score, cigar = ref.align(q, t)
        assert got[k] == (cigar, score)
        assert (aligner.ops(k) == ops).all()
    aligner.reset()


def test_argument_and_state_errors(aligner):
    from racon_gpu_b200 import aligner as A
    aligner.reset()
    lib = aligner.lib
    assert lib.b200aln_batch_sync(aligner.h) == A.UNINITIALIZED  # nothing aligned yet
    assert lib.b200aln_batch_add_alignment(aligner.h, None, 5, b"ACGT", 4) == A.INVALID_ARGUMENT
    assert lib.b200aln_batch_add_alignment(aligner.h, b"ACGT", -1, b"ACGT", 4) == A.INVALID_ARGUMENT
    aligner.align_all()  # an empty batch aligns to nothing
    assert aligner.generate_cigar_strings() == []
    aligner.reset()
    assert aligner.add_overlap(b"ACGT", b"")  # degenerate pairs: all insertions / all deletions / identical
    assert aligner.add_overlap(b"", b"ACG")
    assert aligner.add_overlap(b"ACGTACGT", b"ACGTACGT")
    aligner.align_all()
    assert aligner.generate_cigar_strings() == [(b"4I", 4), (b"3D", 3), (b"8M", 0)]
    aligner.reset()


def test_limits_and_call_order_are_statuses():
    """Nothing crashes or falls back: a pair that can never fit the budget, calls in the wrong order and options set on
    a non-empty batch all come back as status codes (cudaaligner.hpp:34-42 values where they exist)."""
    from racon_gpu_b200 import aligner as A
    al = A.CUDABatchAligner(device_id=0, max_gpu_memory=8 << 20)
    lib, h = al.lib, al.h
    big = b"A" * 3_000_000  # 6 M operations need 48 MB of arenas: more than this batch will ever have
    assert lib.b200aln_batch_add_alignment(h, big, len(big), big, len(big)) == A.EXCEEDED_MAX_LENGTH
    assert not al.has_overlaps()
    assert al.add_overlap(b"ACGTACGTAC", b"ACGTTCGTAC")
    assert lib.b200aln_batch_set_window_length(h, 500, 0) == A.GENERIC_ERROR      # not on a batch that holds overlaps
    assert lib.b200aln_batch_get_breaking_points(h, None, None, None) == A.UNINITIALIZED
    q = np.frombuffer(b"ACGT", dtype=np.uint8)
    off = np.asarray([0, 4], dtype=np.int64)
    with pytest.raises(RuntimeError):
        al.add_overlaps(q, off, q, off, view=True)                                # a view needs an empty batch
    al.align_all()
    assert lib.b200aln_batch_add_alignment(h, b"AC", 2, b"AC", 2) == A.GENERIC_ERROR  # reset() first
    assert al.generate_cigar_strings() == [(b"10M", 1)]
    assert lib.b200aln_batch_get_breaking_points(h, None, None, None) == A.GENERIC_ERROR  # no window length was set
    al.reset()
    assert lib.b200aln_batch_set_window_length(h, 0, 1) == A.INVALID_ARGUMENT     # nothing would come back
    assert lib.b200aln_batch_set_window_length(h, -5, 0) == A.INVALID_ARGUMENT
    al.set_window_length(4)
    assert lib.b200aln_batch_add_overlap(h, b"ACGTACGTAC", 10, b"ACGTTCGTAC", 10, 3, 6) == 0
    al.align_all()
    bp = al.breaking_points()[0]
    # windows of the contig: [6,7] [8,11] [12,15]; every column is a match or mismatch
    assert bp.tolist() == [[6, 3], [8, 5], [8, 5], [12, 9], [12, 9], [16, 13]]
    al.close()
    with pytest.raises(RuntimeError):
        A.CUDABatchAligner(device_id=999)
