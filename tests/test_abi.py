"""CPU: the C-ABI library builds, loads and exports every symbol include/b200poa.h declares."""
import ctypes as C
import os
import re

import numpy as np

from racon_gpu_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols(header="b200poa.h", prefix="b200poa_"):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(" + prefix + r"[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = api.load_library()
    names = declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(api.ABI_SYMBOLS) == names


def test_library_exports_every_aligner_symbol():
    """include/b200aln.h (overlap alignment step, SURVEY 8f-4); no compute calls without a GPU."""
    from racon_gpu_b200 import aligner
    lib = api.load_library()
    names = declared_symbols("b200aln.h", "b200aln_")
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(aligner.ALN_ABI_SYMBOLS) == names
    assert aligner.status_string(2) == "exceeded_max_alignments"


def test_config_default_follows_cudapoa_batchconfig():
    """vendor/GenomeWorks/cudapoa/src/batch.cu:34-71 for racon's BatchConfig(1023, 200, 256, mode)."""
    lib = api.load_library()
    for mode, nodes in ((api.FULL_BAND, 3072), (api.STATIC_BAND, 4092)):
        cfg = api.Config()
        lib.b200poa_config_default(C.byref(cfg), 1023, 200, 256, mode)
        assert cfg.max_sequence_size == 1023 and cfg.max_consensus_size == 2046
        assert cfg.max_sequences_per_poa == 200 and cfg.alignment_band_width == 256
        assert cfg.max_nodes_per_graph == nodes and cfg.band_mode == mode


def test_layer_order_is_racons_sort(ref):
    """src/window.cpp:78-85: libstdc++ introsort is unstable; 33 equal keys give 0,17,32,31,... (SURVEY A.3)."""
    got = api.layer_order(np.zeros(33, dtype=np.int32))
    assert got[:5].tolist() == [0, 17, 32, 31, 30]
    assert sorted(got.tolist()) == list(range(33))
    assert api.layer_order(np.zeros(17, dtype=np.int32)).tolist() == list(range(17))
    rng = np.random.default_rng(0)
    for n in (1, 2, 3, 16, 17, 40, 201):
        begins = rng.integers(0, 50, size=n).astype(np.int32)
        got = api.layer_order(begins)
        assert got[0] == 0 and sorted(got.tolist()) == list(range(n))
        assert (np.diff(begins[got[1:]]) >= 0).all()
        assert got.tolist() == ref.layer_order(begins).tolist()


def test_status_strings_and_invalid_arguments():
    lib = api.load_library()
    assert api.status_string(0) == "success" and api.status_string(1) == "exceeded_maximum_poas"
    assert api.status_string(14) == "partial_span_unsupported"
    handle = C.c_void_p()
    cfg = api.Config()
    lib.b200poa_config_default(C.byref(cfg), 1023, 200, 256, api.FULL_BAND)
    # zero memory is a configuration error (Test_CudapoaBatch.cu: zero-memory batch throws)
    st = lib.b200poa_batch_create(0, None, C.c_size_t(0), 1, C.byref(cfg), C.c_int16(-4), C.c_int16(-5), C.c_int16(3), C.byref(handle))
    assert st == 15 and not handle.value
    assert lib.b200poa_batch_total_poas(None) == 0


def test_window_arena_follows_racons_window_contract():
    """Columnar window construction (b200poa_arena_*, SURVEY 8(f)-2): layers of different windows arrive
    interleaved like in Polisher::initialize; per window they keep their add order; quality -> weight - 33;
    the argument checks of src/window.cpp:15-28,42-63 reject what racon rejects."""
    import numpy as np
    from racon_gpu_b200.windows import WindowBatch, synth_windows
    b = synth_windows(7, 120, 9, 0.1, seed=3, with_quality=True)
    per_win = [b.window(w) for w in range(b.n_windows)]
    arena = api.WindowArena()
    def qual(w):  # weights back to a PHRED+33 string
        return bytes((np.asarray(w, dtype=np.int16) + 33).astype(np.uint8))
    ids = [arena.add_window(bytes(s[0]), qual(w[0])) for s, w, _, _ in per_win]
    assert ids == list(range(7))
    # interleave: layer i of every window, then layer i+1 ...; every third layer without quality
    expect = [[(bytes(s[0]), np.asarray(w[0], dtype=np.int8), 0, 0)] for s, w, _, _ in per_win]
    for i in range(1, 10):
        for wid, (s, w, bg, en) in enumerate(per_win):
            if i >= len(s):
                continue
            q = None if i % 3 == 0 else qual(w[i])
            assert arena.add_layer(wid, bytes(s[i]), q, int(bg[i]), int(en[i]) + 1)
            expect[wid].append((bytes(s[i]), None if q is None else np.asarray(w[i], dtype=np.int8), int(bg[i]), int(en[i]) + 1))
    # what racon rejects or skips (window.cpp:44-58)
    assert arena.add_layer(0, b"", None, 0, 5)                 # empty layer: skipped, not an error
    assert arena.add_layer(0, b"ACGT", None, 7, 7)             # begin == end: skipped
    assert not arena.add_layer(0, b"ACGT", b"!!", 0, 4)        # unequal quality size
    assert not arena.add_layer(0, b"ACGT", None, 9, 3)         # begin >= end
    assert not arena.add_layer(0, b"ACGT", None, 0, 100000)    # end beyond the backbone
    assert not arena.add_layer(99, b"ACGT", None, 0, 4)        # no such window
    assert arena.add_window(b"", b"") == -1 and arena.add_window(b"ACGT", b"!!") == -1
    got = arena.finalize()
    want = WindowBatch.from_lists(expect)
    for f in ("win_seq_off", "seq_off", "bases", "weights", "has_weights", "begins", "ends"):
        assert (getattr(got, f) == getattr(want, f)).all(), f
    assert not arena.add_layer(0, b"ACGT", None, 0, 4)         # read-only after finalize
    arena.close()
