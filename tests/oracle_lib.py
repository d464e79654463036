"""ctypes loaders for the parity checkers (TEST INFRASTRUCTURE: tests/, smoke(), bench cpu legs only).

  Oracle      -> oracle/liboracle.so          plain-C restatement of racon's spoa path
  Ref         -> oracle/_ref/libracon_ref.so  the unmodified reference (racon::Window + spoa + edlib), built
                                              from racon's sources by oracle/Makefile
  RefAnswers  -> tests/golden/ref_answers.npz what Ref answered for the inputs the tests ask it about
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_ANSWERS = os.path.join(ROOT, "tests", "golden", "ref_answers.npz")


def build_oracle(quiet: bool = True) -> None:
    """(Re)build liboracle.so and, when /root/reference is present, _ref/libracon_ref.so."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True,
                   stdout=subprocess.DEVNULL if quiet else None,
                   stderr=subprocess.DEVNULL if quiet else None)


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _flat_args(b):
    return (C.c_int64(b.n_windows), _p(b.win_seq_off, C.c_int64), _p(b.seq_off, C.c_int64),
            _p(b.bases, C.c_uint8), _p(b.weights, C.c_int8), _p(b.has_weights, C.c_uint8),
            _p(b.begins, C.c_int32), _p(b.ends, C.c_int32))


class Oracle:
    def __init__(self):
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            build_oracle()
        self.lib = C.CDLL(path)
        self.lib.poa_oracle_polish_windows.restype = None

    def polish(self, batch, order: np.ndarray, m: int, x: int, g: int, tgs: bool = True,
               trim: bool = True, threads: int = 1, stride: int = 4096, want_stats: bool = False):
        """Returns (list of consensus bytes, list of coverage arrays, polished flags[, stats])."""
        W = batch.n_windows
        cons = np.zeros((W, stride), dtype=np.uint8)
        cov = np.zeros((W, stride), dtype=np.uint16)
        clen = np.zeros(W, dtype=np.int32)
        pol = np.zeros(W, dtype=np.uint8)
        stats = np.zeros((W, 6), dtype=np.int64)
        order = np.ascontiguousarray(order, dtype=np.int32)
        self.lib.poa_oracle_polish_windows(
            *_flat_args(batch), _p(order, C.c_int32), C.c_int32(int(tgs)), C.c_int32(int(trim)),
            C.c_int32(m), C.c_int32(x), C.c_int32(g), C.c_int32(threads),
            cons.ctypes.data_as(C.c_char_p), _p(cov, C.c_uint16), C.c_int32(stride),
            _p(clen, C.c_int32), _p(pol, C.c_uint8), _p(stats, C.c_int64))
        assert (clen >= 0).all(), "oracle output stride too small"
        out = [cons[w, :clen[w]].tobytes() for w in range(W)]
        covs = [cov[w, :clen[w]].copy() for w in range(W)]
        if want_stats:
            return out, covs, pol.astype(bool), stats
        return out, covs, pol.astype(bool)


def _seq_arrays(seqs, weights):
    n = len(seqs)
    arr_s = (C.c_char_p * n)(*[bytes(s) for s in seqs])
    lens = np.asarray([len(s) for s in seqs], dtype=np.int32)
    keep = [None if w is None else np.ascontiguousarray(w, dtype=np.int8) for w in weights]
    arr_w = (C.POINTER(C.c_int8) * n)(*[
        C.cast(None, C.POINTER(C.c_int8)) if w is None else _p(w, C.c_int8) for w in keep])
    return n, arr_s, lens, keep, arr_w


def window_sequences(batch, order: np.ndarray, w: int):
    """Window w of a flat batch as (seqs, weights, begins, ends) in PROCESSING order."""
    s0, s1 = int(batch.win_seq_off[w]), int(batch.win_seq_off[w + 1])
    seqs, wts, bg, en = [], [], [], []
    for k in range(s1 - s0):
        s = s0 + int(order[s0 + k])
        a, b = int(batch.seq_off[s]), int(batch.seq_off[s + 1])
        seqs.append(batch.bases[a:b].tobytes())
        wts.append(batch.weights[a:b].copy() if batch.has_weights[s] else None)
        bg.append(int(batch.begins[s]))
        en.append(int(batch.ends[s]))
    return seqs, wts, bg, en


def oracle_window_msa(oracle: "Oracle", seqs, weights, begins, ends, m: int, x: int, g: int):
    """spoa's MSA (one row per sequence, processing order) of a window built like racon builds it; begins None:
    every layer spans the window (a plain cudapoa group)."""
    lib = oracle.lib
    n, arr_s, lens, keep, arr_w = _seq_arrays(seqs, weights)
    rows = C.c_void_p()
    L = C.c_int32(0)
    lib.poa_oracle_window_msa.restype = C.c_int32
    bg = None if begins is None else np.ascontiguousarray(begins, dtype=np.int32)
    en = None if begins is None else np.ascontiguousarray(ends, dtype=np.int32)
    nr = lib.poa_oracle_window_msa(C.c_int32(n), arr_s, _p(lens, C.c_int32), arr_w,
                                   None if bg is None else _p(bg, C.c_int32),
                                   None if en is None else _p(en, C.c_int32),
                                   C.c_int32(m), C.c_int32(x), C.c_int32(g), C.byref(rows), C.byref(L))
    buf = C.string_at(rows.value, nr * L.value)
    lib.poa_oracle_free.argtypes = [C.c_void_p]
    lib.poa_oracle_free(rows)
    return [buf[i * L.value:(i + 1) * L.value] for i in range(nr)]


class Ref:
    """The unmodified reference.  `available` is False when oracle/_ref was not built/shipped."""

    def __init__(self):
        path = os.path.join(ORACLE_DIR, "_ref", "libracon_ref.so")
        if not os.path.exists(path) and os.path.isdir("/root/reference/vendor/spoa/src"):
            build_oracle()
        self.available = os.path.exists(path)
        self.lib = C.CDLL(path) if self.available else None

    def layer_order(self, begins: np.ndarray) -> np.ndarray:
        begins = np.ascontiguousarray(begins, dtype=np.int32)
        out = np.zeros(begins.shape[0], dtype=np.int32)
        self.lib.ref_layer_order(C.c_int32(begins.shape[0]), _p(begins, C.c_int32), _p(out, C.c_int32))
        return out

    def polish(self, batch, m: int, x: int, g: int, tgs: bool = True, trim: bool = True,
               threads: int = 1, window_length: int = 500, stride: int = 4096):
        W = batch.n_windows
        cons = np.zeros((W, stride), dtype=np.uint8)
        clen = np.zeros(W, dtype=np.int32)
        pol = np.zeros(W, dtype=np.uint8)
        self.lib.ref_polish_windows(
            *_flat_args(batch), C.c_int32(int(tgs)), C.c_int32(int(trim)), C.c_int32(m),
            C.c_int32(x), C.c_int32(g), C.c_int32(window_length), C.c_int32(threads),
            cons.ctypes.data_as(C.c_char_p), C.c_int32(stride), _p(clen, C.c_int32),
            _p(pol, C.c_uint8))
        assert (clen <= stride).all()
        return [cons[w, :clen[w]].tobytes() for w in range(W)], pol.astype(bool)

    def spoa_window(self, seqs, weights, m: int, x: int, g: int, max_nodes: int = 1 << 16):
        """seqs in PROCESSING order.  Returns (consensus, coverage, rank_to_node)."""
        n = len(seqs)
        arr_s = (C.c_char_p * n)(*[bytes(s) for s in seqs])
        lens = np.asarray([len(s) for s in seqs], dtype=np.int32)
        keep = [None if w is None else np.ascontiguousarray(w, dtype=np.int8) for w in weights]
        arr_w = (C.POINTER(C.c_int8) * n)(*[
            C.cast(None, C.POINTER(C.c_int8)) if w is None else _p(w, C.c_int8) for w in keep])
        max_out = int(lens.sum()) + 8
        cons = np.zeros(max_out, dtype=np.uint8)
        cov = np.zeros(max_out, dtype=np.uint32)
        rank = np.zeros(max_nodes, dtype=np.int32)
        nn = C.c_int32(0)
        self.lib.ref_spoa_window.restype = C.c_int32
        ln = self.lib.ref_spoa_window(
            C.c_int32(n), arr_s, _p(lens, C.c_int32), arr_w, C.c_int32(m), C.c_int32(x),
            C.c_int32(g), cons.ctypes.data_as(C.c_char_p), _p(cov, C.c_uint32), C.c_int32(max_out),
            _p(rank, C.c_int32), C.c_int32(max_nodes), C.byref(nn))
        return cons[:ln].tobytes(), cov[:ln].copy(), rank[:nn.value].copy()


def ref_window_msa(ref: Ref, seqs, weights, m: int, x: int, g: int):
    """spoa::Graph::generate_multiple_sequence_alignment of the unmodified reference for one group."""
    n, arr_s, lens, keep, arr_w = _seq_arrays(seqs, weights)
    cap = int(lens.sum()) * n + 64
    out = np.zeros(cap, dtype=np.uint8)
    L = C.c_int32(0)
    ref.lib.ref_spoa_window_msa.restype = C.c_int32
    nr = ref.lib.ref_spoa_window_msa(C.c_int32(n), arr_s, _p(lens, C.c_int32), arr_w, C.c_int32(m), C.c_int32(x),
                                     C.c_int32(g), out.ctypes.data_as(C.c_char_p), C.c_int64(cap), C.byref(L))
    assert nr * L.value <= cap
    return [out[i * L.value:(i + 1) * L.value].tobytes() for i in range(nr)]


def processing_order(batch, layer_order_fn) -> np.ndarray:
    """order[s] for a flat batch using a layer-order function (begins[n] -> rank[n])."""
    order = np.zeros(batch.n_seqs, dtype=np.int32)
    for w in range(batch.n_windows):
        s0, s1 = int(batch.win_seq_off[w]), int(batch.win_seq_off[w + 1])
        order[s0:s1] = layer_order_fn(batch.begins[s0:s1])
    return order


# ---------------------------------------------------------------------------------------------------
# overlap alignment (edlib NW path): oracle/aln_oracle.c restatement and the unmodified edlib in oracle/_ref
# ---------------------------------------------------------------------------------------------------
def oracle_align(oracle: "Oracle", q: bytes, t: bytes):
    """(ops uint8 array, edit distance) of the restatement; ops: 0 match, 1 insertion, 2 deletion, 3 mismatch."""
    cap = len(q) + len(t) + 8
    ops = np.zeros(cap, dtype=np.uint8)
    score = C.c_int32(0)
    oracle.lib.aln_oracle_nw.restype = C.c_int64
    n = oracle.lib.aln_oracle_nw(C.c_char_p(q), C.c_int32(len(q)), C.c_char_p(t), C.c_int32(len(t)), _p(ops, C.c_uint8),
                                 C.c_int64(cap), C.byref(score))
    assert n >= 0
    return ops[:n].copy(), int(score.value)


def ops_to_cigar(oracle: "Oracle", ops: np.ndarray) -> bytes:
    ops = np.ascontiguousarray(ops, dtype=np.uint8)
    cap = 16 * ops.shape[0] + 16
    buf = C.create_string_buffer(cap)
    oracle.lib.aln_oracle_cigar.restype = C.c_int64
    n = oracle.lib.aln_oracle_cigar(_p(ops, C.c_uint8), C.c_int64(ops.shape[0]), buf, C.c_int64(cap))
    assert n >= 0
    return buf.raw[:n]


def ref_align(ref: "Ref", q: bytes, t: bytes):
    """(ops, edit distance, CIGAR) of the unmodified edlib called like racon calls it (src/overlap.cpp:205-224)."""
    cap = len(q) + len(t) + 8
    ops = np.zeros(cap, dtype=np.uint8)
    ccap = 16 * cap
    cig = C.create_string_buffer(ccap)
    score = C.c_int32(0)
    ref.lib.ref_edlib_nw.restype = C.c_int64
    n = ref.lib.ref_edlib_nw(C.c_char_p(q), C.c_int32(len(q)), C.c_char_p(t), C.c_int32(len(t)), _p(ops, C.c_uint8),
                             C.c_int64(cap), cig, C.c_int64(ccap), C.byref(score))
    assert n >= 0
    return ops[:n].copy(), int(score.value), cig.value


def oracle_breaking_points(oracle: "Oracle", ops: np.ndarray, q_first: int, t_begin: int, t_end: int, window_length: int):
    """(t, q) pairs, two per window with a match (restatement of src/overlap.cpp:226-290 on operations)."""
    ops = np.ascontiguousarray(ops, dtype=np.uint8)
    cap = 2 * ((t_end - t_begin) // window_length + 3)
    out = np.zeros(2 * cap, dtype=np.uint32)
    oracle.lib.aln_oracle_breaking_points.restype = C.c_int64
    n = oracle.lib.aln_oracle_breaking_points(_p(ops, C.c_uint8), C.c_int64(ops.shape[0]), C.c_int32(q_first),
                                              C.c_int32(t_begin), C.c_int32(t_end), C.c_int32(window_length),
                                              _p(out, C.c_uint32), C.c_int64(cap))
    assert n >= 0
    return out[:2 * n].reshape(-1, 2).copy()


def ref_breaking_points(ref: "Ref", cigar: bytes, q_length: int, q_begin: int, q_end: int, strand: int, t_length: int,
                        t_begin: int, t_end: int, window_length: int):
    """The unmodified racon::Overlap::find_breaking_points (src/overlap.cpp:179-203,226-290) fed this CIGAR."""
    cap = 2 * ((t_end - t_begin) // window_length + 3)
    out = np.zeros(2 * cap, dtype=np.uint32)
    ref.lib.ref_racon_breaking_points.restype = C.c_int64
    n = ref.lib.ref_racon_breaking_points(C.c_char_p(cigar), C.c_uint32(q_length), C.c_uint32(q_begin), C.c_uint32(q_end),
                                          C.c_int(strand), C.c_uint32(t_length), C.c_uint32(t_begin), C.c_uint32(t_end),
                                          C.c_uint32(window_length), _p(out, C.c_uint32), C.c_int64(cap))
    assert n >= 0
    return out[:2 * n].reshape(-1, 2).copy()


# ---------------------------------------------------------------------------------------------------
# stored answers of the unmodified reference: the comparisons with it run where oracle/_ref cannot be built
# ---------------------------------------------------------------------------------------------------
def _digest(kind: str, *parts) -> str:
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, np.ndarray):
            h.update(b"a%s%s:" % (p.dtype.str.encode(), str(p.shape).encode()))
            h.update(np.ascontiguousarray(p).tobytes())
        elif isinstance(p, (bytes, bytearray)):
            h.update(b"b%d:" % len(p))
            h.update(bytes(p))
        elif isinstance(p, (list, tuple)):
            h.update(b"l%d:" % len(p))
            h.update(_digest("", *p).encode())
        elif p is None:
            h.update(b"n")
        else:
            h.update(b"i%d" % int(p))
        h.update(b"|")
    return kind + "_" + h.hexdigest()[:32]


class RefAnswers:
    """The answers of the unmodified reference (Ref) to the questions the tests ask it, with Ref's call signatures.

    Replay (default): answers come from tests/golden/ref_answers.npz, keyed by a digest of the question's inputs; a
    question it has no answer for raises KeyError.  Recording (RefAnswers(Ref())): every question goes to the live
    reference and its answer is kept for save() -- tests/golden/make_ref_answers.py."""

    def __init__(self, live: Ref | None = None):
        self.live = live
        self.store = {} if live is not None else self._load(REF_ANSWERS)

    def _answer(self, key, fields, ask):
        if self.live is not None:
            for f, v in zip(fields, ask()):
                self.store[(key, f)] = np.asarray(v)
        try:
            return [self.store[(key, f)] for f in fields]
        except KeyError:
            raise KeyError(f"{key}: no stored answer of the reference for these inputs "
                           f"(tests/golden/make_ref_answers.py records them)") from None

    # on disk: per (question kind, field) one array of all answers concatenated, their keys and their shapes
    def save(self, path: str = REF_ANSWERS):
        groups = {}
        for (key, f), a in sorted(self.store.items()):
            groups.setdefault(key.split("_")[0] + "_" + f, []).append((key, a))
        out = {}
        for g, items in groups.items():
            out[g + "_keys"] = np.asarray([k for k, _ in items], dtype="S")
            out[g + "_shapes"] = np.asarray([(a.ndim,) + a.shape + (1,) * (2 - a.ndim) for _, a in items], dtype=np.int64)
            out[g] = np.concatenate([a.reshape(-1) for _, a in items])
        np.savez_compressed(path, **out)

    @staticmethod
    def _load(path):
        z = np.load(path)
        store = {}
        for g in (n[:-5] for n in z.files if n.endswith("_keys")):
            f = g.split("_", 1)[1]
            data, at = z[g], 0
            for k, (ndim, rows, cols) in zip(z[g + "_keys"], z[g + "_shapes"]):
                store[(k.decode(), f)] = data[at:at + rows * cols].reshape((rows, cols)[:ndim])
                at += rows * cols
        return store

    def layer_order(self, begins: np.ndarray) -> np.ndarray:
        begins = np.ascontiguousarray(begins, dtype=np.int32)
        return self._answer(_digest("order", begins), ["rank"], lambda: [self.live.layer_order(begins)])[0]

    def polish(self, batch, m: int, x: int, g: int, tgs: bool = True, trim: bool = True,
               threads: int = 1, window_length: int = 500):
        key = _digest("polish", batch.win_seq_off, batch.seq_off, batch.bases, batch.weights, batch.has_weights,
                      batch.begins, batch.ends, m, x, g, tgs, trim, window_length)

        def ask():
            cons, pol = self.live.polish(batch, m, x, g, tgs=tgs, trim=trim, threads=threads, window_length=window_length)
            return [np.frombuffer(b"\n".join(cons), dtype=np.uint8), pol.astype(np.uint8)]
        cons, pol = self._answer(key, ["cons", "polished"], ask)
        return cons.tobytes().split(b"\n"), pol.astype(bool)

    def spoa_window(self, seqs, weights, m: int, x: int, g: int):
        key = _digest("spoa", [bytes(s) for s in seqs], list(weights), m, x, g)

        def ask():
            cons, cov, rank = self.live.spoa_window(seqs, weights, m, x, g)
            return [np.frombuffer(cons, dtype=np.uint8), cov, rank]
        cons, cov, rank = self._answer(key, ["cons", "cov", "rank"], ask)
        return cons.tobytes(), cov, rank

    def window_msa(self, seqs, weights, m: int, x: int, g: int):
        """ref_window_msa: the MSA rows of one group."""
        key = _digest("msa", [bytes(s) for s in seqs], list(weights), m, x, g)

        def ask():
            rows = ref_window_msa(self.live, seqs, weights, m, x, g)
            return [np.frombuffer(b"".join(rows), dtype=np.uint8).reshape(len(rows), -1)]
        return [r.tobytes() for r in self._answer(key, ["rows"], ask)[0]]

    def align(self, q: bytes, t: bytes):
        """ref_align: (ops, edit distance, CIGAR) of edlib called like racon calls it."""
        def ask():
            ops, score, cigar = ref_align(self.live, q, t)
            return [ops, score, np.frombuffer(cigar, dtype=np.uint8)]
        ops, score, cigar = self._answer(_digest("aln", q, t), ["ops", "score", "cigar"], ask)
        return ops, int(score), cigar.tobytes()

    def breaking_points(self, cigar: bytes, q_length: int, q_begin: int, q_end: int, strand: int, t_length: int,
                        t_begin: int, t_end: int, window_length: int):
        """ref_breaking_points: (t, q) pairs of racon::Overlap::find_breaking_points fed this CIGAR."""
        args = (q_length, q_begin, q_end, strand, t_length, t_begin, t_end, window_length)
        return self._answer(_digest("bp", cigar, *args), ["points"],
                            lambda: [ref_breaking_points(self.live, cigar, *args)])[0]
