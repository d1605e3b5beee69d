"""ctypes binding of oracle/liboracle.so — TEST INFRASTRUCTURE ONLY.

The oracle is the CPU restatement of the reference's hot path (see the header of
oracle/tgx_oracle.cpp).  It may be imported only from tests/, from
``__graft_entry__.smoke()`` and from ``bench.py``'s cpu_baseline / ``--impl
reference`` legs — never from ``tokengeex_b200`` (the product).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "tgx_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "liboracle.so"])
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.orc_model_create.restype = C.c_void_p
        L.orc_model_create.argtypes = [u8p, u64p, f64p, u8p, C.c_uint64]
        L.orc_model_destroy.argtypes = [C.c_void_p]
        L.orc_model_vocab_size.restype = C.c_uint64
        L.orc_model_vocab_size.argtypes = [C.c_void_p]
        L.orc_model_vocab_bytes.restype = C.c_uint64
        L.orc_model_vocab_bytes.argtypes = [C.c_void_p]
        L.orc_model_export.argtypes = [C.c_void_p, u8p, u64p, f64p, u8p]
        L.orc_encode.restype = C.c_int64
        L.orc_encode.argtypes = [C.c_void_p, u8p, C.c_uint64, C.c_double, u32p, C.c_uint64, u64p]
        L.orc_encode_keyed.restype = C.c_int64
        L.orc_encode_keyed.argtypes = [C.c_void_p, u8p, C.c_uint64, C.c_double, C.c_uint64, C.c_uint64, u32p,
                                       C.c_uint64, u64p]
        L.orc_crlf.restype = C.c_uint64
        L.orc_crlf.argtypes = [u8p, C.c_uint64, u8p]
        L.orc_encode_batch.restype = C.c_uint64
        L.orc_encode_batch.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_int, u32p,
                                       C.c_uint64, u64p, i32p, u64p]
        L.orc_common_prefix_search.restype = C.c_uint64
        L.orc_common_prefix_search.argtypes = [C.c_void_p, u8p, C.c_uint64, u32p, u32p, C.c_uint64]
        L.orc_marginal.restype = C.c_double
        L.orc_marginal.argtypes = [C.c_void_p, u8p, C.c_uint64, f64p, C.c_int]
        L.orc_alpha_beta.restype = C.c_double
        L.orc_alpha_beta.argtypes = [C.c_void_p, u8p, C.c_uint64, f64p, f64p]
        L.orc_run_e_step.restype = C.c_int
        L.orc_run_e_step.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_int,
                                     C.c_uint64, f64p, i64p, f64p]
        L.orc_run_e_step_dropout.restype = C.c_int
        L.orc_run_e_step_dropout.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_uint64, C.c_double,
                                             C.c_int, C.c_uint64, C.c_uint64, f64p, i64p, f64p]
        L.orc_run_e_step_fixed.restype = C.c_int
        L.orc_run_e_step_fixed.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_uint64, C.c_double,
                                           C.c_int, C.c_uint64, C.c_uint64, u64p, i64p, f64p]
        L.orc_marginal_contributions.restype = C.c_double
        L.orc_marginal_contributions.argtypes = [C.c_void_p, u8p, C.c_uint64, u32p, f64p, C.c_uint64, u64p,
                                                 C.c_double, C.c_uint64, C.c_uint64]
        L.orc_digamma.restype = C.c_double
        L.orc_digamma.argtypes = [C.c_double]
        L.orc_log_sum_exp.restype = C.c_double
        L.orc_log_sum_exp.argtypes = [C.c_double, C.c_double, C.c_int]
        L.orc_run_m_step.restype = C.c_void_p
        L.orc_run_m_step.argtypes = [C.c_void_p, f64p, C.POINTER(C.c_int)]
        L.orc_pair_frequencies.restype = C.c_int64
        L.orc_pair_frequencies.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, u64p, u64p, C.c_uint64, u64p]
        L.orc_token_frequencies.restype = C.c_int
        L.orc_token_frequencies.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, u64p, u64p]
        L.orc_token_alternatives.restype = C.c_uint64
        L.orc_token_alternatives.argtypes = [C.c_void_p, u8p, u64p, u32p, C.c_uint64]
        L.orc_nbest.restype = C.c_uint64
        L.orc_nbest.argtypes = [C.c_void_p, u8p, C.c_uint64, C.c_uint64, u32p, u64p, C.c_uint64]
        L.orc_prune_vocab.restype = C.c_void_p
        L.orc_prune_vocab.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_uint64,
                                      C.c_double, C.POINTER(C.c_int), f64p]
        L.orc_prune.restype = C.c_void_p
        L.orc_prune.argtypes = [C.c_void_p, u8p, u64p, C.c_uint64, C.c_int, C.c_uint64, C.c_double,
                                C.c_uint64, C.POINTER(C.c_int), u64p, C.c_uint64, u64p]
        _lib = L
    return _lib


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def _bytes_arr(b) -> np.ndarray:
    if isinstance(b, np.ndarray):
        return np.ascontiguousarray(b, dtype=np.uint8)
    a = np.frombuffer(bytes(b), dtype=np.uint8)
    return a if a.size else np.zeros(1, dtype=np.uint8)[:0].copy()


def pack_vocab(tokens: Sequence[bytes], scores: Sequence[float], keep: Optional[Sequence[bool]] = None):
    """(blob u8[], offsets u64[V+1], scores f64[V], keep u8[V])"""
    lens = np.fromiter((len(t) for t in tokens), dtype=np.uint64, count=len(tokens))
    off = np.zeros(len(tokens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b"".join(tokens), dtype=np.uint8).copy() if len(tokens) else np.zeros(0, np.uint8)
    if blob.size == 0:
        blob = np.zeros(1, np.uint8)
    sc = np.asarray(scores, dtype=np.float64).copy()
    kp = np.zeros(len(tokens), dtype=np.uint8) if keep is None else np.asarray(keep, dtype=np.uint8).copy()
    return blob, off, sc, kp


def pack_samples(samples: Sequence[bytes]):
    lens = np.fromiter((len(t) for t in samples), dtype=np.uint64, count=len(samples))
    off = np.zeros(len(samples) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b"".join(samples), dtype=np.uint8).copy()
    if blob.size == 0:
        blob = np.zeros(1, np.uint8)
    return blob, off


class NoPath(Exception):
    def __init__(self, pos: int, length: int):
        super().__init__(f"no path to position {pos}/{length}")  # src/lib.rs:243-245
        self.pos, self.length = pos, length


class OracleModel:
    """Model (src/model.rs) + the prune.rs functions, CPU."""

    def __init__(self, tokens: Sequence[bytes] = (), scores: Sequence[float] = (),
                 keep: Optional[Sequence[bool]] = None, _handle=None):
        L = lib()
        if _handle is not None:
            self._h = _handle
        else:
            blob, off, sc, kp = pack_vocab(tokens, scores, keep)
            self._h = L.orc_model_create(_p(blob, u8p), _p(off, u64p), _p(sc, f64p), _p(kp, u8p), len(tokens))
        self.V = int(L.orc_model_vocab_size(self._h))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().orc_model_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # -- vocab -------------------------------------------------------------
    def export(self) -> Tuple[List[bytes], np.ndarray, np.ndarray]:
        L = lib()
        nb = int(L.orc_model_vocab_bytes(self._h))
        blob = np.zeros(max(nb, 1), np.uint8)
        off = np.zeros(self.V + 1, np.uint64)
        sc = np.zeros(self.V, np.float64)
        kp = np.zeros(self.V, np.uint8)
        L.orc_model_export(self._h, _p(blob, u8p), _p(off, u64p), _p(sc, f64p), _p(kp, u8p))
        raw = blob.tobytes()
        toks = [raw[int(off[i]):int(off[i + 1])] for i in range(self.V)]
        return toks, sc, kp

    # -- encode ------------------------------------------------------------
    def encode(self, text: bytes, dropout: float = 0.0) -> List[int]:
        L = lib()
        a = _bytes_arr(text)
        n = len(text)
        out = np.zeros(max(n, 1), np.uint32)
        err = np.zeros(2, np.uint64)
        k = L.orc_encode(self._h, _p(a, u8p), n, dropout, _p(out, u32p), out.size, _p(err, u64p))
        if k == -1:
            raise NoPath(int(err[0]), int(err[1]))
        assert k >= 0
        return out[:k].tolist()

    def encode_keyed(self, text: bytes, dropout: float, seed: int, sample: int) -> List[int]:
        """Model::encode with the product's keyed dropout draw (tgx_model_set_dropout): `sample` is the index of
        `text` in the call, positions are bytes of the processed text."""
        L = lib()
        a = _bytes_arr(text)
        n = len(text)
        out = np.zeros(max(n, 1), np.uint32)
        err = np.zeros(2, np.uint64)
        k = L.orc_encode_keyed(self._h, _p(a, u8p), n, dropout, seed & 0xFFFFFFFFFFFFFFFF, sample, _p(out, u32p),
                               out.size, _p(err, u64p))
        if k == -1:
            raise NoPath(int(err[0]), int(err[1]))
        assert k >= 0
        return out[:k].tolist()

    def encode_batch(self, blob: np.ndarray, off: np.ndarray, crlf: bool = False, threads: int = 1):
        """→ (ids u32[T], id_off u64[S+1], status i32[S], proc_len u64[S], first_bad)"""
        L = lib()
        S = len(off) - 1
        cap = int(off[-1]) - int(off[0]) + 1
        ids = np.zeros(cap, np.uint32)
        id_off = np.zeros(S + 1, np.uint64)
        status = np.zeros(max(S, 1), np.int32)
        plen = np.zeros(max(S, 1), np.uint64)
        bad = L.orc_encode_batch(self._h, _p(blob, u8p), _p(off, u64p), S, int(crlf), threads,
                                 _p(ids, u32p), cap, _p(id_off, u64p), _p(status, i32p), _p(plen, u64p))
        return ids[:int(id_off[S])], id_off, status[:S], plen[:S], int(bad)

    def common_prefix_search(self, text: bytes):
        L = lib()
        a = _bytes_arr(text)
        ids = np.zeros(max(len(text), 1), np.uint32)
        lens = np.zeros(max(len(text), 1), np.uint32)
        k = L.orc_common_prefix_search(self._h, _p(a, u8p), len(text), _p(ids, u32p), _p(lens, u32p), ids.size)
        return ids[:k].tolist(), lens[:k].tolist()

    # -- forward-backward ----------------------------------------------------
    def marginal(self, text: bytes, literal: bool = True):
        L = lib()
        a = _bytes_arr(text)
        ex = np.zeros(self.V, np.float64)
        z = L.orc_marginal(self._h, _p(a, u8p), len(text), _p(ex, f64p), int(literal))
        return float(z), ex

    def alpha_beta(self, text: bytes):
        L = lib()
        a = _bytes_arr(text)
        A = np.zeros(len(text) + 1)
        B = np.zeros(len(text) + 1)
        z = L.orc_alpha_beta(self._h, _p(a, u8p), len(text), _p(A, f64p), _p(B, f64p))
        return float(z), A, B

    def run_e_step(self, blob: np.ndarray, off: np.ndarray, threads: int = 1, literal: bool = False,
                   max_sample_length: int = 81920):
        L = lib()
        ex = np.zeros(self.V, np.float64)
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = L.orc_run_e_step(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads, int(literal),
                              max_sample_length, _p(ex, f64p), C.byref(bad), C.byref(badz))
        return ex, rc, int(bad.value), float(badz.value)

    def run_e_step_dropout(self, blob: np.ndarray, off: np.ndarray, dropout: float, seed: int, keyed: bool = True,
                           byte_base: int = 0, threads: int = 1, max_sample_length: int = 81920):
        """run_e_step with populate_nodes(.., dropout): keyed = the product's draw (tgx_model_set_dropout), else a
        sequential seeded generator in the reference's loop order."""
        L = lib()
        ex = np.zeros(self.V, np.float64)
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = L.orc_run_e_step_dropout(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads,
                                      max_sample_length, dropout, int(keyed), seed & 0xFFFFFFFFFFFFFFFF, byte_base,
                                      _p(ex, f64p), C.byref(bad), C.byref(badz))
        return ex, rc, int(bad.value), float(badz.value)

    def run_e_step_fixed(self, blob: np.ndarray, off: np.ndarray, dropout: float = 0.0, seed: int = 0,
                         keyed: bool = True, byte_base: int = 0, threads: int = 1, max_sample_length: int = 81920):
        """run_e_step (dropout 0) or run_e_step_dropout with exact sums: → (counts, rc, bad_sample), counts[id] = the
        Python int sum(floor(c * 2^128)) over token id's contributions c."""
        L = lib()
        fx = np.zeros((max(self.V, 1), 3), np.uint64)
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = L.orc_run_e_step_fixed(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads, max_sample_length,
                                    dropout, int(keyed), seed & 0xFFFFFFFFFFFFFFFF, byte_base, _p(fx, u64p),
                                    C.byref(bad), C.byref(badz))
        counts = [int(w0) | (int(w1) << 64) | (int(w2) << 128) for w0, w1, w2 in fx[:self.V].tolist()]
        return counts, rc, int(bad.value)

    def marginal_contributions(self, text: bytes, dropout: float = 0.0, seed: int = 0, byte_base: int = 0):
        """(z, [(id, contribution), ...]) of one lattice, in the order populate_marginal adds them.  dropout > 0: the
        keyed draw of run_e_step_fixed, `text` starting at byte `byte_base` of the call's text."""
        L = lib()
        a = _bytes_arr(text)
        n = C.c_uint64(0)
        args = (dropout, seed & 0xFFFFFFFFFFFFFFFF, byte_base)
        L.orc_marginal_contributions(self._h, _p(a, u8p), len(text), None, None, 0, C.byref(n), *args)
        k = int(n.value)
        ids = np.zeros(max(k, 1), np.uint32)
        vals = np.zeros(max(k, 1), np.float64)
        z = L.orc_marginal_contributions(self._h, _p(a, u8p), len(text), _p(ids, u32p), _p(vals, f64p), k,
                                         C.byref(n), *args)
        return float(z), list(zip(ids[:k].tolist(), vals[:k].tolist()))

    def run_m_step(self, expected: np.ndarray) -> "OracleModel":
        L = lib()
        rc = C.c_int(0)
        ex = np.ascontiguousarray(expected, np.float64)
        h = L.orc_run_m_step(self._h, _p(ex, f64p), C.byref(rc))
        m = OracleModel(_handle=h)
        if rc.value:
            raise FloatingPointError("M-step: alternative vocabulary contains invalid frequency")
        return m

    def token_frequencies(self, blob: np.ndarray, off: np.ndarray, threads: int = 1) -> np.ndarray:
        L = lib()
        fr = np.zeros(self.V, np.uint64)
        err = np.zeros(2, np.uint64)
        rc = L.orc_token_frequencies(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads,
                                     _p(fr, u64p), _p(err, u64p))
        if rc:
            raise NoPath(int(err[0]), int(err[1]))
        return fr

    def pair_frequencies(self, blob: np.ndarray, off: np.ndarray, threads: int = 1):
        """Pair-frequency pass of `tokengeex merge` (src/merge.rs:36-84): (pairs u32[n, 2], counts u64[n]),
        frequency-descending, ties by (first, second) ascending."""
        L = lib()
        cap = max(int(off[-1]), 1)
        pairs = np.zeros(cap, np.uint64)
        counts = np.zeros(cap, np.uint64)
        err = np.zeros(2, np.uint64)
        n = L.orc_pair_frequencies(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads, _p(pairs, u64p),
                                   _p(counts, u64p), cap, _p(err, u64p))
        if n < 0:
            raise NoPath(int(err[0]), int(err[1]))
        p = pairs[:n]
        return np.stack([(p >> np.uint64(32)).astype(np.uint32), (p & np.uint64(0xFFFFFFFF)).astype(np.uint32)], axis=1), counts[:n].copy()

    def token_alternatives(self):
        L = lib()
        ak = np.zeros(self.V, np.uint8)
        aoff = np.zeros(self.V + 1, np.uint64)
        cap = int(L.orc_model_vocab_bytes(self._h)) + 16
        aids = np.zeros(cap, np.uint32)
        n = L.orc_token_alternatives(self._h, _p(ak, u8p), _p(aoff, u64p), _p(aids, u32p), cap)
        assert n <= cap
        return ak, aoff, aids[:n]

    def nbest(self, text: bytes, n: int) -> List[List[int]]:
        L = lib()
        a = _bytes_arr(text)
        cap = (len(text) + 2) * max(n, 1) + 8
        ids = np.zeros(cap, np.uint32)
        poff = np.zeros(n + 2, np.uint64)
        k = L.orc_nbest(self._h, _p(a, u8p), len(text), n, _p(ids, u32p), _p(poff, u64p), cap)
        return [ids[int(poff[i]):int(poff[i + 1])].tolist() for i in range(k)]

    def prune_vocab(self, blob, off, target: int, shrink: float, threads: int = 1):
        L = lib()
        rc = C.c_int(0)
        audit = np.zeros(8)
        h = L.orc_prune_vocab(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads, target,
                              shrink, C.byref(rc), _p(audit, f64p))
        m = OracleModel(_handle=h)
        if rc.value:
            raise RuntimeError(f"prune_vocab failed rc={rc.value}")
        return m, audit

    def prune(self, blob, off, vocab_size: int, shrink: float = 0.8, em_subiters: int = 1, threads: int = 1):
        L = lib()
        rc = C.c_int(0)
        iters = np.zeros(4096, np.uint64)
        n_it = C.c_uint64(0)
        h = L.orc_prune(self._h, _p(blob, u8p), _p(off, u64p), len(off) - 1, threads, vocab_size, shrink,
                        em_subiters, C.byref(rc), _p(iters, u64p), iters.size, C.byref(n_it))
        m = OracleModel(_handle=h)
        if rc.value:
            raise RuntimeError(f"prune failed rc={rc.value}")
        return m, iters[:int(n_it.value)].tolist()


def crlf(text: bytes) -> bytes:
    L = lib()
    a = _bytes_arr(text)
    out = np.zeros(max(len(text), 1), np.uint8)
    k = L.orc_crlf(_p(a, u8p), len(text), _p(out, u8p))
    return out[:k].tobytes()


def digamma(x: float) -> float:
    return float(lib().orc_digamma(x))


def log_sum_exp(x: float, y: float, init: bool) -> float:
    return float(lib().orc_log_sum_exp(x, y, int(init)))
