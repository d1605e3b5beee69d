"""ctypes binding of libtokengeex_b200.so (the C ABI in include/tokengeex_b200.h).

The library is built in-tree by ``make -C tokengeex_b200/csrc`` (or
``__graft_entry__.build()``).  There is no Python or CPU fallback: if the shared
library is missing, importing this module raises, and every compute entry point
fails with TGX_ERR_NO_DEVICE when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import weakref
import os
from typing import Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtokengeex_b200.so")

TGX_OK, TGX_ERR_INVALID, TGX_ERR_UNSUPPORTED, TGX_ERR_NO_DEVICE = 0, 1, 2, 3
TGX_ERR_CUDA, TGX_ERR_CAPACITY, TGX_ERR_NO_PATH, TGX_ERR_BAD_Z = 4, 5, 6, 7
TGX_ERR_NOT_UTF8 = 8
TGX_FLAG_CRLF = 1
SNIPPET_LEN = 8192 * 10  # MAX_SAMPLE_LENGTH, /root/reference/src/prune.rs:75

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)


class ModelInfo(C.Structure):
    _fields_ = [("vocab_size", C.c_uint64), ("max_token_len", C.c_uint32), ("trie_nodes", C.c_uint32),
                ("trie_slots", C.c_uint32), ("trie_terminals", C.c_uint32), ("device", C.c_int32)]


# every symbol include/tokengeex_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("tgx_last_error", C.c_char_p, []),
    ("tgx_model_create", C.c_int, [u8p, u64p, f64p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    ("tgx_model_destroy", None, [C.c_void_p]),
    ("tgx_model_get_info", C.c_int, [C.c_void_p, C.POINTER(ModelInfo)]),
    ("tgx_model_common_prefix_search", C.c_int, [C.c_void_p, u8p, C.c_uint64, u32p, u32p, C.c_uint64, u64p]),
    ("tgx_crlf_batch", C.c_int, [C.c_void_p, u8p, u64p, C.c_uint64, u8p, u64p]),
    ("tgx_encode_batch", C.c_int, [C.c_void_p, u8p, u64p, C.c_uint64, C.c_uint32, u32p, C.c_uint64, u64p, i32p,
                                   u64p, i64p]),
    ("tgx_encode_batch_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                       C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, u64p, i64p]),
    ("tgx_encode_corpus", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_int64, C.c_uint32,
                                    C.c_void_p, C.c_uint64, u64p, C.c_uint64, u64p, u64p, i64p, u64p]),
    ("tgx_expected_counts", C.c_int, [C.c_void_p, u8p, u64p, C.c_uint64, C.c_uint64, f64p, i64p, f64p]),
    ("tgx_expected_counts_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                          C.c_void_p, i64p, f64p]),
    ("tgx_expected_counts_fixed_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                                C.c_void_p, i64p, f64p]),
    ("tgx_counts_from_limbs_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    ("tgx_token_frequencies", C.c_int, [C.c_void_p, u8p, u64p, C.c_uint64, C.c_uint32, u64p, i64p, u64p]),
    ("tgx_token_frequencies_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                            C.c_void_p, i64p, u64p]),
    ("tgx_pair_frequencies", C.c_int, [C.c_void_p, u8p, u64p, C.c_uint64, C.c_uint32, u64p, u64p, C.c_uint64, u64p, i64p,
                                       u64p]),
    ("tgx_pair_frequencies_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                           C.c_void_p, C.c_void_p, C.c_uint64, u64p, i64p, u64p]),
    ("tgx_m_step", C.c_int, [f64p, u8p, C.c_uint64, u8p, f64p, u64p]),
    ("tgx_prune_select", C.c_int, [u8p, u64p, f64p, u8p, C.c_uint64, u64p, C.c_uint64, C.c_uint64, C.c_double,
                                   C.c_int, u32p, u64p, f64p]),
    ("tgx_model_prune_select", C.c_int, [C.c_void_p, u8p, u64p, f64p, u8p, C.c_uint64, u64p, C.c_uint64, C.c_uint64,
                                         C.c_double, C.c_int, u32p, u64p, f64p]),
    ("tgx_host_alloc", C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    ("tgx_host_free", C.c_int, [C.c_void_p]),
    ("tgx_model_last_stat", C.c_double, [C.c_void_p, C.c_int]),
    ("tgx_model_set_option", C.c_int, [C.c_void_p, C.c_int, C.c_int64]),
    ("tgx_model_rebuild", C.c_int, [C.c_void_p, u8p, u64p, f64p, C.c_uint64]),
    ("tgx_model_set_dropout", C.c_int, [C.c_void_p, C.c_double, C.c_uint64]),
]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C tokengeex_b200/csrc` "
                "(there is no Python / CPU fallback for the tokengeex_b200 hot path)")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class TgxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[tgx {code}] {msg}")
        self.code = code
        self.msg = msg


def _check(rc: int, ok: Sequence[int] = (TGX_OK,)) -> int:
    if rc not in ok:
        raise TgxError(rc, lib().tgx_last_error().decode(errors="replace"))
    return rc


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def pack(items: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """blob u8[] (>= 1 element) + offsets u64[len+1]."""
    lens = np.fromiter(map(len, items), dtype=np.uint64, count=len(items))
    off = np.zeros(len(items) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    joined = b"".join(items)
    blob = np.frombuffer(joined, dtype=np.uint8).copy() if joined else np.zeros(1, np.uint8)
    return blob, off


class Model:
    """Device-resident vocabulary: Model::from(vocab) (/root/reference/src/model.rs:16-30)."""

    def __init__(self, tokens: Sequence[bytes], scores, device: Optional[int] = 0):
        L = lib()
        blob, off = pack(tokens)
        sc = np.ascontiguousarray(scores, dtype=np.float64)
        if sc.size == 0:
            sc = np.zeros(1, np.float64)
        h = C.c_void_p()
        _check(L.tgx_model_create(_p(blob, u8p), _p(off, u64p), _p(sc, f64p), len(tokens),
                                  -1 if device is None else int(device), C.byref(h)))
        self._h = h
        self.V = len(tokens)
        self.device = -1 if device is None else int(device)

    def rebuild(self, tokens: Sequence[bytes], scores, packed=None):
        """`*model = Model::from(vocab)` in place (/root/reference/src/prune.rs:48,53): new trie, same workspaces.
        packed = pack(tokens) when the caller has it already (the EM loop packs a vocabulary once for the rebuild and
        the selection: 250k tokens take ~30 ms of Python)."""
        blob, off = packed if packed is not None else pack(tokens)
        sc = np.ascontiguousarray(scores, dtype=np.float64)
        if sc.size == 0:
            sc = np.zeros(1, np.float64)
        _check(lib().tgx_model_rebuild(self._h, _p(blob, u8p), _p(off, u64p), _p(sc, f64p), len(tokens)))
        self.V = len(tokens)

    def prune_select(self, tokens: Sequence[bytes], scores, keep, freq, n_samples: int, target: int, shrink: float,
                     threads: int = 0, packed=None):
        """prune_select() over the trie this model already holds (tokens / scores = the model's vocabulary)."""
        V = len(tokens)
        blob, off = packed if packed is not None else pack(tokens)
        sc = np.ascontiguousarray(scores, np.float64)
        kp = np.ascontiguousarray(keep, np.uint8)
        fr = np.ascontiguousarray(freq, np.uint64)
        out = np.zeros(max(V, 1), np.uint32)
        n = C.c_uint64(0)
        audit = np.zeros(8, np.float64)
        if threads <= 0:
            threads = max(1, len(os.sched_getaffinity(0)))
        _check(lib().tgx_model_prune_select(self._h, _p(blob, u8p), _p(off, u64p), _p(sc, f64p), _p(kp, u8p), V,
                                            _p(fr, u64p), n_samples, target, shrink, threads, _p(out, u32p),
                                            C.byref(n), _p(audit, f64p)))
        return out[:int(n.value)].copy(), audit

    def close(self):
        if getattr(self, "_h", None):
            lib().tgx_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- info / options --------------------------------------------------------------
    def info(self) -> ModelInfo:
        inf = ModelInfo()
        _check(lib().tgx_model_get_info(self._h, C.byref(inf)))
        return inf

    def set_option(self, key: int, value: int):
        _check(lib().tgx_model_set_option(self._h, key, value))

    def set_dropout(self, dropout: float, seed: int = 0):
        """Model::encode's dropout argument for the following encode calls (include/tokengeex_b200.h)."""
        _check(lib().tgx_model_set_dropout(self._h, float(dropout), int(seed) & 0xFFFFFFFFFFFFFFFF))

    def stat(self, what: int) -> float:
        return float(lib().tgx_model_last_stat(self._h, what))

    def common_prefix_search(self, text: bytes):
        n = len(text)
        a = np.frombuffer(text, np.uint8) if n else np.zeros(1, np.uint8)
        cap = max(n, 1)
        ids = np.zeros(cap, np.uint32)
        lens = np.zeros(cap, np.uint32)
        cnt = C.c_uint64(0)
        _check(lib().tgx_model_common_prefix_search(self._h, _p(a, u8p), n, _p(ids, u32p), _p(lens, u32p), cap,
                                                    C.byref(cnt)))
        k = int(cnt.value)
        return ids[:k].tolist(), lens[:k].tolist()

    # ---- host-buffer API ---------------------------------------------------------------
    def crlf_batch(self, blob: np.ndarray, off: np.ndarray):
        S = len(off) - 1
        out = np.zeros(max(int(off[-1]), 1), np.uint8)
        out_off = np.zeros(S + 1, np.uint64)
        _check(lib().tgx_crlf_batch(self._h, _p(blob, u8p), _p(off, u64p), S, _p(out, u8p), _p(out_off, u64p)))
        return out[:int(out_off[S])], out_off

    def encode_batch(self, blob: np.ndarray, off: np.ndarray, crlf: bool = False, ids_out: np.ndarray = None):
        """→ (ids u32[T], id_off u64[S+1], status i32[S], proc_len u64[S], rc, first_bad)"""
        S = len(off) - 1
        N = int(off[-1])
        ids = ids_out if ids_out is not None else np.empty(max(N, 1), np.uint32)
        id_off = np.zeros(S + 1, np.uint64)
        status = np.zeros(max(S, 1), np.int32)
        plen = np.zeros(max(S, 1), np.uint64)
        bad = C.c_int64(-1)
        rc = lib().tgx_encode_batch(self._h, _p(blob, u8p), _p(off, u64p), S, TGX_FLAG_CRLF if crlf else 0,
                                    _p(ids, u32p), ids.size, _p(id_off, u64p), _p(status, i32p), _p(plen, u64p),
                                    C.byref(bad))
        _check(rc, (TGX_OK, TGX_ERR_NO_PATH))
        return ids[:int(id_off[S])], id_off, status[:S], plen[:S], rc, int(bad.value)

    def encode_corpus(self, data: np.ndarray, crlf: bool = False, sample_base: int = 0, sep_id: int = -1,
                      dtype=np.uint32, ids_out: np.ndarray = None, off_out: np.ndarray = None):
        """tgx_encode_corpus over a NUL-separated corpus image (u8[n]) → (ids, id_off u64[S+1], rc, first_bad,
        bad_pos); rc is TGX_OK, TGX_ERR_NOT_UTF8 or TGX_ERR_NO_PATH (see include/tokengeex_b200.h).  ids_out / off_out:
        buffers to write into (e.g. pinned); too small ones are replaced by ones of the size the call reports."""
        dtype = np.dtype(dtype)
        n = int(data.size)
        ids = ids_out if ids_out is not None else np.empty(n + 1, dtype)
        off = off_out if off_out is not None else np.empty(n // 64 + 2, np.uint64)
        while True:
            ns, ni, bad, pos = C.c_uint64(0), C.c_uint64(0), C.c_int64(-1), C.c_uint64(0)
            rc = lib().tgx_encode_corpus(self._h, data.ctypes.data, n, TGX_FLAG_CRLF if crlf else 0, sample_base,
                                         sep_id, dtype.itemsize, ids.ctypes.data, ids.size, _p(off, u64p), off.size,
                                         C.byref(ns), C.byref(ni), C.byref(bad), C.byref(pos))
            if rc != TGX_ERR_CAPACITY:
                break
            if int(ni.value) > ids.size:
                ids = np.empty(int(ni.value), dtype)
            if int(ns.value) + 1 > off.size:
                off = np.empty(int(ns.value) + 1, np.uint64)
        _check(rc, (TGX_OK, TGX_ERR_NOT_UTF8, TGX_ERR_NO_PATH))
        S = int(ns.value)
        return ids[:int(ni.value)], off[:S + 1], rc, int(bad.value), int(pos.value)

    def expected_counts(self, blob: np.ndarray, off: np.ndarray, snippet_len: int = SNIPPET_LEN):
        """→ (expected f64[V], rc, bad_sample, bad_z)"""
        S = len(off) - 1
        ex = np.zeros(max(self.V, 1), np.float64)
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = lib().tgx_expected_counts(self._h, _p(blob, u8p), _p(off, u64p), S, snippet_len, _p(ex, f64p),
                                       C.byref(bad), C.byref(badz))
        _check(rc, (TGX_OK, TGX_ERR_BAD_Z))
        return ex[:self.V], rc, int(bad.value), float(badz.value)

    def token_frequencies(self, blob: np.ndarray, off: np.ndarray, crlf: bool = False):
        """→ (freq u64[V], rc, first_bad, bad_len)"""
        S = len(off) - 1
        fr = np.zeros(max(self.V, 1), np.uint64)
        bad = C.c_int64(-1)
        blen = C.c_uint64(0)
        rc = lib().tgx_token_frequencies(self._h, _p(blob, u8p), _p(off, u64p), S, TGX_FLAG_CRLF if crlf else 0,
                                         _p(fr, u64p), C.byref(bad), C.byref(blen))
        _check(rc, (TGX_OK, TGX_ERR_NO_PATH))
        return fr[:self.V], rc, int(bad.value), int(blen.value)

    def pair_frequencies(self, blob: np.ndarray, off: np.ndarray, crlf: bool = False, cap: int = 0):
        """Pair-frequency pass of `tokengeex merge` (/root/reference/src/merge.rs:36-84)
        → (pairs u32[n, 2], counts u64[n], rc, first_bad, bad_len); count-descending, ties by ids ascending."""
        S = len(off) - 1
        cap = int(cap) or max(1, min(int(off[-1]), 1 << 22))
        while True:
            pairs = np.zeros(cap, np.uint64)
            counts = np.zeros(cap, np.uint64)
            n = C.c_uint64(0)
            bad = C.c_int64(-1)
            blen = C.c_uint64(0)
            rc = lib().tgx_pair_frequencies(self._h, _p(blob, u8p), _p(off, u64p), S, TGX_FLAG_CRLF if crlf else 0,
                                            _p(pairs, u64p), _p(counts, u64p), cap, C.byref(n), C.byref(bad),
                                            C.byref(blen))
            if rc == TGX_ERR_CAPACITY and int(n.value) > cap:
                cap = int(n.value)
                continue
            _check(rc, (TGX_OK, TGX_ERR_NO_PATH))
            k = int(n.value)
            p = pairs[:k]
            ab = np.stack([(p >> np.uint64(32)).astype(np.uint32), (p & np.uint64(0xFFFFFFFF)).astype(np.uint32)], axis=1)
            return ab, counts[:k].copy(), rc, int(bad.value), int(blen.value)

    # ---- device-pointer API (torch tensors' data_ptr()) ---------------------------------
    def encode_batch_dev(self, d_text: int, d_off: int, S: int, n_bytes: int, crlf: bool, d_ids: int, ids_cap: int,
                         d_id_off: int, d_status: int = 0, d_proc_len: int = 0):
        tot = C.c_uint64(0)
        bad = C.c_int64(-1)
        rc = lib().tgx_encode_batch_dev(self._h, d_text, d_off, S, n_bytes, TGX_FLAG_CRLF if crlf else 0, d_ids,
                                        ids_cap, d_id_off, d_status or None, d_proc_len or None, C.byref(tot),
                                        C.byref(bad))
        _check(rc, (TGX_OK, TGX_ERR_NO_PATH))
        return int(tot.value), rc, int(bad.value)

    def expected_counts_dev(self, d_text: int, d_off: int, S: int, n_bytes: int, d_expected: int,
                            snippet_len: int = SNIPPET_LEN):
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = lib().tgx_expected_counts_dev(self._h, d_text, d_off, S, n_bytes, snippet_len, d_expected,
                                           C.byref(bad), C.byref(badz))
        _check(rc, (TGX_OK, TGX_ERR_BAD_Z))
        return rc, int(bad.value), float(badz.value)

    def expected_counts_fixed_dev(self, d_text: int, d_off: int, S: int, n_bytes: int, d_limbs: int,
                                  snippet_len: int = SNIPPET_LEN):
        """E-step with exact integer counts: d_limbs int64[5 V] += limbs (see include/tokengeex_b200.h).  → (rc, bad_sample, bad_z)"""
        bad = C.c_int64(-1)
        badz = C.c_double(0.0)
        rc = lib().tgx_expected_counts_fixed_dev(self._h, d_text, d_off, S, n_bytes, snippet_len, d_limbs, C.byref(bad),
                                                 C.byref(badz))
        _check(rc, (TGX_OK, TGX_ERR_BAD_Z))
        return rc, int(bad.value), float(badz.value)

    def counts_from_limbs_dev(self, d_limbs: int, V: int, d_expected: int):
        _check(lib().tgx_counts_from_limbs_dev(self._h, d_limbs, V, d_expected))

    def token_frequencies_dev(self, d_text: int, d_off: int, S: int, n_bytes: int, crlf: bool, d_freq: int):
        bad = C.c_int64(-1)
        blen = C.c_uint64(0)
        rc = lib().tgx_token_frequencies_dev(self._h, d_text, d_off, S, n_bytes, TGX_FLAG_CRLF if crlf else 0,
                                             d_freq, C.byref(bad), C.byref(blen))
        _check(rc, (TGX_OK, TGX_ERR_NO_PATH))
        return rc, int(bad.value), int(blen.value)

    def pair_frequencies_dev(self, d_text: int, d_off: int, S: int, n_bytes: int, crlf: bool, d_pairs: int,
                             d_counts: int, cap: int):
        """tgx_pair_frequencies_dev: the n distinct pairs ((first << 32) | second, u64[cap]) and their counts
        (u64[cap]) into device buffers, count-descending.  → (n, rc, first_bad, bad_len); rc is TGX_OK,
        TGX_ERR_NO_PATH or TGX_ERR_CAPACITY (n > cap: n = pairs needed, nothing written)."""
        n = C.c_uint64(0)
        bad = C.c_int64(-1)
        blen = C.c_uint64(0)
        rc = lib().tgx_pair_frequencies_dev(self._h, d_text, d_off, S, n_bytes, TGX_FLAG_CRLF if crlf else 0,
                                            d_pairs or None, d_counts or None, cap, C.byref(n), C.byref(bad),
                                            C.byref(blen))
        _check(rc, (TGX_OK, TGX_ERR_NO_PATH, TGX_ERR_CAPACITY))
        return int(n.value), rc, int(bad.value), int(blen.value)


def pinned_empty(nbytes: int) -> np.ndarray:
    """uint8 numpy array over cudaHostAlloc'd memory.  The allocation lives as long as the ctypes buffer every view of
    the array keeps alive through `.base`, and is released (tgx_host_free) when that buffer is collected."""
    p = C.c_void_p()
    _check(lib().tgx_host_alloc(C.byref(p), nbytes))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    weakref.finalize(buf, _free_pinned, p.value)
    return np.frombuffer(buf, dtype=np.uint8)[:nbytes]


def _free_pinned(addr: int) -> None:
    try:
        lib().tgx_host_free(C.c_void_p(addr))
    except Exception:
        pass


# ---- host half of the EM pruning loop (tokengeex_b200/csrc/prune_host.cpp) -------------------------
def m_step(expected: np.ndarray, keep: np.ndarray):
    """run_m_step → (kept mask u8[V], new_scores f64[V]); raises on NaN/inf scores."""
    V = len(expected)
    ex = np.ascontiguousarray(expected, np.float64)
    kp = np.ascontiguousarray(keep, np.uint8)
    kept = np.zeros(max(V, 1), np.uint8)
    ns = np.zeros(max(V, 1), np.float64)
    nk = C.c_uint64(0)
    rc = lib().tgx_m_step(_p(ex, f64p), _p(kp, u8p), V, _p(kept, u8p), _p(ns, f64p), C.byref(nk))
    if rc:
        raise TgxError(rc, "M-step: alternative vocabulary contains invalid frequency")
    return kept[:V], ns[:V]


def prune_select(tokens: Sequence[bytes], scores, keep, freq, n_samples: int, target: int, shrink: float,
                 threads: int = 0):
    """prune_vocab minus its frequency pass → (ids of survivors in final order u32[], audit f64[8])."""
    V = len(tokens)
    blob, off = pack(tokens)
    sc = np.ascontiguousarray(scores, np.float64)
    kp = np.ascontiguousarray(keep, np.uint8)
    fr = np.ascontiguousarray(freq, np.uint64)
    out = np.zeros(max(V, 1), np.uint32)
    n = C.c_uint64(0)
    audit = np.zeros(8, np.float64)
    if threads <= 0:
        threads = max(1, len(os.sched_getaffinity(0)))
    rc = lib().tgx_prune_select(_p(blob, u8p), _p(off, u64p), _p(sc, f64p), _p(kp, u8p), V, _p(fr, u64p), n_samples,
                                target, shrink, threads, _p(out, u32p), C.byref(n), _p(audit, f64p))
    if rc:
        raise TgxError(rc, "prune_vocab failed (loss is not normal, or vocabulary unsupported)")
    return out[:int(n.value)].copy(), audit
