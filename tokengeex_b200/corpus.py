"""Pretokenized corpora on disk: a NUL-separated corpus file (docs/DATASET.md:69, what `load_sources` reads) → token ids.

One corpus is three files next to each other:

    PREFIX.ids   raw little-endian uint16 / uint32 token ids, every sample's ids (and separator) back to back
    PREFIX.idx   raw little-endian uint64, n_samples + 1 entries: sample i is ids[idx[i]:idx[i + 1]]
    PREFIX.json  format name and version, dtype, n_samples, n_ids, separator, sha256 of the tokenizer, source name and
                 size, dropout and seed

`encode_file` streams the source in windows cut after a NUL byte: the next window is read into pinned memory while the
current one encodes on the GPU (Tokenizer.encode_corpus, which runs the sample split, the UTF-8 check and the encode on
the device).  The outputs are written under temporary names and renamed when the whole file is done, so a failed run
leaves no partial corpus behind.  `load_ids` maps the files back read-only.
"""
from __future__ import annotations

import hashlib
import json
import os
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import Optional, Tuple, Union

import numpy as np

from . import _native as N
from .tokenizer import Tokenizer

FORMAT = "tokengeex-b200-ids"
VERSION = 1
DEFAULT_WINDOW_BYTES = 2 << 30

_pinned = N.pinned_empty  # host buffers the copies to and from the device run at full speed from
# Pinned buffers outlive a call: pinning GBs of memory costs about as much as encoding them, so a process that encodes
# many files pins its window buffers once.  encode_file holds _lock while it uses them.
_cache = {}
_lock = threading.Lock()


def _buffer(key, nbytes: int) -> np.ndarray:
    b = _cache.get(key)
    if b is None or b.size < nbytes:
        _cache.pop(key, None)
        b = _cache[key] = _pinned(nbytes)
    return b


def _read_full(f, view: np.ndarray) -> int:
    got = 0
    mv = memoryview(view)
    while got < len(mv):
        k = f.readinto(mv[got:])
        if not k:
            break
        got += k
    return got


def _last_nul(view: np.ndarray) -> int:
    """Index of the last NUL byte in view, -1 if there is none (searched from the end in 1 MiB steps)."""
    end = view.size
    step = 1 << 20
    while end > 0:
        lo = max(0, end - step)
        z = np.flatnonzero(view[lo:end] == 0)
        if z.size:
            return lo + int(z[-1])
        end = lo
    return -1


class _Windows:
    """Windows of a file that end right after a NUL byte (the last one at the end of the file), each in one of two
    alternating host buffers.  A sample longer than the window enlarges its window."""

    def __init__(self, f, window_bytes: int):
        self.f = f
        self.window_bytes = max(1, int(window_bytes))

    def fill(self, i: int, carry: np.ndarray):
        """→ (window, carry for the next window, eof); the window lives in buffer i."""
        size = max(self.window_bytes, carry.size + 1)
        while True:
            b = _buffer(("window", i), size)
            c = carry.size
            b[:c] = carry
            got = c + _read_full(self.f, b[c:size])
            if got < size:  # end of file: the rest is the last window
                return b[:got], np.zeros(0, np.uint8), True
            last = _last_nul(b[c:got])
            if last >= 0:
                last += c
                return b[:last + 1], b[last + 1:got].copy(), False
            carry = b[:got].copy()  # no NUL after the carry: a sample longer than the window
            size *= 2


def _sha256(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 20), b""):
            h.update(block)
    return h.hexdigest()


def encode_file(tokenizer: Union[str, Tokenizer], path: str, prefix: str, separator: Optional[str] = None,
                dtype=None, dropout: float = 0.0, dropout_seed: Optional[int] = None,
                window_bytes: int = DEFAULT_WINDOW_BYTES, device: Optional[int] = None) -> dict:
    """Encodes the NUL-separated corpus at `path` into PREFIX.{ids,idx,json} and returns the metadata.
    `tokenizer`: a tokenizer JSON file (its sha256 goes into the metadata) or a Tokenizer (sha256 null).
    `dropout_seed`: seed of the keyed dropout draw (default: a fresh one, recorded in the metadata).  The draw is keyed
    by the sample's index in the file, so the ids do not depend on `window_bytes`."""
    if isinstance(tokenizer, Tokenizer):
        tok, tok_sha = tokenizer, None
    else:
        tok, tok_sha = Tokenizer.from_file(tokenizer, device=device), _sha256(tokenizer)
    if not (0.0 <= dropout < 1.0):
        raise ValueError("dropout must be in [0, 1)")
    dt = tok.corpus_dtype(dtype)
    sep_id = tok.separator_id(separator)
    if dropout_seed is None:
        import secrets
        dropout_seed = secrets.randbits(63)
    size = os.path.getsize(path)
    if not tok.corpus_on_device():
        window_bytes = max(size, 1)  # the host path keys the dropout draw by the index within one call
    window_bytes = min(window_bytes, size + 1)  # (a window buffer never needs to be larger than the file)
    tmp = {ext: f"{prefix}.{ext}.tmp{os.getpid()}" for ext in ("ids", "idx", "json")}
    d = os.path.dirname(os.path.abspath(prefix))
    os.makedirs(d, exist_ok=True)
    n_samples = n_ids = 0
    try:
        with _lock, open(path, "rb") as src, open(tmp["ids"], "wb") as fi, open(tmp["idx"], "wb") as fx, \
                ThreadPoolExecutor(1) as pool:
            windows = _Windows(src, window_bytes)
            cur = windows.fill(0, np.zeros(0, np.uint8))
            k = 0
            while True:
                window, carry, eof = cur
                nxt = None if eof else pool.submit(windows.fill, (k + 1) & 1, carry)
                ids_buf = _buffer("ids", (window.size + 1) * dt.itemsize)[:(window.size + 1) * dt.itemsize].view(dt)
                off_buf = _buffer("idx", (window.size // 64 + 2) * 8)[:(window.size // 64 + 2) * 8].view(np.uint64)
                ids, off = tok._encode_corpus(window, dropout, sep_id, dt, n_samples, dropout_seed, path, ids_buf, off_buf)
                fi.write(memoryview(np.ascontiguousarray(ids)))
                fx.write(memoryview(off[:-1] + np.uint64(n_ids)))
                n_samples += len(off) - 1
                n_ids += int(off[-1])
                if nxt is None:
                    break
                cur = nxt.result()
                k += 1
            fx.write(memoryview(np.array([n_ids], np.uint64)))
        meta = {"format": FORMAT, "version": VERSION, "dtype": dt.name, "n_samples": n_samples, "n_ids": n_ids,
                "separator": None if sep_id < 0 else {"token": separator, "id": sep_id},
                "tokenizer_sha256": tok_sha, "source": {"name": os.path.basename(path), "bytes": size},
                "dropout": dropout, "dropout_seed": dropout_seed}
        with open(tmp["json"], "w") as f:
            json.dump(meta, f, indent=1)
        for ext in ("ids", "idx", "json"):
            os.replace(tmp[ext], f"{prefix}.{ext}")
        return meta
    finally:
        for t in tmp.values():
            if os.path.exists(t):
                os.remove(t)


def load_ids(prefix: str) -> Tuple[np.ndarray, np.ndarray, dict]:
    """→ (ids, idx, metadata) with ids / idx read-only memory maps of PREFIX.ids / PREFIX.idx."""
    with open(f"{prefix}.json") as f:
        meta = json.load(f)
    if meta.get("format") != FORMAT or meta.get("version") != VERSION:
        raise ValueError(f"{prefix}.json is not a {FORMAT} v{VERSION} corpus")

    def mapped(path, dt, count):
        if count == 0:
            a = np.zeros(0, dt)
            a.flags.writeable = False
            return a
        return np.memmap(path, dtype=dt, mode="r", shape=(count,))

    ids = mapped(f"{prefix}.ids", np.dtype(meta["dtype"]).newbyteorder("<"), meta["n_ids"])
    idx = mapped(f"{prefix}.idx", np.dtype("<u8"), meta["n_samples"] + 1)
    return ids, idx, meta
