"""Corpus files → token ids (tokengeex_b200/corpus.py, `cli.py encode`): the host side.  CPU only: the device call is
replaced by a host stand-in that maps every byte to an id."""
import io
import json
import os

import numpy as np
import pytest

from tokengeex_b200 import _native as N
from tokengeex_b200 import cli, corpus
from tokengeex_b200.tokenizer import TokenGeeXError, Tokenizer, corpus_layout


def fake_encode(self, arr, dropout, sep_id, dt, sample_base, seed, source, ids_out=None, off_out=None):
    pieces = [p for p in arr.tobytes().split(b"\x00") if p]
    ids = np.frombuffer(b"".join(pieces), np.uint8).astype(np.uint32)
    off = np.zeros(len(pieces) + 1, np.uint64)
    np.cumsum([len(p) for p in pieces], out=off[1:])
    return corpus_layout(ids, off, sep_id, dt)


@pytest.fixture
def host_only(monkeypatch):
    monkeypatch.setattr(Tokenizer, "_encode_corpus", fake_encode)
    monkeypatch.setattr(corpus, "_pinned", lambda n: np.empty(n, np.uint8))
    monkeypatch.setattr(corpus, "_cache", {})


def byte_tokenizer(extra=(), specials=("<eos>",)):
    toks = [bytes([b]) for b in range(256)] + list(extra)
    return Tokenizer(toks, [-1.0] * len(toks), special_tokens=specials)


def test_encode_arguments(monkeypatch):
    seen = {}
    monkeypatch.setattr(cli, "encode_cmd", lambda *a: seen.setdefault("args", a))
    assert cli.main(["encode", "-i", "t.json", "--input", "c.bin", "-o", "out/p", "--separator", "<eos>", "--dtype",
                     "uint32", "--dropout", "0.1", "--dropout-seed", "7", "--device", "1", "--window-bytes", "4096"]) == 0
    assert seen["args"] == ("t.json", "c.bin", "out/p", "<eos>", "uint32", 0.1, 7, 1, 4096)
    seen.clear()
    cli.main(["encode", "-i", "t.json", "--input", "c.bin", "-o", "p"])
    assert seen["args"] == ("t.json", "c.bin", "p", None, "auto", 0.0, None, None, None)
    with pytest.raises(SystemExit):
        cli.main(["encode", "-i", "t.json", "-o", "p"])  # --input is required
    with pytest.raises(SystemExit):
        cli.main(["encode", "-i", "t.json", "--input", "c", "-o", "p", "--dtype", "int8"])


def test_dtype_auto():
    assert byte_tokenizer(specials=()).corpus_dtype() == np.uint16
    t = Tokenizer([b"%d" % i for i in range(65535)], [-1.0] * 65535, special_tokens=["<eos>"])
    assert t.vocab_size() == 65536 and t.corpus_dtype() == np.uint16
    t.add_special_tokens(["<pad>"])
    assert t.corpus_dtype() == np.uint32
    assert t.corpus_dtype("uint16") == np.uint16
    with pytest.raises(TokenGeeXError):
        t.corpus_dtype(np.int64)


def test_separator_resolution():
    t = byte_tokenizer(extra=[b"ab"])
    assert t.separator_id(None) == -1
    assert t.separator_id("<eos>") == 257
    assert t.separator_id("ab") == 256
    with pytest.raises(TokenGeeXError, match="unknown separator"):
        t.separator_id("<nope>")


def test_corpus_layout():
    ids = np.array([1, 2, 3, 4, 5], np.uint32)
    off = np.array([0, 2, 3, 5], np.uint64)
    a, o = corpus_layout(ids, off, 9, np.dtype(np.uint16))
    assert a.dtype == np.uint16 and a.tolist() == [1, 2, 9, 3, 9, 4, 5, 9] and o.tolist() == [0, 3, 5, 8]
    a, o = corpus_layout(ids, off, -1, np.dtype(np.uint32))
    assert a.tolist() == ids.tolist() and o.tolist() == off.tolist()


@pytest.mark.parametrize("window", [1, 3, 7, 64, 1 << 20])
def test_windows_end_at_nul(window, monkeypatch):
    monkeypatch.setattr(corpus, "_pinned", lambda n: np.empty(n, np.uint8))
    monkeypatch.setattr(corpus, "_cache", {})
    rng = np.random.default_rng(window)
    data = rng.integers(0, 4, 3000, dtype=np.uint8).tobytes() + b"x" * 200 + b"\0\0y"  # one sample longer than windows
    w = corpus._Windows(io.BytesIO(data), window)
    got, carry, i = [], np.zeros(0, np.uint8), 0
    while True:
        win, carry, eof = w.fill(i & 1, carry)
        got.append(win.tobytes())
        i += 1
        if eof:
            break
    assert b"".join(got) == data
    assert all(g.endswith(b"\0") for g in got[:-1])  # cut right after a NUL byte
    if window >= 3:  # windows too short for the 201-byte sample grew to hold it
        assert any(b"x" * 200 + b"\0" in g for g in got)


def test_write_read_round_trip(tmp_path, host_only):
    src = tmp_path / "c.bin"
    src.write_bytes(b"\0ab\0\0cde\0f\0")
    tj = tmp_path / "t.json"
    byte_tokenizer().save(str(tj))
    meta = corpus.encode_file(str(tj), str(src), str(tmp_path / "out" / "p"), separator="<eos>", window_bytes=4)
    ids, idx, m2 = corpus.load_ids(str(tmp_path / "out" / "p"))
    assert m2 == meta
    assert meta["dtype"] == "uint16" and meta["n_samples"] == 3 and meta["n_ids"] == 9
    assert meta["separator"] == {"token": "<eos>", "id": 256} and meta["source"] == {"name": "c.bin", "bytes": 11}
    assert meta["tokenizer_sha256"] == corpus._sha256(str(tj))
    assert ids.tolist() == [97, 98, 256, 99, 100, 101, 256, 102, 256] and idx.tolist() == [0, 3, 7, 9]
    assert not ids.flags.writeable and not idx.flags.writeable
    assert (tmp_path / "out" / "p.ids").read_bytes() == np.array(ids).astype("<u2").tobytes()
    assert sorted(os.listdir(tmp_path / "out")) == ["p.ids", "p.idx", "p.json"]
    # empty corpus
    src.write_bytes(b"\0\0")
    corpus.encode_file(str(tj), str(src), str(tmp_path / "e"), dtype="uint32")
    ids, idx, meta = corpus.load_ids(str(tmp_path / "e"))
    assert ids.size == 0 and idx.tolist() == [0] and meta["dtype"] == "uint32" and meta["separator"] is None


def test_no_partial_output_after_failure(tmp_path, monkeypatch):
    calls = []

    def failing(self, *a, **k):
        calls.append(1)
        if len(calls) == 2:
            raise ValueError("injected")
        return fake_encode(self, *a, **k)

    monkeypatch.setattr(Tokenizer, "_encode_corpus", failing)
    monkeypatch.setattr(corpus, "_pinned", lambda n: np.empty(n, np.uint8))
    monkeypatch.setattr(corpus, "_cache", {})
    src = tmp_path / "c.bin"
    src.write_bytes(b"abc\0" * 100)
    with pytest.raises(ValueError, match="injected"):
        corpus.encode_file(byte_tokenizer(), str(src), str(tmp_path / "p"), window_bytes=64)
    assert len(calls) == 2
    assert sorted(os.listdir(tmp_path)) == ["c.bin"]


def test_encode_corpus_needs_a_device():
    m = N.Model([b"a", b"b"], [-1.0, -1.0], device=None)
    data = np.frombuffer(b"ab\0a", np.uint8)
    ids = np.zeros(8, np.uint32)
    off = np.zeros(4, np.uint64)
    ns, ni, bad, pos = (N.C.c_uint64(), N.C.c_uint64(), N.C.c_int64(), N.C.c_uint64())
    rc = N.lib().tgx_encode_corpus(m._h, data.ctypes.data, 4, 0, 0, -1, 4, ids.ctypes.data, 8,
                                   off.ctypes.data_as(N.u64p), 4, N.C.byref(ns), N.C.byref(ni), N.C.byref(bad),
                                   N.C.byref(pos))
    assert rc == N.TGX_ERR_NO_DEVICE
    assert b"no CPU compute path" in N.lib().tgx_last_error()


def test_metadata_is_json(tmp_path, host_only):
    src = tmp_path / "c.bin"
    src.write_bytes(b"a\0b")
    corpus.encode_file(byte_tokenizer(), str(src), str(tmp_path / "p"), dropout=0.25, dropout_seed=5)
    meta = json.loads((tmp_path / "p.json").read_text())
    assert meta["format"] == corpus.FORMAT and meta["version"] == corpus.VERSION
    assert meta["dropout"] == 0.25 and meta["dropout_seed"] == 5
