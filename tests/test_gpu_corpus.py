"""Tokenizer.encode_corpus / tgx_encode_corpus / corpus.encode_file on the GPU: the device split of a NUL-separated
corpus (sample boundaries, strict UTF-8, compaction), the chunk pipeline around it and the files it writes, all
against load_sources + Model.encode_batch on the host-split samples."""
import json
import random

import numpy as np
import pytest

from tokengeex_b200 import _native as N
from tokengeex_b200 import cli, corpus, synth
from tokengeex_b200.tokenizer import TokenGeeXError, Tokenizer, _Processor, corpus_layout

pytestmark = pytest.mark.gpu

CRLF = [_Processor("crlf")]


def all_bytes_vocab(seed=0, missing=()):
    """Every byte 0x01-0xFF plus multi-byte tokens with \\r\\n in them: a wrong sample boundary changes the ids."""
    rng = random.Random(seed)
    toks = [bytes([b]) for b in range(1, 256) if b not in missing]
    toks += [b"\r\n", b"a\r\n", b"\r\n\r\n", b"\r\r\n", b"\n\r", b"ab", b"abc", b"zz", b"ok", b"tail", b"\xc3\xa9"]
    return toks, [-(rng.random() * 4 + 1) for _ in toks]


def reference(tmp_path, data, procs, toks, scores):
    """load_sources + pack + Model.encode_batch → (ids u32, id_off) or the ValueError text."""
    p = tmp_path / "ref.bin"
    p.write_bytes(data)
    try:
        src = cli.load_sources([f"c:{p}"], procs)[0]
    except ValueError as e:
        return None, str(e).replace(repr(str(p)), "SRC")
    m = N.Model(toks, scores, device=0)
    if not src.processed_samples:
        return np.zeros(0, np.uint32), np.zeros(1, np.uint64)
    blob, off = N.pack(src.processed_samples)
    ids, id_off, _, _, rc, _ = m.encode_batch(blob, off)
    assert rc == 0
    return ids, id_off


def run(tok, data, **kw):
    try:
        return tok.encode_corpus(data, source="SRC", dtype=np.uint32, **kw)
    except ValueError as e:
        return None, str(e).replace("'SRC'", "SRC")


SPLIT_CASES = [b"", b"\0", b"\0\0\0", b"\0\0ab\r\0\0\ncd\0\0", b"one sample, no NUL", b"\r\0\n", b"\r\r\n", b"ab\r",
               b"\0\r\n\0\r", b"abc\r\n\r\nx\0\r\n\0"]


@pytest.mark.parametrize("crlf", [False, True])
@pytest.mark.parametrize("data", SPLIT_CASES)
def test_split_semantics(tmp_path, data, crlf):
    toks, scores = all_bytes_vocab()
    procs = CRLF if crlf else []
    tok = Tokenizer(toks, scores, processors=procs)
    want_ids, want_off = reference(tmp_path, data, procs, toks, scores)
    ids, off = tok.encode_corpus(data, dtype=np.uint32)
    assert ids.tolist() == want_ids.tolist() and off.tolist() == want_off.tolist()
    ids16, off16 = tok.encode_corpus(np.frombuffer(data, np.uint8))  # default dtype: uint16 for this vocabulary
    assert ids16.dtype == np.uint16 and ids16.tolist() == want_ids.tolist() and off16.tolist() == want_off.tolist()


INVALID = [b"\xc0\x80", b"\xc1\xbf", b"\xe0\x80\x80", b"\xe0\x9f\xbf", b"\xf0\x80\x80\x80", b"\xf0\x8f\xbf\xbf",
           b"\xed\xa0\x80", b"\xed\xbf\xbf", b"\xf4\x90\x80\x80", b"\xf5\x80\x80\x80", b"\xff", b"\xfe", b"\x80",
           b"\xbf", b"a\x80\x80", b"\xe2\x82", b"\xf0\x9f\x98", b"\xc3", b"\xe2\x82\0\xac"]
VALID = [c.encode() for c in ("\u0080", "߿", "ࠀ", "￿", "\U00010000", "\U0010ffff", "﻿", "é")]


def placements(x):
    return [b"ok\0" + x + b"zz\0tail", b"ok\0zz" + x + b"zz\0tail", b"ok\0zz" + x + b"\0tail",
            b"ok\0tail\0zz" + x, b"a" * 5000 + b"\0" + x + b"zz\0tail"]


@pytest.mark.parametrize("x", INVALID + VALID)
def test_utf8(tmp_path, x):
    toks, scores = all_bytes_vocab()
    tok = Tokenizer(toks, scores)
    for i, data in enumerate(placements(x)):
        tok._dev(0.0).set_option(7, 4096 if i == 4 else 352 << 20)  # the last placement starts the second chunk
        want = reference(tmp_path, data, [], toks, scores)
        got = run(tok, data)
        if want[0] is None:
            assert got == want, (x, i)
        else:
            assert got[0].tolist() == want[0].tolist() and got[1].tolist() == want[1].tolist(), (x, i)
    tok._dev(0.0).set_option(7, 352 << 20)


def first_invalid(data: bytes):
    s = 0
    pos = 0
    for piece in data.split(b"\0"):
        if piece:
            try:
                piece.decode("utf-8")
            except UnicodeDecodeError:
                return s, pos
            s += 1
        pos += len(piece) + 1
    return -1, 0


def test_utf8_fuzz():
    rng = random.Random(1234)
    toks, scores = all_bytes_vocab()
    m = N.Model(toks, scores, device=0)
    for it in range(2000):
        n = rng.randrange(0, 24)
        b = bytes(rng.choice([rng.randrange(0x80, 0x100)] * 3 + [rng.randrange(0, 0x80)]) for _ in range(n))
        if it % 3 == 0:
            m.set_option(7, 4096)
            b = b"y" * rng.randrange(4000, 6000) + b"\0" + b
        elif it % 3 == 1:
            m.set_option(7, 352 << 20)
        want_s, want_pos = first_invalid(b)
        ids, off, rc, bad, pos = m.encode_corpus(np.frombuffer(b, np.uint8) if b else np.zeros(0, np.uint8))
        if want_s < 0:
            assert rc == 0, b
        else:
            assert rc == N.TGX_ERR_NOT_UTF8 and bad == want_s and pos == want_pos, (b, bad, pos, want_s, want_pos)


def joined(blob, off):
    """Samples joined with NUL bytes (the dataset format), and the offsets of its non-empty samples."""
    S = len(off) - 1
    lens = np.diff(off).astype(np.int64)
    data = np.zeros(int(off[-1]) + max(S - 1, 0), np.uint8)
    starts = off[:-1].astype(np.int64) + np.arange(S, dtype=np.int64)
    idx = np.repeat(starts - off[:-1].astype(np.int64), lens) + np.arange(int(off[-1]), dtype=np.int64)
    data[idx] = blob[:int(off[-1])]
    keep = lens > 0
    ne_off = np.zeros(int(keep.sum()) + 1, np.uint64)
    np.cumsum(lens[keep], out=ne_off[1:])
    return data, ne_off


@pytest.fixture(scope="module")
def big():
    blob, off = synth.corpus(3, 11, 256 << 20)
    toks, sc, _ = synth.vocab(blob, off, 11, 131072, 16, 0.05)
    data, ne_off = joined(blob, off)
    return blob, off, toks, sc, data, ne_off


@pytest.mark.parametrize("chunk", [None, 8 << 20])
@pytest.mark.parametrize("crlf", [False, True])
def test_at_size(big, chunk, crlf):
    blob, off, toks, sc, data, ne_off = big
    lens = np.diff(off)
    ne_blob = blob[:int(off[-1])][np.repeat(lens > 0, lens.astype(np.int64))] if (lens == 0).any() else blob
    m = N.Model(toks, sc, device=0)
    want_ids, want_off, _, _, rc, _ = m.encode_batch(ne_blob, ne_off, crlf=crlf)
    assert rc == 0
    tok = Tokenizer(toks, sc, processors=CRLF if crlf else [])
    if chunk:
        tok._dev(0.0).set_option(7, chunk)
    ids, id_off = tok.encode_corpus(data)
    assert ids.dtype == np.uint32
    assert np.array_equal(ids, want_ids) and np.array_equal(id_off, want_off)
    assert tok._dev(0.0).stat(11) > 0
    with pytest.raises(TokenGeeXError):  # u16 with a vocabulary above 65 536
        tok.encode_corpus(data[:1 << 20], dtype=np.uint16)


def test_u16_refused_by_the_library(big):
    _, _, toks, sc, data, _ = big
    m = N.Model(toks, sc, device=0)
    with pytest.raises(N.TgxError) as ei:
        m.encode_corpus(data[:1 << 20], dtype=np.uint16)
    assert ei.value.code == N.TGX_ERR_UNSUPPORTED


@pytest.mark.parametrize("chunk", [None, 4 << 20])
def test_separator_u16_u32(chunk):
    blob, off = synth.corpus(3, 12, 64 << 20)
    toks, sc, _ = synth.vocab(blob, off, 12, 60000, 16, 0.05)
    data, _ = joined(blob, off)
    tok = Tokenizer(toks, sc, special_tokens=["<eos>"])
    if chunk:
        tok._dev(0.0).set_option(7, chunk)
    plain, poff = tok.encode_corpus(data, dtype=np.uint32)
    sep = tok.separator_id("<eos>")
    want, woff = corpus_layout(plain, poff, sep, np.dtype(np.uint32))
    for dt in (np.uint16, np.uint32):
        ids, id_off = tok.encode_corpus(data, separator="<eos>", dtype=dt)
        assert ids.dtype == dt and np.array_equal(ids.astype(np.uint32), want) and np.array_equal(id_off, woff)
    ids16, off16 = tok.encode_corpus(data)
    assert ids16.dtype == np.uint16 and np.array_equal(ids16, plain.astype(np.uint16)) and np.array_equal(off16, poff)


def test_dropout_matches_encode_batch(tmp_path):
    blob, off = synth.corpus(3, 13, 4 << 20)
    toks, sc, _ = synth.vocab(blob, off, 13, 8000, 16, 0.05)
    data, ne_off = joined(blob, off)
    lens = np.diff(off)
    ne_blob = blob[:int(off[-1])][np.repeat(lens > 0, lens.astype(np.int64))]
    for p in (0.1, 0.5):
        tok = Tokenizer(toks, sc)
        tok.dropout_seed = 99
        tok._dev(p).set_option(7, 1 << 20)
        ids, id_off = tok.encode_corpus(data, dropout=p, dtype=np.uint32)
        m = N.Model(toks, sc, device=0)
        m.set_dropout(p, 99)
        want, woff, _, _, rc, _ = m.encode_batch(ne_blob, ne_off)
        assert rc == 0 and np.array_equal(ids, want) and np.array_equal(id_off, woff)
        m.set_dropout(0.0, 0)
        plain, _, _, _, _, _ = m.encode_batch(ne_blob, ne_off)
        assert not np.array_equal(plain, want)
    # encode_file: tiny windows write the same files as one window (the draw is keyed by the index in the file)
    src = tmp_path / "c.bin"
    data.tofile(src)
    tok = Tokenizer(toks, sc, special_tokens=["<eos>"])
    for p in (0.0, 0.3):
        outs = []
        for w in (64 << 10, 1 << 30):
            prefix = str(tmp_path / f"o{w}")
            corpus.encode_file(tok, str(src), prefix, separator="<eos>", dropout=p, dropout_seed=5, window_bytes=w)
            outs.append([open(f"{prefix}.{e}", "rb").read() for e in ("ids", "idx", "json")])
        assert outs[0] == outs[1]


def test_no_path():
    toks, scores = all_bytes_vocab(missing=(ord("q"),))
    tok = Tokenizer(toks, scores)
    samples = ["abc", "zz", "ok", "aqa", "q"]
    data = "\0\0".join(samples).encode()
    with pytest.raises(TokenGeeXError) as want:
        tok.encode_batch(samples, 0.0)
    with pytest.raises(TokenGeeXError) as got:
        tok.encode_corpus(data)
    assert str(got.value) == str(want.value) == "no path to position 3/3"
    ids, off, rc, bad, pos = tok._dev(0.0).encode_corpus(np.frombuffer(data, np.uint8))
    assert rc == N.TGX_ERR_NO_PATH and bad == 3 and pos == 3


def write_tokenizer(path, processors):
    toks, scores = all_bytes_vocab()
    toks = [t for t in toks if t < b"\x80" or t == b"\xc3\xa9"]  # UTF-8 strings only in this JSON
    toks += [c.encode() for c in "éü漢字"]
    scores = [-(i % 7) - 1.0 for i in range(len(toks))]
    vocab = [{"value": t.decode(), "score": s} for t, s in zip(toks, scores)]
    path.write_text(json.dumps({"version": "2.0", "special_tokens": ["<eos>"], "processors": processors,
                                "vocab": vocab}))
    return toks, scores


def test_cli_end_to_end(tmp_path):
    tj = tmp_path / "t.json"
    write_tokenizer(tj, [{"type": "crlf"}])
    rng = random.Random(3)
    samples = ["".join(rng.choice("ab\r\n xé漢字<eos>") for _ in range(rng.randrange(0, 60))) for _ in range(500)]
    src = tmp_path / "c.bin"
    src.write_bytes("\0".join(samples).encode())
    prefix = str(tmp_path / "out" / "p")
    assert cli.main(["encode", "-i", str(tj), "--input", str(src), "-o", prefix, "--separator", "<eos>"]) == 0
    ids, idx, meta = corpus.load_ids(prefix)
    tok = Tokenizer.from_file(str(tj))
    sep = tok.separator_id("<eos>")
    processed = [s.replace("\r\n", "\n") for s in samples if s]
    assert meta["n_samples"] == len(processed) and meta["dtype"] == "uint16" and meta["separator"]["id"] == sep
    for i, s in enumerate(processed):
        row = ids[int(idx[i]):int(idx[i + 1])].tolist()
        assert row[-1] == sep and tok.decode(row[:-1], True) == s
    # `<eos>` in the text is ordinary text: the special token's id appears only as the separator
    assert int((np.asarray(ids) == sep).sum()) == len(processed)


def test_host_path_for_other_processors(tmp_path):
    tj = tmp_path / "t.json"
    toks, scores = write_tokenizer(tj, [{"type": "unicode", "form": "nfkc"}, {"type": "crlf"}])
    rng = random.Random(4)
    samples = ["".join(rng.choice("ab\r\n xﬁ①é") for _ in range(rng.randrange(0, 40))) for _ in range(300)]
    src = tmp_path / "c.bin"
    src.write_bytes("\0".join(samples).encode())
    tok = Tokenizer.from_file(str(tj))
    assert not tok.corpus_on_device()
    prefix = str(tmp_path / "p")
    corpus.encode_file(str(tj), str(src), prefix, separator="<eos>", window_bytes=256)
    ids, idx, meta = corpus.load_ids(prefix)
    src_ = cli.load_sources([f"c:{src}"], tok._processors)[0]
    blob, off = N.pack(src_.processed_samples)
    want, woff, _, _, rc, _ = N.Model(toks, scores, device=0).encode_batch(blob, off)
    want, woff = corpus_layout(want, woff, tok.separator_id("<eos>"), np.dtype(np.uint16))
    assert rc == 0 and np.array_equal(ids, want) and np.array_equal(idx, woff)
