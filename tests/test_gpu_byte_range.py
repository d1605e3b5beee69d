"""Every device path over the whole byte range, against the CPU oracle.

The other device tests draw their text from 'a'..'d' or from the synthetic corpora (ASCII and one CJK range).  Here:
NUL (a child with label 0 lands on its parent's base; the text is padded with zero bytes past the blob's end, so a token
that ends in NUL meets that padding at the last bytes of a batch), bytes above 0x7F and 0xFF (the kernels pull bytes
out of words with __byte_perm, funnel shifts and window_bytes), a root with 256 children and depth-1 nodes with 256
children each (the second trie level no longer fits the pair kernel's shared-memory stage; every entry of
match2_kernel's two-byte table is used), ids of 65 536 and above, text whose start and end take every alignment, and a
mixed-script UTF-8 corpus.  Encode is compared bit for bit (ids, offsets, status, processed length, return code,
first failing sample), the frequency passes exactly and the E-step's fixed-point limbs to the last bit.
"""
import random

import numpy as np
import pytest

from oracle import oracle as O
from tests.test_gpu_exact_counts import KERNEL_SETS, assert_limbs_equal, configure, limbs_to_ints, run_fixed
from tests.util import (BYTE_ALPHABETS, byte_samples, byte_vocab, fixed_point_samples, mixed_script_setup,
                        rand_samples, split_ids, wide_samples, wide_vocab)

pytestmark = pytest.mark.gpu

SNIP = 81920
ALL = 1 << 30


@pytest.fixture(scope="module")
def N():
    from tokengeex_b200 import _native
    return _native


def assert_encode_equal(N, got, want, ctx=None):
    ids, id_off, status, plen, rc, bad = got
    wids, wid_off, wstatus, wplen, wbad = want
    first = wbad - 1  # the oracle returns the lowest failing index + 1, or 0
    assert np.array_equal(id_off, wid_off) and np.array_equal(ids, wids), ctx
    assert np.array_equal(status, np.where(wstatus != 0, N.TGX_ERR_NO_PATH, 0)), ctx
    assert np.array_equal(plen, wplen), ctx
    assert bad == first and rc == (N.TGX_ERR_NO_PATH if first >= 0 else N.TGX_OK), (ctx, rc, bad, first)


def check_batch(N, gm, om, samples, crlf=False, ctx=None):
    blob, off = N.pack(samples)
    assert_encode_equal(N, gm.encode_batch(blob, off, crlf=crlf), om.encode_batch(blob, off, crlf=crlf, threads=8), ctx)


def set_options(gm, opts):
    for k, v in opts.items():
        gm.set_option(k, v)


# forward pass (option 3) with what it reads: 37 match2_kernel / match_kernel, 13 / 14 the pair kernel's staged trie
# levels and shape, 16 emit through the token hash or a second trie walk, 32 the team / pair-kernel split of forward
# pass 3, 24 / 26 / 35 bytes of trie / row table staged in shared memory (0 and everything)
ENCODE_CONFIGS = [
    {3: 0, 37: 1, 16: 1, 24: 0, 26: 0},
    {3: 0, 37: 0, 16: 0, 24: ALL, 26: ALL},
    {3: 1, 16: 1},
    {3: 1, 16: 0, 0: 8, 1: 64},
    {3: 2, 13: 0, 14: 1, 16: 1},
    {3: 2, 13: 1, 14: 2, 16: 0},
    {3: 2, 13: 2, 14: 1, 16: 1},
    {3: 2, 13: 2, 14: 2, 16: 0},
    {3: 3, 32: ALL, 37: 1, 35: 0},
    {3: 3, 32: 1, 37: 0, 35: ALL, 16: 0},
    {3: 3, 32: 150, 37: 1, 35: ALL, 24: 0},
    {3: 3, 32: 150, 37: 0, 35: 0, 24: ALL, 16: 0},
    {3: 4},
]


def cfg_id(c):
    return "-".join(f"{k}={'all' if v == ALL else v}" for k, v in c.items())


@pytest.fixture(scope="module")
def byte_cases():
    """(name, tokens, scores, samples) over every alphabet: complete and incomplete vocabularies, float and integer
    scores, the hand-placed NUL / 0xFF tokens; one vocabulary per alphabet has tokens longer than 16 bytes."""
    rng = random.Random(2401)
    cases = []
    for name, alphabet in BYTE_ALPHABETS.items():
        for it in range(4):
            toks, scores = byte_vocab(rng, alphabet, n_tok=rng.randrange(20, 300), max_len=rng.randrange(2, 17),
                                      complete=(it != 2), int_scores=(it % 2 == 1), long=(it == 3))
            cases.append((f"{name}-{it}", toks, scores, byte_samples(rng, alphabet, toks)))
    return cases


@pytest.mark.parametrize("cfg", ENCODE_CONFIGS, ids=cfg_id)
def test_encode_byte_alphabets(N, byte_cases, cfg):
    """Every forward pass and emit path on the byte alphabets.  The batch ends in a sample that ends in NUL, or in the
    one-byte sample b"x" while b"x\\x00" and b"x\\x00\\x00" are tokens (the walk at the blob's last byte reads the zero
    padding); short samples at the end of the batch put the blob's last bytes at every offset."""
    for name, toks, scores, samples in byte_cases:
        gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
        set_options(gm, cfg)
        for tail in ([b"a\x00"], [b"x"], [b"\xff" * 7 + b"x\x00"], [b"x", b"\x00"]):
            check_batch(N, gm, om, samples + tail, ctx=(name, tail))


def test_nul_without_nul_tokens_is_nopath(N):
    """NUL in the text and no token with a NUL byte in it: NoPath with the sample's length, the lowest failing index
    reported, the other samples encoded.  (A NUL probe from a root whose base is 0 lands on the root's own slot.)"""
    rng = random.Random(2402)
    for it in range(4):
        toks, scores = byte_vocab(rng, BYTE_ALPHABETS["high"], n_tok=rng.randrange(130, 400), max_len=8,
                                  complete=True, int_scores=(it % 2 == 0), edges=False)
        gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
        samples = byte_samples(rng, BYTE_ALPHABETS["high"], toks, n=30)
        samples = [s for s in samples if 0 not in s]
        samples[5:5] = [b"\x80\x00", b"\x00" + toks[0], b"\x00", toks[1] + b"\x00" + toks[2]]
        for cfg in ENCODE_CONFIGS:
            set_options(gm, cfg)
            check_batch(N, gm, om, samples, ctx=(it, cfg))
            check_batch(N, gm, om, samples[7:] + [b"\xfe\x00"], ctx=(it, cfg, "last"))
        fr, rc, bad, blen = gm.token_frequencies(*N.pack(samples))
        assert rc == N.TGX_ERR_NO_PATH and bad == 5 and blen == 2


def test_token_hash_keys_on_length(N):
    """b"a" and b"a\\x00" (and b"x", b"x\\x00", b"x\\x00\\x00"): the same bytes as a 16-byte word padded with zeros,
    so the emit's token hash must key on the length as well (a model whose hash cannot be built is refused at creation).
    Every emit path must give each its own id."""
    toks = [b"a", b"a\x00", b"\x00", b"x", b"x\x00", b"x\x00\x00", b"\x00" * 16, b"a" + b"\x00" * 15]
    scores = [-1.0, -1.5, -4.0, -2.0, -2.5, -2.25, -3.0, -2.0]
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    samples = [b"a", b"a\x00", b"x\x00\x00", b"x\x00", b"\x00" * 16, b"a" + b"\x00" * 15, b"a" + b"\x00" * 40, b"x"]
    for cfg in ENCODE_CONFIGS:
        set_options(gm, cfg)
        check_batch(N, gm, om, samples, ctx=cfg)
    gm.set_option(16, 1)
    ids, id_off, *_ = gm.encode_batch(*N.pack([b"a", b"a\x00", b"x\x00\x00"]))
    assert split_ids(ids, id_off) == [[0], [1], [5]]


@pytest.fixture(scope="module")
def wide():
    toks, scores = wide_vocab()
    rng = random.Random(2403)
    samples = wide_samples(rng, toks)
    return list(toks), list(scores), samples


@pytest.mark.parametrize("cfg", ENCODE_CONFIGS, ids=cfg_id)
def test_encode_wide_vocabulary(N, wide, cfg):
    """All 65 536 two-byte tokens and 3 000 longer ones: the pair kernel falls back to one staged level, every entry of
    the two-byte table is read, ids above 65 535."""
    toks, scores, samples = wide
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    set_options(gm, cfg)
    check_batch(N, gm, om, samples + [b"\x00\xff\x00"], ctx=cfg)
    ids, *_ = gm.encode_batch(*N.pack(samples))
    assert int(ids.max()) >= 65536


def test_encode_lengths_at_every_residue(N):
    """Total lengths at every residue mod 24 (load_window reads 24 bytes from an 8-byte aligned address and takes a byte
    path for the blob's last 24 bytes), for the forward passes over the match stream and the pair kernel."""
    rng = random.Random(2404)
    toks, scores = byte_vocab(rng, BYTE_ALPHABETS["edges"], n_tok=120, max_len=9, int_scores=True)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    head = byte_samples(rng, BYTE_ALPHABETS["edges"], toks, n=10, hi=50)
    n0 = sum(map(len, head))
    for cfg in ({3: 0, 37: 1}, {3: 3, 37: 0, 32: ALL}, {3: 2}, {3: 1}):
        set_options(gm, cfg)
        for k in range(24):
            pad = (k - n0) % 24 + 24
            for last in (b"x", b"\x00"):
                tail = bytes(rng.choice(b"\x00\xffx") for _ in range(pad - len(last))) + last
                check_batch(N, gm, om, head + [tail], ctx=(cfg, k, last))


def test_long_samples_full_range(N):
    """Samples around 16 bytes, 64 KiB (forward pass 3 puts samples of at least option 32 bytes, default 65 536, on the
    pair kernel) and 81 920 bytes (the E-step's snippet length), over all 256 bytes."""
    rng = random.Random(2405)
    toks, scores = byte_vocab(rng, BYTE_ALPHABETS["all"], n_tok=3000, max_len=8)
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    lens = (15, 16, 17, 65535, 65536, 65537, SNIP - 1, SNIP, SNIP + 1, 3)
    samples = [bytes(rng.randrange(256) for _ in range(n)) for n in lens]
    samples[4] = samples[4][:-1] + b"\x00"
    for cfg in ({3: 3}, {3: 3, 32: 70000}, {3: 2}, {3: 0}, {3: 1}, {3: 4}):
        set_options(gm, cfg)
        check_batch(N, gm, om, samples, ctx=cfg)
        check_batch(N, gm, om, samples[:-1] + [b"x\x00"], ctx=(cfg, "nul"))
    blob, off = N.pack(samples)
    gm.set_option(3, 4)
    limbs = limbs_to_ints(run_fixed(gm, blob, off), len(toks))
    want, rc, _ = om.run_e_step_fixed(blob, off, threads=8)
    assert rc == 0
    assert_limbs_equal(limbs, want)


def test_host_chunks_and_device_alignments(N, byte_cases):
    """The chunked host entry point (option 7) and encode_batch_dev with the text at byte offsets 0..7 of a larger
    device allocation: the blob's first and last bytes take every alignment."""
    import torch
    name, toks, scores, samples = byte_cases[2]  # over all 256 bytes, incomplete: NoPath samples in several chunks
    gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
    rng = random.Random(2406)
    samples = samples + rand_samples(rng, BYTE_ALPHABETS["all"], 300, 0, 400) + [b"x"]
    blob, off = N.pack(samples)
    want = om.encode_batch(blob, off, threads=8)
    for chunk in (4096, 5000, 40_000):
        gm.set_option(7, chunk)
        assert_encode_equal(N, gm.encode_batch(blob, off), want, chunk)
    gm.set_option(7, 1 << 28)
    S, n = len(off) - 1, int(off[-1])
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    for cfg in ({3: 0}, {3: 2}, {3: 3, 32: 300}, {3: 1}):
        set_options(gm, cfg)
        for k in range(8):
            buf = torch.full((n + 64,), 0x5A, dtype=torch.uint8, device="cuda")
            buf[k:k + n] = torch.from_numpy(blob[:n]).cuda()
            d_ids = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
            d_id_off = torch.zeros(S + 1, dtype=torch.int64, device="cuda")
            d_st = torch.zeros(S, dtype=torch.int32, device="cuda")
            d_pl = torch.zeros(S, dtype=torch.int64, device="cuda")
            tot, rc, bad = gm.encode_batch_dev(buf.data_ptr() + k, d_off.data_ptr(), S, n, False, d_ids.data_ptr(),
                                               n + 1, d_id_off.data_ptr(), d_st.data_ptr(), d_pl.data_ptr())
            got = (d_ids.cpu().numpy().view(np.uint32)[:tot], d_id_off.cpu().numpy().view(np.uint64),
                   d_st.cpu().numpy(), d_pl.cpu().numpy().view(np.uint64), rc, bad)
            assert_encode_equal(N, got, want, (cfg, k))


@pytest.mark.parametrize("algo", [1, 2, 3, 4])
def test_dropout_encode_full_range(N, wide, byte_cases, algo):
    """The keyed dropout draw (pair kernel with the draw in its producers, one staged trie level when it fits, else
    none; lane-group kernels for longer tokens) against the oracle's keyed encode, on the byte alphabets and the wide
    vocabulary."""
    rng = random.Random(2407 + algo)
    cases = [c[1:] for c in byte_cases[::3]] + [wide]
    for ci, (toks, scores, samples) in enumerate(cases):
        gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
        gm.set_option(3, algo)
        samples = samples[:60] + [b"x\x00"]
        blob, off = N.pack(samples)
        for p, seed in ((0.3, ci), (0.8, 2 ** 63 + rng.randrange(1 << 20))):
            gm.set_dropout(p, seed)
            ids, id_off, status, plen, rc, bad = gm.encode_batch(blob, off)
            got = split_ids(ids, id_off)
            first = -1
            for i, s in enumerate(samples):
                try:
                    want = om.encode_keyed(s, p, seed, i)
                    assert status[i] == 0 and got[i] == want, (ci, p, i)
                except O.NoPath as e:
                    assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == e.length, (ci, p, i)
                    first = i if first < 0 else first
            assert bad == first and (rc == 0) == (first < 0)
        gm.set_dropout(0.0, 0)


def test_frequency_passes_full_range(N, wide, byte_cases):
    """The token-frequency and pair-frequency passes against the oracle on the wide vocabulary and on the complete
    byte vocabularies (the frequency pass through forward pass 3 as well)."""
    cases = [c[1:] for c in byte_cases if not c[0].endswith("-2")] + [wide]
    for ci, (toks, scores, samples) in enumerate(cases):
        gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
        blob, off = N.pack(samples + [b"x\x00"])
        want = om.token_frequencies(blob, off, threads=8)
        for cfg in ({3: 4}, {3: 3, 32: 150}):
            set_options(gm, cfg)
            fr, rc, bad, blen = gm.token_frequencies(blob, off)
            assert rc == 0 and np.array_equal(fr, want), (ci, cfg)
        pairs, counts, rc, bad, blen = gm.pair_frequencies(blob, off)
        wp, wc = om.pair_frequencies(blob, off, threads=8)
        assert rc == 0 and np.array_equal(pairs, wp) and np.array_equal(counts, wc), ci


# ----------------------------------------------------------------------------- E-step
@pytest.fixture(scope="module")
def estep_cases(byte_cases, wide):
    """Byte-alphabet vocabularies (incomplete ones keep only the samples fixed_point_samples accepts) and the wide
    vocabulary, with the oracle's exact sums."""
    rng = random.Random(2408)
    cases = []
    for i, (name, toks, scores, samples) in enumerate(byte_cases[::3]):
        om = O.OracleModel(toks, scores)
        snip = [SNIP, 64, 7][i % 3]
        samples = fixed_point_samples(om, [s for s in samples if s] + [b"x\x00", b"\x00" * 20], snip)
        assert samples
        blob, off = O.pack_samples(samples)
        want, rc, _ = om.run_e_step_fixed(blob, off, threads=8, max_sample_length=snip)
        assert rc == 0
        cases.append((name, toks, scores, blob, off, snip, want))
    toks, scores, samples = wide
    blob, off = O.pack_samples([s for s in samples if s] + [bytes(rng.randrange(256) for _ in range(5000))])
    want, rc, _ = O.OracleModel(toks, scores).run_e_step_fixed(blob, off, threads=8)
    assert rc == 0
    cases.append(("wide", toks, scores, blob, off, SNIP, want))
    return cases


@pytest.mark.parametrize("g", KERNEL_SETS)
def test_estep_limbs_full_range(N, estep_cases, g):
    for name, toks, scores, blob, off, snip, want in estep_cases:
        gm = N.Model(toks, scores, device=0)
        configure(gm, g)
        assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off, snip=snip), len(toks)), want, (g, name))


@pytest.mark.parametrize("g", KERNEL_SETS)
def test_estep_keyed_dropout_full_range(N, byte_cases, wide, g):
    """Keyed dropout with a byte base (option 22) on complete byte vocabularies and the wide one."""
    cases = [c[1:] for c in byte_cases if c[0].endswith("-0") or c[0].endswith("-3")][:4] + [wide]
    for ci, (toks, scores, samples) in enumerate(cases):
        om, gm = O.OracleModel(toks, scores), N.Model(toks, scores, device=0)
        blob, off = O.pack_samples([s for s in samples if s][:50] + [b"x\x00"])
        p, seed, base, snip = [(0.3, 11, 0, SNIP), (0.7, 2 ** 62 + 5, 123457, 300)][ci % 2]
        want, rc, _ = om.run_e_step_fixed(blob, off, p, seed, keyed=True, byte_base=base, threads=8,
                                          max_sample_length=snip)
        assert rc == 0
        gm.set_option(22, base)
        gm.set_dropout(p, seed)
        configure(gm, g)
        assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off, snip=snip), len(toks)), want, (ci, g))


def test_estep_placement_options_bit_identical(N, estep_cases):
    """Option 18 (lane blocks per SM), options 30 / 31 (cuts between the lane snippet groups) and options 20 / 21
    (hot-id replicas) place work and accumulators; the limbs must not move by one bit."""
    for name, toks, scores, blob, off, snip, want in estep_cases[-2:]:
        gm = N.Model(toks, scores, device=0)
        for opts in ({18: 1}, {18: 16}, {18: 0, 30: 0, 31: 0}, {30: 1000, 31: 1000}, {30: 700, 31: 200},
                     {30: 1, 31: 999}, {20: 1, 21: 0}, {20: 4096, 21: 1 << 20}, {20: 7, 21: 3}):
            set_options(gm, opts)
            assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off, snip=snip), len(toks)), want, (name, opts))


# ----------------------------------------------------------------------------- crlf, Python surface, corpus
def test_crlf_full_range(N):
    """crlf_batch and encode_batch(crlf=True) on the CR / LF / NUL / 0xFF alphabet with tokens that contain \\r, \\n and
    \\r\\n."""
    rng = random.Random(2409)
    alphabet = BYTE_ALPHABETS["crlf"]
    samples = byte_samples(rng, alphabet, [b"\r\n", b"\r\r", b"\n\r"], n=80, hi=3000)
    samples += [b"\r", b"\n", b"\r\n", b"\x00\r\n\x00", b"\xff\r", b"\r\n\xff", b"\r" * 40 + b"\n", b"a\r"]
    blob, off = N.pack(samples)
    m = N.Model([b"a"], [-1.0], device=0)
    out, out_off = m.crlf_batch(blob, off)
    for i, s in enumerate(samples):
        assert out[int(out_off[i]):int(out_off[i + 1])].tobytes() == O.crlf(s) == s.replace(b"\r\n", b"\n"), i
    for it in range(3):
        toks, scores = byte_vocab(rng, alphabet, n_tok=80, max_len=6, int_scores=(it == 1))
        toks += [t for t in (b"\r\n", b"a\r\n", b"\r\n\r\n", b"\r\r\n", b"\n\r", b"\r\x00", b"\n\xff") if t not in toks]
        scores += [-2.0] * (len(toks) - len(scores))
        gm, om = N.Model(toks, scores, device=0), O.OracleModel(toks, scores)
        for cfg in ({3: 4}, {3: 0}, {3: 3, 32: 1000}, {3: 1}):
            set_options(gm, cfg)
            check_batch(N, gm, om, samples + [b"x\r\n\r"], crlf=True, ctx=(it, cfg))


def test_tokenizer_non_utf8_base_tokens():
    """tokengeex.Tokenizer from JSON whose base tokens are not UTF-8 (the base64 "encoded" form): every single byte,
    NUL and 0xFF tokens, pieces of multi-byte characters.  Strings with "\\x00" and astral characters encode like the
    oracle, and decode(.., True) gives them back."""
    import base64
    import json
    import tokengeex
    samples, toks, scores = mixed_script_setup()
    toks = list(toks) + [b"\x00\x00", b"\x00\xf0\x9f", b"\xff\xff", b"\x98\x80", b"x\x00"]
    scores = list(scores) + [-5.0, -6.0, -7.0, -6.5, -4.0]
    vocab = []
    for t, s in zip(toks, scores):
        try:
            vocab.append({"value": t.decode("utf-8"), "score": s})
        except UnicodeDecodeError:
            vocab.append({"value": base64.b64encode(t).decode().rstrip("="), "score": s, "encoded": True})
    js = json.dumps({"version": "2.0", "special_tokens": [], "processors": [], "vocab": vocab})
    tok = tokengeex.Tokenizer.from_str(js)
    assert tok.base_vocab_size() == len(toks) and all(tok.id_to_base_token(i)[0] == t for i, t in enumerate(toks))
    om = O.OracleModel(toks, scores)
    texts = [s.decode("utf-8") for s in samples[:60]]
    texts += ["\x00", "x\x00", "\x00\U0001f600\x00", "\U0010ffff" * 5, "a\x00b\x00\x00", "�\x00\U00010000", ""]
    got = tok.encode_batch(texts, 0.0)
    for t, ids in zip(texts, got):
        assert ids == om.encode(t.encode("utf-8"), 0.0), t
        assert tok.decode(ids, True) == t


def test_encode_corpus_mixed_script(N, wide):
    """encode_corpus over the NUL-separated mixed-script corpus equals encode_batch of its samples; uint16 ids with a
    vocabulary past 65 536 tokens are refused."""
    samples, toks, scores = mixed_script_setup()
    gm = N.Model(list(toks), list(scores), device=0)
    data = np.frombuffer(b"\x00".join(samples) + b"\x00", np.uint8).copy()
    blob, off = N.pack(list(samples))
    ids, id_off, status, plen, rc, bad = gm.encode_batch(blob, off)
    assert rc == 0
    for dtype in (np.uint32, np.uint16):
        cids, coff, crc, cbad, cpos = gm.encode_corpus(data, dtype=dtype)
        assert crc == 0 and np.array_equal(coff, id_off) and np.array_equal(cids.astype(np.uint32), ids), dtype
    wtoks, wscores, _ = wide
    gw = N.Model(wtoks, wscores, device=0)
    with pytest.raises(N.TgxError) as ei:
        gw.encode_corpus(data, dtype=np.uint16)
    assert ei.value.code == N.TGX_ERR_UNSUPPORTED
    cids, coff, crc, *_ = gw.encode_corpus(data, dtype=np.uint32)
    om = O.OracleModel(wtoks, wscores)
    wids, wid_off, wst, wplen, wbad = om.encode_batch(blob, off, threads=8)
    assert crc == 0 and wbad == 0 and np.array_equal(coff, wid_off) and np.array_equal(cids, wids)
