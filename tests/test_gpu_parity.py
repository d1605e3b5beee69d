"""Parity of the CUDA hot path (through the C ABI) against the CPU oracle.

Bars (BASELINE.json north_star): token ids bit-exact; token frequencies exact;
expected counts within 1e-9 relative.  All tests need a CUDA device.
"""
import math
import random

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import counts_rel_err, estep_cfg, rand_samples, rand_vocab, split_ids, synth_setup

pytestmark = pytest.mark.gpu

REL_TOL = 1e-9  # north_star: "expected counts within 1e-9 relative"
# The kernels restate glibc's exp/log bit for bit (tgx_libm.h), so alpha/beta/z and every single
# contribution equal the oracle's exactly; only the order of the f64 additions into expected[id]
# differs (atomics).  That leaves ~1e-16 * sqrt(#addends) — checked here as a stricter bound.
ORDER_TOL = 1e-12


@pytest.fixture(scope="module")
def N():
    from tokengeex_b200 import _native
    return _native


def both(N, toks, scores):
    return N.Model(toks, scores, device=0), O.OracleModel(toks, scores)


def gpu_encode(N, m, samples, crlf=False):
    blob, off = N.pack(samples)
    ids, id_off, status, plen, rc, bad = m.encode_batch(blob, off, crlf=crlf)
    return split_ids(ids, id_off), status.tolist(), plen.tolist(), rc, bad


# ----------------------------------------------------------------------------- goldens
def test_reference_goldens_encode(N):
    # /root/reference/src/model.rs:209-215
    m = N.Model([b"a", b"b", b"c", b"ab"], [-3.0, -3.0, -3.0, -4.0])
    assert gpu_encode(N, m, [b"abc"])[0] == [[3, 2]]
    # src/model.rs:218-236 with dropout 0.0
    m = N.Model([b"a", b"b", b"c", b"d", b"e", b"f", b"ab", b"abc", b"abcd", b"abcde", b"abcdef"],
                [-3.0] * 6 + [-4.0, -5.0, -6.0, -7.0, -8.0])
    assert gpu_encode(N, m, [b"abcdef"])[0] == [[10]]
    # src/model.rs:243-252: 256-byte default vocab, Chinese text
    toks = [bytes([i]) for i in range(256)]
    m = N.Model(toks, [1.0 / 256.0] * 256)
    text = "你好，我叫罗杰斯".encode()
    ids = gpu_encode(N, m, [text])[0][0]
    assert len(ids) == len(text) and bytes(ids) == text
    # tie rule (SURVEY H2): smallest start wins
    m = N.Model([b"a", b"b", b"c", b"ab", b"bc"], [-3.0, -3.0, -3.0, -4.0, -4.0])
    assert gpu_encode(N, m, [b"abc"])[0] == [[0, 4]]


def test_empty_nopath_duplicates(N):
    m = N.Model([b"a", b"ab"], [-1.0, -1.5])
    ids, status, plen, rc, bad = gpu_encode(N, m, [b"", b"ab", b"abx", b"a", b"", b"xx"])
    assert ids == [[], [1], [], [0], [], []]
    assert status == [0, 0, N.TGX_ERR_NO_PATH, 0, 0, N.TGX_ERR_NO_PATH]
    assert rc == N.TGX_ERR_NO_PATH and bad == 2 and plen[2] == 3  # NoPath(3,3)
    m = N.Model([b"ab", b"a", b"b", b"ab"], [-1.0, -5.0, -5.0, -2.0])  # last duplicate wins
    assert gpu_encode(N, m, [b"ab"])[0] == [[3]]
    # empty batch
    ids, id_off, status, plen, rc, bad = m.encode_batch(np.zeros(1, np.uint8), np.zeros(1, np.uint64))
    assert ids.size == 0 and rc == 0


@pytest.mark.parametrize("g,thr", [(1, 1 << 30), (2, 1 << 30), (4, 40), (8, 1 << 30), (16, 25), (32, 1), (8, 30)])
def test_random_small_vs_oracle(N, g, thr):
    rng = random.Random(100 + g)
    for it in range(25):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(4, 40), max_len=rng.randrange(1, 9),
                                  complete=(it % 4 != 0), int_scores=(it % 2 == 0))
        gm, om = both(N, toks, scores)
        gm.set_option(3, 1)  # lane-group kernels
        gm.set_option(0, g)
        gm.set_option(1, thr)
        samples = rand_samples(rng, b"abcd", rng.randrange(1, 70), 0, 90)
        got, status, plen, rc, bad = gpu_encode(N, gm, samples)
        for i, s in enumerate(samples):
            try:
                want = om.encode(s)
                assert status[i] == 0 and got[i] == want, (it, i, s, toks, scores)
            except O.NoPath as e:
                assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == e.length


@pytest.mark.parametrize("seed,shape", [(2, 1), (4, 1), (2, 2), (4, 2)])
def test_random_small_vs_oracle_cta(N, seed, shape):
    """CTA-cooperative producer/consumer kernel (the default path), both shapes (option 14: 5 / 6 groups per CTA)."""
    rng = random.Random(300 + seed)
    for it in range(25):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(4, 60), max_len=rng.randrange(1, 12),
                                  complete=(it % 4 != 0), int_scores=(it % 2 == 0))
        gm, om = both(N, toks, scores)
        gm.set_option(3, 2)  # pair-CTA kernel
        gm.set_option(14, shape)
        samples = rand_samples(rng, b"abcd", rng.randrange(1, 70), 0, 400)
        got, status, plen, rc, bad = gpu_encode(N, gm, samples)
        for i, s in enumerate(samples):
            try:
                want = om.encode(s)
                assert status[i] == 0 and got[i] == want, (it, i, s, toks, scores)
            except O.NoPath as e:
                assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == e.length


@pytest.mark.parametrize("seed,shape,hot", [(2, 1, 2), (4, 1, 2), (4, 2, 1), (2, 2, 0), (4, 1, 0)])
def test_pair_kernel_full_window(N, seed, shape, hot):
    """Tokens of every length 1..16 (length 16 re-uses the dp cell that is being finalised), samples that span many
    32-position tiles and rounds, sample switches inside a CTA, unreachable stretches, exact ties."""
    rng = random.Random(900 + seed)
    for it in range(12):
        alphabet = b"ab" if it % 2 == 0 else b"abc"
        toks, scores = rand_vocab(rng, alphabet=alphabet, n_tok=rng.randrange(30, 400), max_len=16,
                                  complete=(it % 3 != 0), int_scores=(it % 2 == 1))
        toks = list(toks) + [alphabet[:1] * 16, alphabet[1:2] * 16, (alphabet[:2] * 8)]
        scores = list(scores) + [-2.5, -30.0, -4.0]
        gm, om = both(N, toks, scores)
        gm.set_option(3, 2)  # pair-CTA kernel
        gm.set_option(14, shape)
        gm.set_option(13, hot)  # trie levels staged in shared memory
        samples = rand_samples(rng, alphabet, rng.randrange(3, 40), 0, 5000)
        samples += [alphabet[:1] * rng.randrange(1, 700), alphabet[1:2] * 333, alphabet[:2] * 517, b""]
        got, status, plen, rc, bad = gpu_encode(N, gm, samples)
        for i, s in enumerate(samples):
            try:
                want = om.encode(s)
                assert status[i] == 0 and got[i] == want, (it, i, len(s))
            except O.NoPath as e:
                assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == e.length


def check_against_oracle(N, gm, om, samples, ctx=None):
    got, status, plen, rc, bad = gpu_encode(N, gm, samples)
    first_bad = -1
    for i, s in enumerate(samples):
        try:
            want = om.encode(s)
            assert status[i] == 0 and got[i] == want, (ctx, i, len(s))
        except O.NoPath as e:
            assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == e.length, (ctx, i)
            if first_bad < 0:
                first_bad = i
    assert bad == first_bad and (rc == 0) == (first_bad < 0), (ctx, rc, bad, first_bad)


@pytest.mark.parametrize("stage,hot,warps,threads", [(0, 0, 1, 32), (4096, 256, 4, 256), (160 << 10, 96 << 10, 16, 1024),
                                                     (1 << 30, 1 << 30, 32, 512)])
def test_match_rows_random_vs_oracle(N, stage, hot, warps, threads):
    """The default forward pass (match_kernel + viterbi_rows_kernel, tgx_match_kernels.cuh) alone, for every staging
    split of the trie / the row table between shared memory and L2: random vocabularies incl. incomplete ones (NoPath,
    positions where no token starts, unreachable stretches), integer scores (exact ties), tokens of every length up to
    16, samples crossing many 32-position tiles, empty samples, more samples than half-warps (work fetch)."""
    rng = random.Random(1700 + warps)
    for it in range(30):
        alphabet = [b"ab", b"abcd", b"abc"][it % 3]
        toks, scores = rand_vocab(rng, alphabet=alphabet, n_tok=rng.randrange(4, 300), max_len=rng.randrange(1, 17),
                                  complete=(it % 4 != 0), int_scores=(it % 2 == 0))
        gm, om = both(N, toks, scores)
        gm.set_option(3, 0)
        gm.set_option(23, threads)
        gm.set_option(24, stage)
        gm.set_option(25, warps)
        gm.set_option(26, hot)
        samples = rand_samples(rng, alphabet, rng.randrange(1, 200), 0, 700) + rand_samples(rng, alphabet, 4, 1000, 9000)
        samples += [alphabet[:1] * k for k in (1, 15, 16, 17, 31, 32, 33, 47, 48, 49, 64, 65, 511, 512, 513, 1300)] + [b""]
        rng.shuffle(samples)
        check_against_oracle(N, gm, om, samples, it)


@pytest.mark.parametrize("match2", [1, 0])
@pytest.mark.parametrize("thr,ctas", [(1 << 30, 1), (2000, 8), (1, 64), (300, 3)])
def test_team_kernel_random_vs_oracle(N, thr, ctas, match2):
    """match2_kernel (or match_kernel, option 37) + viterbi_team_kernel (four lanes per sample, a dp cell travels through
    them: tgx_team_kernel.cuh) with the samples of at least `thr` bytes on the pair-CTA kernel beside it (option 32; 2^30 =
    everything on teams, 1 = everything on the pair kernel): random vocabularies incl. incomplete ones (NoPath, positions
    where no token starts, unreachable stretches), integer scores (exact ties), tokens of every length up to 16, sample
    starts at every alignment of the record stream, empty samples, more samples than lanes."""
    rng = random.Random(3100 + ctas)
    for it in range(30):
        alphabet = [b"ab", b"abcd", b"abc"][it % 3]
        toks, scores = rand_vocab(rng, alphabet=alphabet, n_tok=rng.randrange(4, 300), max_len=rng.randrange(1, 17),
                                  complete=(it % 4 != 0), int_scores=(it % 2 == 0))
        gm, om = both(N, toks, scores)
        gm.set_option(3, 3)
        gm.set_option(32, thr)
        gm.set_option(33, ctas)
        gm.set_option(37, match2)
        gm.set_option(39, it % 2)
        gm.set_option(38, [20, 1, 3][it % 3])
        gm.set_option(43, [4, 0, 2, 5][it % 4])
        gm.set_option(35, [160 << 10, 0, 4096, 300][it % 4])
        samples = rand_samples(rng, alphabet, rng.randrange(1, 400), 0, 700) + rand_samples(rng, alphabet, 4, 1000, 9000)
        samples += [alphabet[:1] * k for k in (1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 47, 48, 49, 64, 65, 511, 512, 513, 1300)] + [b""]
        rng.shuffle(samples)
        check_against_oracle(N, gm, om, samples, it)


def test_team_kernel_full_window(N):
    """Tokens of every length 1..16 (length 16 lands on the ring cell that was just recycled), overlapping tokens
    everywhere, long samples next to short ones in one warp."""
    rng = random.Random(3201)
    for it in range(8):
        toks = [b"a", b"b"] + [bytes(rng.choice(b"ab") for _ in range(rng.randrange(2, 17))) for _ in range(600)]
        toks = sorted(set(toks)) + [b"a" * 16, b"b" * 16, b"ab" * 8]
        scores = [-(rng.random() * 6 + 0.5) if it % 2 else -float(rng.randrange(2, 6)) for _ in toks]
        gm, om = both(N, toks, scores)
        gm.set_option(3, 3)
        gm.set_option(32, [1 << 30, 50000, 1000, 1 << 30][it % 4])
        gm.set_option(37, it % 2)
        samples = rand_samples(rng, b"ab", 30, 0, 3000) + [b"ab" * 4000, b"a" * 70000, b"aab" * 1000, b"b" * 333]
        samples += [b"a" * k for k in range(1, 20)]
        check_against_oracle(N, gm, om, samples, it)


def test_match_rows_full_window(N):
    """Tokens of every length 1..16 (length 16 lands on the cell that was just recycled), vocabularies whose tokens
    overlap everywhere, long samples, rows deeper than the staged prefix."""
    rng = random.Random(1801)
    for it in range(8):
        toks = [b"a", b"b"] + [bytes(rng.choice(b"ab") for _ in range(rng.randrange(2, 17))) for _ in range(600)]
        toks = sorted(set(toks)) + [b"a" * 16, b"b" * 16, b"ab" * 8]
        scores = [-(rng.random() * 6 + 0.5) if it % 2 else -float(rng.randrange(2, 6)) for _ in toks]
        gm, om = both(N, toks, scores)
        gm.set_option(3, 0)
        gm.set_option(26, [0, 512, 4096, 1 << 20][it % 4])
        samples = rand_samples(rng, b"ab", 30, 0, 3000) + [b"ab" * 4000, b"a" * 70000, b"aab" * 1000, b"b" * 333]
        samples += [b"a" * k for k in range(1, 20)]
        check_against_oracle(N, gm, om, samples, it)


def test_match_rows_synth_corpus(N):
    """Bench-like corpus and vocabulary: ids, offsets and processed lengths bit-exact with and without crlf, device
    entry point and chunked host entry point; the frequency pass through the same kernels; the three forward passes
    agree on a second corpus kind (code + Chinese)."""
    blob, off, toks, sc, kp = synth_setup(1, 11, 6_000_000, 32768, 16)
    gm, om = both(N, toks, sc)
    gm.set_option(3, 0)
    for crlf in (True, False):
        wids, wid_off, wstatus, wplen, wbad = om.encode_batch(blob, off, crlf=crlf, threads=8)
        for chunk in (1 << 30, 700_000):
            gm.set_option(7, chunk)
            ids, id_off, status, plen, rc, bad = gm.encode_batch(blob, off, crlf=crlf)
            assert rc == 0 and wbad == 0
            assert np.array_equal(id_off, wid_off) and np.array_equal(ids, wids) and np.array_equal(plen, wplen)
    fr, rc, bad, blen = gm.token_frequencies(blob, off)
    want = om.token_frequencies(blob, off, threads=8)
    assert rc == 0 and np.array_equal(fr, want)
    blob, off, toks, sc, kp = synth_setup(2, 12, 3_000_000, 20000, 16)
    gm = N.Model(toks, sc, device=0)
    res = []
    for algo in (0, 1, 2, 3):
        gm.set_option(3, algo)
        gm.set_option(32, 20000)
        res.append(gm.encode_batch(blob, off, crlf=True))
    for r in res[1:]:
        assert r[4] == 0 and np.array_equal(r[0], res[0][0]) and np.array_equal(r[1], res[0][1])
    # the frequency pass through the lane teams (forced: the automatic choice keeps it on the pair-CTA kernel)
    gm.set_option(3, 3)
    gm.set_option(32, 20000)
    fr, rc, bad, blen = gm.token_frequencies(blob, off)
    assert rc == 0 and np.array_equal(fr, O.OracleModel(toks, sc).token_frequencies(blob, off, threads=8))


@pytest.mark.parametrize("algo", [0, 1, 2])
def test_long_tokens(N, algo):
    """max_token_len > 16 cannot use the 16-cell windows of the pair / lane kernels: whatever forward algorithm is
    selected, the lane-group kernels take over."""
    rng = random.Random(77)
    for toks, scores in [
        ([bytes([c]) for c in b"ab"] + [b"ab" * 20, b"a" * 33, b"b" * 64, b"ba" * 7], [-3.0, -3.0, -9.0, -8.0, -20.0, -5.0]),
        ([bytes([c]) for c in b"ab"] + [b"ab" * 10, b"a" * 17, b"b" * 32, b"ba" * 7], [-3.0, -3.0, -9.0, -8.0, -20.0, -5.0]),
    ]:
        gm, om = both(N, toks, scores)
        gm.set_option(3, algo)
        samples = [b"ab" * 50, b"a" * 100, b"b" * 200, b"abba" * 30] + rand_samples(rng, b"ab", 20, 0, 300)
        check_against_oracle(N, gm, om, samples)


def test_chunked_host_entry_point(N):
    """tgx_encode_batch splits large inputs into chunks of whole samples and overlaps the copies with the kernels;
    forcing tiny chunks must not change ids, offsets, statuses, or which sample is reported as the first failure."""
    blob, off, toks, sc, kp = synth_setup(2, 31, 1_200_000, 6000, 16)
    gm, om = both(N, toks, sc)
    wids, wid_off, wstatus, wplen, wbad = om.encode_batch(blob, off, crlf=True, threads=8)
    for chunk in (4096, 100_000, 300_000, 1 << 30):
        gm.set_option(7, chunk)
        for rep in range(2):
            ids, id_off, status, plen, rc, bad = gm.encode_batch(blob, off, crlf=True)
            assert rc == 0 and np.array_equal(ids, wids) and np.array_equal(id_off, wid_off), (chunk, rep)
        assert np.array_equal(plen, wplen) and not status.any()
    # a vocabulary without some bytes: NoPath samples in several chunks; the LOWEST index is reported
    toks2 = [t for t in toks if t not in (b"e", b"{")]
    sc2 = [s for t, s in zip(toks, sc) if t not in (b"e", b"{")]
    gm2, om2 = both(N, toks2, sc2)
    wids, wid_off, wstatus, wplen, wbad = om2.encode_batch(blob, off, crlf=False, threads=8)
    gm2.set_option(7, 50_000)
    ids, id_off, status, plen, rc, bad = gm2.encode_batch(blob, off, crlf=False)
    assert np.array_equal(status != 0, wstatus != 0) and np.array_equal(id_off, wid_off) and np.array_equal(ids, wids)
    if (wstatus != 0).any():
        assert rc == N.TGX_ERR_NO_PATH and bad == int(np.flatnonzero(wstatus)[0])


def test_crlf_batch_vs_oracle(N):
    m = N.Model([b"a"], [-1.0])
    rng = random.Random(7)
    samples = [b"a\r\nb", b"\r\r\n", b"\r", b"\n", b"x\r", b"\ny", b"", b"\r\n\r\n\r", b"\r\n"]
    samples += [bytes(rng.choice(b"\r\nab") for _ in range(rng.randrange(0, 9000))) for _ in range(60)]
    blob, off = N.pack(samples)
    out, out_off = m.crlf_batch(blob, off)
    for i, s in enumerate(samples):
        assert out[int(out_off[i]):int(out_off[i + 1])].tobytes() == O.crlf(s) == s.replace(b"\r\n", b"\n"), i


def test_synth_corpus_bit_exact_with_crlf(N):
    blob, off, toks, sc, kp = synth_setup(1, 11, 6_000_000, 32768, 16)
    gm, om = both(N, toks, sc)
    wids, wid_off, wstatus, wplen, wbad = om.encode_batch(blob, off, crlf=True, threads=8)
    for algo, g, thr in [(0, 8, 32768), (2, 8, 32768), (1, 8, 32768), (1, 4, 4096), (1, 1, 2048)]:
        gm.set_option(3, algo)
        gm.set_option(0, g)
        gm.set_option(1, thr)
        ids, id_off, status, plen, rc, bad = gm.encode_batch(blob, off, crlf=True)
        assert rc == 0 and wbad == 0
        assert np.array_equal(id_off, wid_off)
        assert np.array_equal(ids, wids)
        assert np.array_equal(plen, wplen)
    # property (ii): decode(encode(x)) == crlf(x)
    lens = np.array([len(t) for t in toks])
    assert int(lens[ids].sum()) == int(plen.sum())
    s0 = blob[int(off[3]):int(off[4])].tobytes()
    dec = b"".join(toks[i] for i in ids[int(id_off[3]):int(id_off[4])])
    assert dec == s0.replace(b"\r\n", b"\n")


def test_token_frequencies_exact(N):
    blob, off, toks, sc, kp = synth_setup(2, 12, 3_000_000, 20000, 16)
    gm, om = both(N, toks, sc)
    fr, rc, bad, blen = gm.token_frequencies(blob, off)
    want = om.token_frequencies(blob, off, threads=8)
    assert rc == 0 and np.array_equal(fr, want)
    lens = np.array([len(t) for t in toks], dtype=np.uint64)
    assert int((fr * lens).sum()) == int(off[-1])  # invariant (iv)
    # NoPath surfaces like src/prune.rs:218-221
    gm2 = N.Model([b"a"], [-1.0])
    b2, o2 = N.pack([b"aaa", b"aba"])
    fr, rc, bad, blen = gm2.token_frequencies(b2, o2)
    assert rc == N.TGX_ERR_NO_PATH and bad == 1 and blen == 3


# ----------------------------------------------------------------------------- E-step
LATTICE_VOCAB = [(b"<", -3.0), (b" value", -6.0), (b">", -3.0), (b"DC value", -8.0), (b"<DC", -4.0),
                 (b"<DC value>", -12.0)]


@pytest.mark.parametrize("g", [0, -2, -3, 1, 8, 32])
def test_reference_lattice_marginals(N, g):
    toks = [t for t, _ in LATTICE_VOCAB]
    sc = [s for _, s in LATTICE_VOCAB]
    m = N.Model(toks, sc)
    estep_cfg(m, g)
    blob, off = N.pack([b"<DC value>"])
    ex, rc, bad, badz = m.expected_counts(blob, off)
    want = {b"<DC value>": 0.665241, b">": 0.334759, b"<DC": 0.244728, b" value": 0.244728, b"<": 0.090031,
            b"DC value": 0.090031}  # /root/reference/src/lattice.rs:447-452
    assert rc == 0
    for t, e in zip(toks, ex):
        assert abs(e - want[t]) < 5e-7
    # Q7: positions nothing ends at keep log 1
    m = N.Model([b"ab", b"c", b"bc"], [-1.0, -2.0, -3.0])
    estep_cfg(m, g)
    blob, off = N.pack([b"abc"])
    ex, rc, bad, badz = m.expected_counts(blob, off)
    assert rc == 0 and np.allclose(ex, [0.5, 0.5, 0.5], rtol=1e-12)


@pytest.mark.parametrize("g", [0, -2, -3, 1, 4, 32])
def test_expected_counts_random_vs_oracle(N, g):
    rng = random.Random(200 + abs(g))
    for it in range(20):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(5, 40), max_len=rng.randrange(1, 8),
                                  complete=True)
        gm, om = both(N, toks, scores)
        estep_cfg(gm, g)
        samples = rand_samples(rng, b"abcd", rng.randrange(1, 60), 1, 300)
        blob, off = N.pack(samples)
        snip = rng.choice([7, 64, 81920])
        ex, rc, bad, badz = gm.expected_counts(blob, off, snippet_len=snip)
        want, wrc, wbad, _ = om.run_e_step(blob, off, threads=1, literal=True, max_sample_length=snip)
        assert rc == 0 and wrc == 0
        assert np.allclose(ex, want, rtol=REL_TOL, atol=1e-27), np.max(np.abs(ex - want) / np.maximum(want, 1e-300))
        assert np.allclose(ex, want, rtol=ORDER_TOL, atol=1e-27), np.max(np.abs(ex - want) / np.maximum(want, 1e-300))
        tot = sum(e * len(t) for e, t in zip(ex, toks))
        assert abs(tot - int(off[-1])) < 1e-9 * int(off[-1])  # invariant (i)


def test_expected_counts_long_tokens(N):
    """max_token_len > 16: the lane-per-snippet and split-form kernels do not apply (16-slot windows); the lane-group
    kernels take every snippet, whatever the options say."""
    rng = random.Random(4242)
    toks = [bytes([c]) for c in b"ab"] + [b"ab" * 10, b"a" * 17, b"b" * 32, b"ba" * 7, b"abb"]
    scores = [-3.0, -3.5, -9.0, -8.0, -20.0, -5.0, -4.0]
    gm, om = both(N, toks, scores)
    samples = [b"ab" * 50, b"a" * 100, b"b" * 200, b"abba" * 30] + rand_samples(rng, b"ab", 20, 1, 300)
    blob, off = N.pack(samples)
    want = om.run_e_step(blob, off, threads=1, literal=True)[0]
    for g in (0, -2, -3, 4, 32):
        estep_cfg(gm, g)
        ex, rc, bad, badz = gm.expected_counts(blob, off)
        assert rc == 0 and np.allclose(ex, want, rtol=ORDER_TOL, atol=1e-27), (g, np.max(np.abs(ex - want)))


def test_expected_counts_bad_z(N):
    m = N.Model([b"a"], [-1.0])
    blob, off = N.pack([b"aa", b"ab", b"a"])
    ex, rc, bad, badz = m.expected_counts(blob, off)
    assert rc == N.TGX_ERR_BAD_Z and bad == 1 and badz == 0.0  # Q11: z == 0.0 is not normal


def test_expected_counts_synth_vs_oracle(N):
    blob, off, toks, sc, kp = synth_setup(2, 13, 2_000_000, 30000, 16)
    gm, om = both(N, toks, sc)
    want, wrc, wbad, _ = om.run_e_step(blob, off, threads=8, literal=False)
    for g in (0, -2, -3, 1, 8, -1):
        if g != -1:
            estep_cfg(gm, g)
        else:  # the default split: lanes below 16 KB, lane groups above, warps for the longest
            gm.set_option(17, 16384)
            gm.set_option(2, 4)
        ex, rc, bad, badz = gm.expected_counts(blob, off)
        assert rc == 0 and wrc == 0
        rel = counts_rel_err(ex, want)
        assert rel < REL_TOL, rel
        assert rel < ORDER_TOL, rel
        lens = np.array([len(t) for t in toks], dtype=np.float64)
        assert abs(float((ex * lens).sum()) - int(off[-1])) < 1e-9 * int(off[-1])


def test_expected_counts_replica_shapes_bit_identical(N):
    """The replicas of the hot ids (options 20 / 21) are a placement of the fixed-point accumulators, not arithmetic:
    every shape — none, one id, more ids than the vocabulary has — gives the same counts to the bit (the exact sum
    that stands in for the f64 merge of src/prune.rs:104-112)."""
    blob, off, toks, sc, kp = synth_setup(2, 17, 1_500_000, 20000, 16)
    gm, om = both(N, toks, sc)
    base = gm.expected_counts(blob, off)[0]
    want = om.run_e_step(blob, off, threads=8, literal=False)[0]
    assert counts_rel_err(base, want) < REL_TOL
    for r, k in ((1, 4096), (64, 0), (7, 1), (4096, 16), (3, 1 << 20), (256, 4096)):
        gm.set_option(20, r)
        gm.set_option(21, k)
        ex, rc, bad, badz = gm.expected_counts(blob, off)
        assert rc == 0
        assert np.array_equal(ex.view(np.uint64), base.view(np.uint64)), (r, k)


def test_very_long_samples(N):
    """Samples far beyond the 64-position rounds, the 1024-position backtrack chunks and the 81920-byte snippet
    length of the E-step (src/prune.rs:75,83): one of 400 KB, one of exactly 2 * 81920 bytes, one of 81920 + 1."""
    rng = random.Random(2024)
    toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=150, max_len=10)
    gm, om = both(N, toks, scores)
    samples = [bytes(rng.choice(b"abcd") for _ in range(n)) for n in (400_000, 2 * 81920, 81921, 7, 0, 81920)]
    for algo in (0, 1, 2, 3):
        gm.set_option(3, algo)
        check_against_oracle(N, gm, om, samples, algo)
    gm.set_option(32, 1 << 30)
    check_against_oracle(N, gm, om, samples, "teams only")
    gm.set_option(3, 0)
    blob, off = N.pack(samples)
    ex, rc, bad, badz = gm.expected_counts(blob, off)
    want = om.run_e_step(blob, off, threads=8)[0]
    assert rc == 0 and counts_rel_err(ex, want) < REL_TOL
    fr = gm.token_frequencies(blob, off)[0]
    assert np.array_equal(fr, om.token_frequencies(blob, off, threads=8))


def test_host_entry_point_rejects_bad_offsets(N):
    """Offsets that decrease are an argument error (nothing is encoded, nothing is truncated silently)."""
    import ctypes as C
    m = N.Model([b"a", b"b"], [-1.0, -1.0])
    blob = np.frombuffer(b"abab", np.uint8).copy()
    off = np.array([0, 3, 2, 4], np.uint64)
    ids, id_off = np.zeros(8, np.uint32), np.zeros(4, np.uint64)
    rc = N.lib().tgx_encode_batch(m._h, blob.ctypes.data_as(N.u8p), off.ctypes.data_as(N.u64p), 3, 0,
                                  ids.ctypes.data_as(N.u32p), 8, id_off.ctypes.data_as(N.u64p), None, None, None)
    assert rc == N.TGX_ERR_INVALID and b"decrease" in N.lib().tgx_last_error()
    ids2, id_off2, status, plen, rc, bad = m.encode_batch(blob, np.array([0, 2, 2, 4], np.uint64))
    assert rc == 0 and ids2.tolist() == [0, 1, 0, 1] and id_off2.tolist() == [0, 2, 2, 4]
