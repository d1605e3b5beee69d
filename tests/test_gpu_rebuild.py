"""Every device path on a model rebuilt in place, against a fresh model and the oracle, bit for bit.

The EM loop rebuilds its model about twice per iteration (tokengeex_b200/prune.py).  For a subset of at least option 45
per mille of the vocabulary the double-array was built for, tgx_model_rebuild keeps the array's layout and rewrites
terminal flags, ids and scores in place (retarget_double_array, trie_build.cpp).  That leaves states a fresh build never
makes: leaves of dropped tokens that are neither terminals nor parents, subtrees without a terminal, a max_token_len that
is the array's depth rather than the longest token's, ids permuted against a layout placed for other ids, and a BFS
layout (from an earlier fresh rebuild) under a retarget.  The match tables (slots8 / rows / row_ids / pair2: forward
passes 0 and 3, E-step form 2) and the emit's token hash are rebuilt from that state.

Each chain applies its steps with Model.rebuild to ONE handle and asserts which path every step took.  After every
step the handle, a fresh N.Model of the same vocabulary and the oracle must agree bit for bit: encode on every forward
pass and emit path, keyed dropout, the E-step's fixed-point limbs on every kernel set, the frequency passes,
encode_corpus and prune_select.  Refused rebuilds must leave the old vocabulary answering on the device, and the whole
EM schedule must end in the same vocabulary with and without the retarget.
"""
import random
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import estep_cfg, fixed_point_samples, rand_samples, rand_vocab, split_ids, synth_setup

pytestmark = pytest.mark.gpu

ONE = 1 << 128
SNIP = 81920
KERNEL_SETS = [0, -2, -3, 1, 4, 32, "split"]
LONG = 8192  # option 32 lowered: samples of at least this many bytes run on the side pair kernel of forward pass 3

# forward pass (option 3), match2_kernel or match_kernel (37), emit through the token hash or a trie walk (16)
ENCODE_CONFIGS = ([{3: 0, 37: c, 16: e} for c in (0, 1) for e in (0, 1)]
                  + [{3: a, 16: e} for a in (1, 2) for e in (0, 1)]
                  + [{3: 3, 32: LONG, 37: c, 16: e} for c in (0, 1) for e in (0, 1)])


@pytest.fixture(scope="module")
def N():
    from tokengeex_b200 import _native
    return _native


# ----------------------------------------------------------------------------- helpers (as in test_gpu_exact_counts)
def configure(gm, g):
    if g == "split":  # the default split: lanes below 16 KB, lane groups above, warps for the longest
        gm.set_option(17, 16384)
        gm.set_option(2, 4)
    else:
        estep_cfg(gm, g)


def to_dev(blob, off):
    import torch
    return torch.from_numpy(np.ascontiguousarray(blob)).cuda(), torch.from_numpy(off.astype(np.uint64).view(np.int64)).cuda()


def run_fixed(gm, blob, off, snip=SNIP):
    """tgx_expected_counts_fixed_dev over (blob, off) into new zero limbs."""
    import torch
    d_text, d_off = to_dev(blob, off)
    limbs = torch.zeros(5 * max(gm.V, 1), dtype=torch.int64, device="cuda")
    rc, bad, _ = gm.expected_counts_fixed_dev(d_text.data_ptr(), d_off.data_ptr(), len(off) - 1, int(off[-1]),
                                              limbs.data_ptr(), snippet_len=snip)
    assert rc == 0 and bad == -1
    return limbs


def limbs_to_ints(limbs, V):
    rows = limbs.cpu().numpy().reshape(-1, 5)[:V].tolist()
    return [l0 + (l1 << 32) + (l2 << 64) + (l3 << 96) + (l4 << 128) for l0, l1, l2, l3, l4 in rows]


def nearest(xs):
    return np.array([float(Fraction(x, ONE)) for x in xs], np.float64)


def assert_same_bits(got, want, ctx=None):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, (ctx, bad[:5].tolist(), got[bad[:5]].tolist(), want[bad[:5]].tolist())


def assert_limbs_equal(got, want, ctx=None):
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert len(got) == len(want) and not bad, (ctx, bad[:5], [(got[i] - want[i]) for i in bad[:5]])


def assert_encode_equal(N, got, want, ctx=None):
    ids, id_off, status, plen, rc, bad = got
    wids, wid_off, wstatus, wplen, wbad = want
    first = wbad - 1  # the oracle returns the lowest failing index + 1, or 0
    assert np.array_equal(id_off, wid_off) and np.array_equal(ids, wids), ctx
    assert np.array_equal(status, np.where(wstatus != 0, N.TGX_ERR_NO_PATH, 0)), ctx
    assert np.array_equal(plen, wplen), ctx
    assert bad == first and rc == (N.TGX_ERR_NO_PATH if first >= 0 else N.TGX_OK), (ctx, rc, bad, first)


def set_options(gm, opts):
    for k, v in opts.items():
        gm.set_option(k, v)


def with_path(om, samples):
    """The samples the oracle encodes without NoPath."""
    blob, off = O.pack_samples(samples)
    status = om.encode_batch(blob, off, threads=8)[2]
    return [s for s, st in zip(samples, status) if st == 0]


# ----------------------------------------------------------------------------- chains
class Step:
    def __init__(self, name, toks, scores, path):
        self.name, self.toks, self.scores, self.path = name, list(toks), [float(s) for s in scores], path


class Chain:
    def __init__(self, name, steps, samples, em_blob=None):
        self.name, self.steps, self.samples = name, steps, samples
        self.em_blob = em_blob  # (blob, off) of the synthetic corpus (EM chain only)
        # the rule of tgx_model_rebuild: retarget a subset of >= 45 % of the size the array was built for
        built = None
        for k, st in enumerate(steps):
            if k and st.path == "retarget":
                assert len(st.toks) * 1000 >= len(built) * 450 and set(st.toks) - {b""} <= prefixes(built), (name, k)
            if k == 0 or st.path == "fresh":
                built = st.toks
        assert {st.path for st in steps[1:]} == {"retarget", "fresh"}, name


def prefixes(toks):
    return {t[:k] for t in toks for k in range(1, len(t) + 1)}


def pick(rng, toks, scores, frac, keep_singles=True, drop=()):
    """Indices of a subset in id order: every single byte (unless in `drop`) and about `frac` of the rest."""
    return [i for i, t in enumerate(toks)
            if t not in drop and ((keep_singles and len(t) == 1) or rng.random() < frac)]


@pytest.fixture(scope="module")
def em_chain():
    """The EM loop's sequence on a 2 MB synthetic corpus with 6000 tokens of at most 16 bytes (the retarget's host
    threads engage from 2048 tokens)."""
    rng = random.Random(4101)
    blob, off, toks, sc, kp = synth_setup(2, 41, 2_000_000, 6000, 16)
    toks, sc = list(toks), [float(x) for x in sc]
    steps = [Step("create", toks, sc, "fresh")]
    # M-step: ~85 % in id order, every single byte, scores shifted by a non-integer
    idx = pick(rng, toks, sc, 0.85)
    t1, s1 = [toks[i] for i in idx], [sc[i] - 0.375 for i in idx]
    steps.append(Step("m-step", t1, s1, "retarget"))
    # prune step: ~75 % in score-descending order (ids permuted against the layout)
    order = sorted(range(len(t1)), key=lambda i: (-s1[i], i))
    keep = set(i for i in order[:int(0.75 * len(t1))]) | {i for i, t in enumerate(t1) if len(t) == 1}
    order = [i for i in order if i in keep]
    t2, s2 = [t1[i] for i in order], [s1[i] for i in order]
    steps.append(Step("prune", t2, s2, "retarget"))
    idx = pick(rng, t2, s2, 0.85)
    t3, s3 = [t2[i] for i in idx], [s2[i] - 0.8125 for i in idx]
    steps.append(Step("m-step-2", t3, s3, "retarget"))
    # under 45 % of the built size: a fresh build in BFS order
    others = [i for i, t in enumerate(t3) if len(t) > 1]
    rng.shuffle(others)
    n_single = sum(len(t) == 1 for t in t3)
    idx = sorted([i for i, t in enumerate(t3) if len(t) == 1] + others[:2650 - n_single])
    t4, s4 = [t3[i] for i in idx], [s3[i] for i in idx]
    assert len(t4) * 1000 < len(toks) * 450
    steps.append(Step("small", t4, s4, "fresh"))
    # a subset of that (>= 2048 tokens) retargets the BFS layout
    idx = pick(rng, t4, s4, 0.82)
    t5, s5 = [t4[i] for i in idx], [s4[i] + 0.125 for i in idx]
    assert len(t5) >= 2048
    steps.append(Step("bfs-retarget", t5, s5, "retarget"))
    # a superset with a token the array has no node for
    new = b"\xf0\x9f\x98\x80zq"
    assert new not in prefixes(t4)
    steps.append(Step("superset", t5 + [new], s5 + [-7.25], "fresh"))
    samples = [blob[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(off) - 1)]
    singles = {t for t in toks if len(t) == 1}
    missing = next(bytes([b]) for b in range(256) if bytes([b]) not in singles)
    extra = [b"", b"x" + missing + b"y", b"".join(rng.choice(t5) for _ in range(3000)), missing, b""]
    return Chain("em", steps, samples + extra, em_blob=(blob, off))


@pytest.fixture(scope="module")
def depth_chain():
    """Tokens up to 24 bytes over an alphabet with NUL and bytes >= 0x80, integer scores (exact ties).  A retarget to
    a subset without any token over 16 bytes keeps max_token_len = 24 (the lane-group kernels) while a fresh model of
    that vocabulary takes the <= 16-byte paths; then back to a subset with long tokens."""
    rng = random.Random(4102)
    alphabet = b"\x00a\x80\xfe\xff\r\n"
    toks, sc = rand_vocab(rng, alphabet=alphabet, n_tok=400, max_len=24, int_scores=True)
    for t in (b"\x00" * 24, b"a\x80" * 12, b"\xff" * 17):
        if t not in toks:
            toks.append(t)
            sc.append(-3.0)
    steps = [Step("create", toks, sc, "fresh")]
    idx = pick(rng, toks, sc, 0.85, drop={t for t in toks if len(t) > 16})
    t1, s1 = [toks[i] for i in idx], [sc[i] - 1.0 for i in idx]
    steps.append(Step("short-only", t1, s1, "retarget"))
    longs = [t for t in toks if len(t) > 16]
    back = t1 + longs[::2]
    rng.shuffle(back)
    steps.append(Step("long-again", back, [-float(rng.randrange(2, 6)) for _ in back], "retarget"))
    idx = pick(rng, t1, s1, 0.25)
    t3, s3 = [t1[i] for i in idx], [s1[i] for i in idx]
    steps.append(Step("small", t3, s3, "fresh"))
    steps.append(Step("superset-long", t3 + longs, s3 + [-4.0] * len(longs), "fresh"))
    samples = rand_samples(rng, alphabet, 60, 0, 300)
    samples += [b"".join(rng.choice(toks) for _ in range(rng.randrange(1, 40))) for _ in range(30)]
    samples += [b"".join(rng.choice(longs) for _ in range(600)), bytes(rng.choice(alphabet) for _ in range(9000))]
    samples += [b"", b"az\x00", b"z", b"\x00" * 24 + b"\r\n" + b"\x00" * 17]
    rng.shuffle(samples)
    return Chain("depth", steps, samples)


@pytest.fixture(scope="module")
def edges_chain():
    """All 256 single bytes and 250 longer tokens; every step but the last two retargets: a duplicate byte string (the
    last id wins), the empty token, only the single bytes (every multi-byte node a non-terminal), a byte dropped
    (NoPath samples); then V = 0 and back to the full vocabulary."""
    rng = random.Random(4103)
    alphabet = b"ab\x00\xff\r\n"
    multi = set()
    while len(multi) < 250:
        multi.add(bytes(rng.choice(alphabet) for _ in range(rng.randrange(2, 11))))
    toks = [bytes([b]) for b in range(256)] + sorted(multi)
    rng.shuffle(toks)
    sc = [-float(rng.randrange(2, 7)) if rng.random() < 0.3 else -(rng.random() * 6 + 0.5) for _ in toks]
    steps = [Step("create", toks, sc, "fresh")]
    idx = pick(rng, toks, sc, 0.8)
    t1, s1 = [toks[i] for i in idx], [sc[i] for i in idx]
    dup = next(i for i, t in enumerate(t1) if len(t) > 2)
    steps.append(Step("duplicate", t1 + [t1[dup]], s1 + [-0.75], "retarget"))
    idx = pick(rng, toks, sc, 0.8)
    t2, s2 = [toks[i] for i in idx], [sc[i] - 0.5 for i in idx]
    t2.insert(len(t2) // 2, b"")
    s2.insert(len(s2) // 2, -1.0)
    steps.append(Step("empty-token", t2, s2, "retarget"))
    idx = [i for i, t in enumerate(toks) if len(t) == 1]
    steps.append(Step("singles", [toks[i] for i in idx], [sc[i] for i in idx], "retarget"))
    idx = pick(rng, toks, sc, 0.85, drop={b"b"})
    steps.append(Step("byte-dropped", [toks[i] for i in idx], [sc[i] + 0.25 for i in idx], "retarget"))
    steps.append(Step("empty-vocabulary", [], [], "fresh"))
    steps.append(Step("full", toks, sc, "fresh"))
    samples = rand_samples(rng, alphabet, 60, 0, 200) + rand_samples(rng, bytes(range(256)), 10, 1, 100)
    samples += [b"".join(rng.choice(sorted(multi)) for _ in range(rng.randrange(1, 30))) for _ in range(20)]
    samples += [b"b", b"ab" * 5000, b"", b"a\rb\r\n"]
    rng.shuffle(samples)
    return Chain("edges", steps, samples)


@pytest.fixture(scope="module", params=["em", "depth", "edges"])
def chain(request):
    return request.getfixturevalue(f"{request.param}_chain")


def walk(N, chain, prepare=lambda gm: None):
    """Creates one handle from the chain's first vocabulary, lets `prepare` set its options / dropout once, and applies
    every later step with Model.rebuild.  Yields (k, step, handle, fresh model of the step's vocabulary, prepared the
    same way) after each step, asserting the path it took: a retarget keeps trie_nodes / trie_slots / max_token_len of
    the array (which holds nodes the new vocabulary does not need), a fresh build has the fresh model's nodes."""
    first = chain.steps[0]
    gm = N.Model(first.toks, first.scores, device=0)
    prepare(gm)
    paths = []
    for k, st in enumerate(chain.steps):
        before = gm.info()
        if k:
            gm.rebuild(st.toks, st.scores)
        fresh = N.Model(st.toks, st.scores, device=0)
        prepare(fresh)
        got, want = gm.info(), fresh.info()
        assert got.vocab_size == len(st.toks) and got.trie_terminals == want.trie_terminals, (chain.name, st.name)
        if k:
            arr = (got.trie_nodes, got.trie_slots, got.max_token_len)
            if st.path == "retarget":
                assert arr == (before.trie_nodes, before.trie_slots, before.max_token_len), (chain.name, st.name)
                assert want.trie_nodes < got.trie_nodes, (chain.name, st.name)
            else:
                assert got.trie_nodes == want.trie_nodes != before.trie_nodes, (chain.name, st.name)
                assert got.max_token_len == want.max_token_len, (chain.name, st.name)
            paths.append(st.path)
        yield k, st, gm, fresh
        fresh.close()
    assert "retarget" in paths and "fresh" in paths
    gm.close()


# ----------------------------------------------------------------------------- B1: encode
def test_encode_every_forward_pass(N, chain):
    """Ids, offsets, status, processed length and first failing sample of every forward pass and emit path, with and
    without crlf, on the rebuilt handle and on a fresh model.  Forward passes 0 and 3 must run on the match tables
    whenever the array's tokens fit 16 bytes (tgx_model_last_stat 10)."""
    blob, off = N.pack(chain.samples)
    for k, st, gm, fresh in walk(N, chain):
        om = O.OracleModel(st.toks, st.scores)
        tables = gm.info().max_token_len <= 16
        for crlf in (False, True):
            want = om.encode_batch(blob, off, crlf=crlf, threads=8)
            for cfg in ENCODE_CONFIGS:
                for which, m in (("rebuilt", gm), ("fresh", fresh)):
                    set_options(m, cfg)
                    assert_encode_equal(N, m.encode_batch(blob, off, crlf=crlf), want, (chain.name, st.name, which, crlf, cfg))
                if cfg[3] in (0, 3) and tables and st.toks:
                    assert gm.stat(10) == cfg[3], (chain.name, st.name, cfg)
        if chain.name == "depth" and st.name == "short-only":  # the array's depth stays: still the lane-group kernels
            assert gm.info().max_token_len == 24 and fresh.info().max_token_len <= 16


# ----------------------------------------------------------------------------- B2: keyed dropout encode
@pytest.mark.parametrize("algo", [1, 2])
def test_keyed_dropout_encode_survives_rebuilds(N, chain, algo):
    """Dropout and option 3 are set once, on the handle as created: every rebuilt vocabulary must encode like the
    oracle's keyed draw."""
    p, seed = 0.3, 977 + algo
    samples = chain.samples
    blob, off = N.pack(samples)

    def prepare(m):
        m.set_option(3, algo)
        m.set_dropout(p, seed)

    for k, st, gm, fresh in walk(N, chain, prepare):
        om = O.OracleModel(st.toks, st.scores)
        want = []  # ids, or the length of a NoPath sample
        for i, s in enumerate(samples):
            try:
                want.append(om.encode_keyed(s, p, seed, i))
            except O.NoPath as e:
                want.append(e.length)
        first = next((i for i, w in enumerate(want) if isinstance(w, int)), -1)
        for which, m in (("rebuilt", gm), ("fresh", fresh)):
            ids, id_off, status, plen, rc, bad = m.encode_batch(blob, off)
            got = split_ids(ids, id_off)
            for i, w in enumerate(want):
                if isinstance(w, int):
                    assert status[i] == N.TGX_ERR_NO_PATH and got[i] == [] and plen[i] == w, (st.name, which, i)
                else:
                    assert status[i] == 0 and got[i] == w, (chain.name, st.name, which, i)
            assert bad == first and (rc == 0) == (first < 0), (chain.name, st.name, which)


# ----------------------------------------------------------------------------- B3: E-step limbs
def estep_batch(chain, om, toks, dropout=False):
    """The samples whose lattices the E-step accepts.  With dropout: the samples made of single-byte tokens only (the
    draw never drops those, so every position stays reachable whatever it drops)."""
    if chain.em_blob is not None:  # every byte of the corpus is a token at every step
        return chain.em_blob
    if dropout:
        singles = {t[0] for t in toks if len(t) == 1}
        return O.pack_samples([s for s in chain.samples if s and set(s) <= singles])
    return O.pack_samples(fixed_point_samples(om, [s for s in chain.samples if s], SNIP))


def test_estep_limbs_every_kernel_set(N, chain):
    """The limbs of every E-step kernel set equal the oracle's exact sums on the rebuilt handle and on a fresh model,
    and tgx_expected_counts returns the nearest f64 to them."""
    for k, st, gm, fresh in walk(N, chain):
        if not st.toks:
            continue
        om = O.OracleModel(st.toks, st.scores)
        blob, off = estep_batch(chain, om, st.toks)
        want, rc, _ = om.run_e_step_fixed(blob, off, threads=8)
        assert rc == 0
        for g in KERNEL_SETS:
            for which, m in (("rebuilt", gm), ("fresh", fresh)):
                configure(m, g)
                assert_limbs_equal(limbs_to_ints(run_fixed(m, blob, off), len(st.toks)), want, (chain.name, st.name, which, g))
        ex, rc, *_ = gm.expected_counts(blob, off)
        assert rc == 0
        assert_same_bits(ex, nearest(want), (chain.name, st.name))


def test_estep_keyed_dropout_limbs(N, chain):
    """Keyed dropout and a byte base (option 22), set once on the handle as created, on every kernel set."""
    p, seed, base = 0.3, 2 ** 61 + 17, 123457

    def prepare(m):
        m.set_option(22, base)
        m.set_dropout(p, seed)

    for k, st, gm, fresh in walk(N, chain, prepare):
        if not st.toks:
            continue
        om = O.OracleModel(st.toks, st.scores)
        blob, off = estep_batch(chain, om, st.toks, dropout=True)
        want, rc, _ = om.run_e_step_fixed(blob, off, p, seed, keyed=True, byte_base=base, threads=8)
        assert rc == 0
        for g in KERNEL_SETS:
            for which, m in (("rebuilt", gm), ("fresh", fresh)):
                configure(m, g)
                assert_limbs_equal(limbs_to_ints(run_fixed(m, blob, off), len(st.toks)), want, (chain.name, st.name, which, g))


# ----------------------------------------------------------------------------- B4: frequency passes, encode_corpus
def test_frequency_passes(N, chain):
    """Token frequencies on every forward pass and pair frequencies against the oracle, over the samples that have a
    path; encode_corpus (u32, u16 while V < 65536, with and without a separator) against the fresh model."""
    for k, st, gm, fresh in walk(N, chain):
        if not st.toks:
            continue
        om = O.OracleModel(st.toks, st.scores)
        blob, off = N.pack(with_path(om, chain.samples))
        want = om.token_frequencies(blob, off, threads=8)
        for cfg in ({3: 2}, {3: 0, 37: 1}, {3: 3, 32: LONG}, {3: 1}):
            for which, m in (("rebuilt", gm), ("fresh", fresh)):
                set_options(m, cfg)
                fr, rc, bad, blen = m.token_frequencies(blob, off)
                assert rc == 0 and np.array_equal(fr, want), (chain.name, st.name, which, cfg)
        wp, wc = om.pair_frequencies(blob, off, threads=8)
        for which, m in (("rebuilt", gm), ("fresh", fresh)):
            pairs, counts, rc, bad, blen = m.pair_frequencies(blob, off)
            assert rc == 0 and np.array_equal(pairs, wp) and np.array_equal(counts, wc), (chain.name, st.name, which)
        if chain.em_blob is None:
            continue  # (encode_corpus takes NUL-separated UTF-8: the synthetic corpus only)
        cb, co = chain.em_blob
        data = np.frombuffer(b"\x00".join(cb[int(co[i]):int(co[i + 1])].tobytes() for i in range(len(co) - 1)) + b"\x00",
                             np.uint8).copy()
        V = len(st.toks)
        for dtype, sep, crlf in ((np.uint32, -1, False), (np.uint32, V - 1, True), (np.uint16, 0, False)):
            if dtype is np.uint16 and V >= 65536:
                continue
            got = gm.encode_corpus(data, crlf=crlf, sep_id=sep, dtype=dtype)
            ref = fresh.encode_corpus(data, crlf=crlf, sep_id=sep, dtype=dtype)
            assert got[2] == ref[2] == 0 and got[3:] == ref[3:], (st.name, dtype, sep)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), (st.name, dtype, sep)


# ----------------------------------------------------------------------------- B5: prune_select
@pytest.mark.parametrize("which", ["em_chain", "depth_chain"])
def test_prune_select_over_rebuilt_trie(N, request, which):
    """Model.prune_select walks the rebuilt array for the n-best alternatives: the same ids and audit as
    prune_select over a fresh trie, and the oracle's prune_vocab."""
    chain = request.getfixturevalue(which)
    for k, st, gm, fresh in walk(N, chain):
        om = O.OracleModel(st.toks, st.scores)
        samples = with_path(om, chain.samples)
        blob, off = O.pack_samples(samples)
        keep = np.array([len(t) == 1 for t in st.toks], np.uint8)
        fr = om.token_frequencies(blob, off, threads=8)
        target = int(0.7 * len(st.toks))
        try:
            wm, waudit = O.OracleModel(st.toks, st.scores, keep).prune_vocab(blob, off, target, 0.8, threads=8)
        except RuntimeError:  # a loss that is not normal: refused everywhere
            for f in (lambda: gm.prune_select(st.toks, st.scores, keep, fr, len(samples), target, 0.8, threads=4),
                      lambda: N.prune_select(st.toks, st.scores, keep, fr, len(samples), target, 0.8, threads=4)):
                with pytest.raises(N.TgxError):
                    f()
            continue
        ids, audit = gm.prune_select(st.toks, st.scores, keep, fr, len(samples), target, 0.8, threads=4)
        ids2, audit2 = N.prune_select(st.toks, st.scores, keep, fr, len(samples), target, 0.8, threads=4)
        assert np.array_equal(ids, ids2) and np.array_equal(audit, audit2), (chain.name, st.name)
        assert [st.toks[i] for i in ids] == wm.export()[0], (chain.name, st.name)
        assert np.array_equal(audit[:7], waudit[:7]), (chain.name, st.name)


# ----------------------------------------------------------------------------- B6: refused rebuilds
def test_refused_rebuilds_leave_the_device_model(N, em_chain):
    """After a retarget with permuted ids, and with the match tables built, a rebuild with an inf score (a subset that
    would retarget) and one with a 65-byte token are refused; the device then still gives the old vocabulary's
    output on forward pass 0 (match tables), forward pass 2 and E-step form 2 (match stream)."""
    chain = em_chain
    blob, off = N.pack(chain.samples)
    eb, eo = chain.em_blob
    for k, st, gm, fresh in walk(N, chain):
        if st.name != "prune":
            continue
        om = O.OracleModel(st.toks, st.scores)
        want_enc = om.encode_batch(blob, off, threads=8)
        want_lim = om.run_e_step_fixed(eb, eo, threads=8)[0]

        def check(ctx):
            for algo in (0, 2):
                gm.set_option(3, algo)
                assert_encode_equal(N, gm.encode_batch(blob, off), want_enc, (ctx, algo))
            configure(gm, -2)
            assert_limbs_equal(limbs_to_ints(run_fixed(gm, eb, eo), len(st.toks)), want_lim, ctx)

        check("before")
        info = gm.info()
        sub = [i for i in range(len(st.toks)) if i % 7 or len(st.toks[i]) == 1]
        bad_scores = [st.scores[i] for i in sub]
        bad_scores[len(sub) // 2] = float("inf")
        with pytest.raises(N.TgxError) as ei:
            gm.rebuild([st.toks[i] for i in sub], bad_scores)
        assert ei.value.code == N.TGX_ERR_UNSUPPORTED
        check("inf score")
        with pytest.raises(N.TgxError) as ei:
            gm.rebuild(st.toks + [b"a" * 65], st.scores + [-1.0])
        assert ei.value.code == N.TGX_ERR_UNSUPPORTED
        check("65-byte token")
        after = gm.info()
        assert (after.vocab_size, after.trie_nodes, after.trie_slots, after.trie_terminals, after.max_token_len) == \
            (info.vocab_size, info.trie_nodes, info.trie_slots, info.trie_terminals, info.max_token_len)


# ----------------------------------------------------------------------------- C: the whole schedule
@pytest.fixture(scope="module")
def schedule_setup():
    return synth_setup(2, 43, 8_000_000, 20000, 16)


def run_schedule(N, monkeypatch, setup, opts):
    """ModelVocabularyPruner.prune (20 000 -> 6000 tokens, two EM sub-iterations) on models with `opts` set; also
    returns, per rebuild, whether the array kept its layout."""
    from tokengeex_b200 import prune as P
    blob, off, toks, sc, kp = setup
    kept = []
    base = N.Model

    class Configured(base):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            set_options(self, opts)

        def rebuild(self, tokens, scores, packed=None):
            b = self.info()
            super().rebuild(tokens, scores, packed=packed)
            a = self.info()
            kept.append((a.trie_nodes, a.trie_slots) == (b.trie_nodes, b.trie_slots))

    with monkeypatch.context() as mp:
        mp.setattr(P.N, "Model", Configured)
        vocab, report = P.ModelVocabularyPruner(6000, shrink_factor=0.8, em_subiters=2, dropout=0.0).prune(
            P.Vocab(list(toks), np.array(sc), np.array(kp)), blob, off)
    return vocab, report, kept


def test_schedule_bit_identical_with_and_without_retarget(N, monkeypatch, schedule_setup):
    """The counts are exact sums, so neither the layout of the array nor the kernel set may change the schedule: with
    option 45 at its default and at 0, on the default kernels and on the match-table paths (forward pass 3 for the
    frequency pass, E-step form 2), the sizes after every step, the final tokens in order and their scores and keep
    flags are bit-identical."""
    results = {}
    for opts in ({}, {3: 3, 19: 2}):
        for permille in (None, 0):
            o = dict(opts) if permille is None else {**opts, 45: permille}
            vocab, report, kept = run_schedule(N, monkeypatch, schedule_setup, o)
            results[(tuple(opts.items()), permille)] = (vocab, report, kept)
    ref_vocab, ref_report, ref_kept = results[((), None)]
    assert len(ref_vocab) <= 6000 and sum(ref_kept) >= 2  # the default schedule retargets
    for key, (vocab, report, kept) in results.items():
        assert report.vocab_sizes == ref_report.vocab_sizes, key
        assert vocab.tokens == ref_vocab.tokens, key
        assert np.array_equal(np.asarray(vocab.scores).view(np.uint64), np.asarray(ref_vocab.scores).view(np.uint64)), key
        assert np.array_equal(vocab.keep, ref_vocab.keep), key
        if key[1] == 0:  # never retargets: fewer rebuilds keep their layout than with the default
            assert sum(kept) < sum(results[(key[0], None)][2]), key
