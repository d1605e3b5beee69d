"""E-step counts bit for bit against exact integer sums.

The kernels keep every expected count as the exact sum of its contributions, each truncated to 2^-128, in 192-bit
fixed point (acc_add, the hot-id replicas folded by fold_hot_acc_kernel), export it as five int64 limbs per token and
turn (summed) limbs into the nearest f64 (include/tokengeex_b200.h).  The kernels restate the oracle's arithmetic
(((a + score) + beta) - z with separate roundings, glibc's exp), so every contribution equals the oracle's and the limbs
must equal the oracle's exact sums (OracleModel.run_e_step_fixed) to the last bit: for every kernel set, both
accumulator paths, every replica shape, keyed dropout, any split into calls or simulated ranks, and after a rebuild.
The f64 conversion must be the correctly rounded value of the exact sum.
"""
import random
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import estep_cfg, fixed_point_samples, rand_samples, rand_vocab, synth_setup

pytestmark = pytest.mark.gpu

ONE = 1 << 128
SNIP = 81920
KERNEL_SETS = [0, -2, -3, 1, 4, 32, "split"]


@pytest.fixture(scope="module")
def N():
    from tokengeex_b200 import _native
    return _native


def configure(gm, g):
    if g == "split":  # the default split: lanes below 16 KB, lane groups above, warps for the longest
        gm.set_option(17, 16384)
        gm.set_option(2, 4)
    else:
        estep_cfg(gm, g)


def to_dev(blob, off):
    import torch
    return torch.from_numpy(np.ascontiguousarray(blob)).cuda(), torch.from_numpy(off.astype(np.uint64).view(np.int64)).cuda()


def new_limbs(V):
    import torch
    return torch.zeros(5 * max(V, 1), dtype=torch.int64, device="cuda")


def run_fixed(gm, blob, off, limbs=None, snip=SNIP):
    """tgx_expected_counts_fixed_dev over (blob, off) into `limbs` (a new zero tensor by default)."""
    d_text, d_off = to_dev(blob, off)
    if limbs is None:
        limbs = new_limbs(gm.V)
    rc, bad, _ = gm.expected_counts_fixed_dev(d_text.data_ptr(), d_off.data_ptr(), len(off) - 1, int(off[-1]),
                                              limbs.data_ptr(), snippet_len=snip)
    assert rc == 0 and bad == -1
    return limbs


def limbs_to_ints(limbs, V):
    rows = limbs.cpu().numpy().reshape(-1, 5)[:V].tolist()
    return [l0 + (l1 << 32) + (l2 << 64) + (l3 << 96) + (l4 << 128) for l0, l1, l2, l3, l4 in rows]


def ints_to_limbs(xs):
    """Normalised limbs of fixed-point values X (count * 2^128): four 32-bit words and the integer part."""
    return [[(x >> (32 * k)) & 0xFFFFFFFF for k in range(4)] + [x >> 128] for x in xs]


def nearest(xs):
    return np.array([float(Fraction(x, ONE)) for x in xs], np.float64)


def convert(N, gm, rows):
    """counts_from_limbs_dev of int64 limb rows (any carries still pending)."""
    import torch
    lt = torch.tensor(rows, dtype=torch.int64, device="cuda").reshape(-1)
    out = torch.full((len(rows),), float("nan"), dtype=torch.float64, device="cuda")
    gm.counts_from_limbs_dev(lt.data_ptr(), len(rows), out.data_ptr())
    return out.cpu().numpy()


def assert_same_bits(got, want, ctx=None):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, (ctx, bad[:5].tolist(), got[bad[:5]].tolist(), want[bad[:5]].tolist())


def assert_limbs_equal(got, want, ctx=None):
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert len(got) == len(want) and not bad, (ctx, bad[:5], [(got[i] - want[i]) for i in bad[:5]])


# ----------------------------------------------------------------------------- cases shared by the kernel sets
@pytest.fixture(scope="module")
def random_cases():
    """Random vocabularies (complete and incomplete, integer scores for exact ties, tokens up to 16 bytes and longer
    ones for the lane-group kernels) with their samples, snippet length and the oracle's exact sums."""
    rng = random.Random(515)
    cases = []
    for it in range(8):
        alphabet = [b"abcd", b"ab"][it % 2]
        max_len = [6, 12, 16, 24][it % 4]
        complete = it % 3 != 2
        toks, scores = rand_vocab(rng, alphabet=alphabet, n_tok=rng.randrange(8, 120), max_len=max_len,
                                  complete=complete, int_scores=(it % 2 == 0))
        if max_len > 16:
            toks = list(toks) + [alphabet[:1] * 17, alphabet[:2] * 10]
            scores = list(scores) + [-7.0, -9.0]
        om = O.OracleModel(toks, scores)
        snip = [SNIP, 64, 7, SNIP][it % 4] if complete else SNIP
        samples = rand_samples(rng, alphabet, rng.randrange(5, 80), 1, 600)
        samples += [bytes(rng.choice(alphabet) for _ in range(n)) for n in (3000, rng.randrange(1, 40))]
        if not complete:  # text with a path: runs of tokens (positions off every path give contributions above 1)
            samples += [b"".join(rng.choice(toks) for _ in range(rng.randrange(1, 60))) for _ in range(40)]
        samples = fixed_point_samples(om, samples, snip)
        assert samples
        blob, off = O.pack_samples(samples)
        want, rc, _ = om.run_e_step_fixed(blob, off, threads=8, max_sample_length=snip)
        assert rc == 0
        cases.append((toks, scores, blob, off, snip, want))
    # samples at and around the snippet boundary, and two whole snippets
    toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=150, max_len=10, int_scores=True)
    samples = [bytes(rng.choice(b"abcd") for _ in range(n)) for n in (SNIP - 1, SNIP, SNIP + 1, 2 * SNIP, 5)]
    blob, off = O.pack_samples(samples)
    want, rc, _ = O.OracleModel(toks, scores).run_e_step_fixed(blob, off, threads=8)
    assert rc == 0
    cases.append((toks, scores, blob, off, SNIP, want))
    return cases


@pytest.fixture(scope="module")
def synth_case():
    """The corpus of test_expected_counts_synth_vs_oracle: 2 MB, 30 000 tokens (ids on both sides of hot_k)."""
    blob, off, toks, sc, kp = synth_setup(2, 13, 2_000_000, 30000, 16)
    want, rc, _ = O.OracleModel(toks, sc).run_e_step_fixed(blob, off, threads=8)
    assert rc == 0
    return toks, sc, blob, off, want


@pytest.mark.parametrize("g", KERNEL_SETS)
def test_limbs_exact_random_vocabularies(N, random_cases, g):
    for i, (toks, scores, blob, off, snip, want) in enumerate(random_cases):
        gm = N.Model(toks, scores, device=0)
        configure(gm, g)
        assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off, snip=snip), len(toks)), want, (g, i))


@pytest.mark.parametrize("g", KERNEL_SETS)
def test_limbs_exact_synth_corpus(N, synth_case, g):
    toks, sc, blob, off, want = synth_case
    gm = N.Model(toks, sc, device=0)
    configure(gm, g)
    assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off), len(toks)), want, g)


# ----------------------------------------------------------------------------- accumulator paths
def test_replica_shapes_and_both_paths(N, synth_case):
    """Options 20 / 21 (replicas of the hot ids / number of hot ids): (64, 0) sends every atomic to acc; the 30 000-token
    vocabulary has ids on both sides of hot_k, so both paths run in one call."""
    toks, sc, blob, off, want = synth_case
    gm = N.Model(toks, sc, device=0)
    for r, k in ((1, 4096), (64, 0), (7, 1), (4096, 16)):
        gm.set_option(20, r)
        gm.set_option(21, k)
        assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off), len(toks)), want, (r, k))


@pytest.mark.parametrize("r,k", [(64, 4096), (64, 0), (3, 1)])
def test_one_heavy_token_carries_into_the_integer_part(N, r, k):
    """500 000 bytes of 'a' where 'a' carries most of the mass: its fraction words carry into the integer part many
    times, in the replicas and in acc."""
    toks, scores = [b"a", b"aa", b"aaa", b"b"], [-0.05, -4.0, -6.5, -3.0]
    samples = [b"a" * 500_000, b"ab" * 1000, b"a" * 7]
    blob, off = O.pack_samples(samples)
    want, rc, _ = O.OracleModel(toks, scores).run_e_step_fixed(blob, off, threads=8)
    assert rc == 0 and want[0] > 400_000 * ONE
    gm = N.Model(toks, scores, device=0)
    gm.set_option(20, r)
    gm.set_option(21, k)
    for g in (0, 4, "split"):
        configure(gm, g)
        assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off), len(toks)), want, (r, k, g))


# ----------------------------------------------------------------------------- keyed dropout
@pytest.mark.parametrize("p", [0.3, 0.7])
def test_keyed_dropout_limbs_exact(N, p):
    rng = random.Random(int(p * 100))
    for it in range(4):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(8, 80), max_len=rng.randrange(2, 12),
                                  int_scores=(it % 2 == 0))
        om, gm = O.OracleModel(toks, scores), N.Model(toks, scores, device=0)
        samples = rand_samples(rng, b"abcd", 60, 1, 300) + rand_samples(rng, b"abcd", 2, 2000, 4000)
        blob, off = O.pack_samples(samples)
        seed, base, snip = [(11, 0, SNIP), (2 ** 62 + 5, 123456, 300)][it % 2]
        want, rc, _ = om.run_e_step_fixed(blob, off, p, seed, keyed=True, byte_base=base, threads=8,
                                          max_sample_length=snip)
        assert rc == 0
        gm.set_option(22, base)
        gm.set_dropout(p, seed)
        for g in (0, -2, 4, 32):
            configure(gm, g)
            assert_limbs_equal(limbs_to_ints(run_fixed(gm, blob, off, snip=snip), len(toks)), want, (it, g))


# ----------------------------------------------------------------------------- calls, shards, state
def test_calls_and_simulated_ranks_add_up(N):
    """Limbs are an exact sum, so two calls into one buffer = one call on the concatenation = the oracle, and k shards
    (each with its byte offset as option 22) summed as int64 — what an NCCL all-reduce does — convert to the one-call
    counts bit for bit."""
    import torch
    blob, off, toks, sc, kp = synth_setup(2, 17, 1_500_000, 20000, 16)
    om, gm = O.OracleModel(toks, sc), N.Model(toks, sc, device=0)
    V, S = len(toks), len(off) - 1
    for p, seed in ((0.0, 0), (0.3, 5)):
        gm.set_option(22, 0)
        gm.set_dropout(p, seed)
        want, rc, _ = om.run_e_step_fixed(blob, off, p, seed, keyed=True, threads=8)
        assert rc == 0
        whole = run_fixed(gm, blob, off)
        assert_limbs_equal(limbs_to_ints(whole, V), want, p)
        d_whole = torch.empty(V, dtype=torch.float64, device="cuda")
        gm.counts_from_limbs_dev(whole.data_ptr(), V, d_whole.data_ptr())
        assert_same_bits(d_whole.cpu().numpy(), nearest(want), p)
        for k in (2, 3, 8):
            cuts = [S * i // k for i in range(k + 1)]
            total = torch.zeros_like(whole)
            two = new_limbs(V)
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                b = blob[int(off[lo]):int(off[hi])]
                o = (off[lo:hi + 1] - off[lo]).astype(np.uint64)
                gm.set_option(22, int(off[lo]))
                total += run_fixed(gm, b, o)
                if k == 2:
                    run_fixed(gm, b, o, limbs=two)  # both calls into one buffer
            d_ex = torch.empty(V, dtype=torch.float64, device="cuda")
            gm.counts_from_limbs_dev(total.data_ptr(), V, d_ex.data_ptr())
            assert_same_bits(d_ex.cpu().numpy(), d_whole.cpu().numpy(), (p, k))
            if k == 2:
                assert_limbs_equal(limbs_to_ints(two, V), want, (p, "two calls"))
    gm.set_dropout(0.0, 0)
    gm.set_option(22, 0)


def test_no_state_leaks_between_calls_or_rebuilds(N):
    """A call after a different call on the same model sees fresh accumulators; after Model.rebuild in place to a
    subset vocabulary (the EM loop's sequence) the limbs equal the oracle of the new vocabulary."""
    blob, off, toks, sc, kp = synth_setup(2, 13, 2_000_000, 30000, 16)
    gm = N.Model(toks, sc, device=0)
    h = (len(off) - 1) // 2
    b1, o1 = blob[:int(off[h])], off[:h + 1].copy()
    b2, o2 = blob[int(off[h]):], (off[h:] - off[h]).astype(np.uint64)
    om = O.OracleModel(toks, sc)
    want2 = om.run_e_step_fixed(b2, o2, threads=8)[0]
    run_fixed(gm, b1, o1)
    assert_limbs_equal(limbs_to_ints(run_fixed(gm, b2, o2), len(toks)), want2, "after another call")
    # a subset vocabulary: every single byte of the corpus kept, then every other token
    rng = random.Random(3)
    keep = [i for i, t in enumerate(toks) if len(t) == 1 or rng.random() < 0.5]
    t2 = [toks[i] for i in keep]
    s2 = np.asarray(sc, np.float64)[keep] - 0.25
    gm.rebuild(t2, s2)
    want = O.OracleModel(t2, s2).run_e_step_fixed(b2, o2, threads=8)[0]
    assert_limbs_equal(limbs_to_ints(run_fixed(gm, b2, o2), len(t2)), want, "after rebuild")


# ----------------------------------------------------------------------------- conversion
def conversion_cases():
    rng = random.Random(99)
    M32 = 0xFFFFFFFF
    rows = []
    for _ in range(4000):  # random words
        rows.append([rng.getrandbits(32) for _ in range(4)] + [rng.choice([0, 1, rng.getrandbits(20),
                                                                           rng.getrandbits(62)])])
    for _ in range(2000):  # sums over up to 1024 ranks, carries pending in every limb
        r = rng.randrange(1, 1025)
        rows.append([rng.randrange(0, r * 1024 * M32 + 1) for _ in range(4)] + [rng.randrange(0, r * 1024 + 1)])
    rows += [[M32] * 4 + [ip] for ip in (0, 1, 2 ** 53 - 1, 2 ** 53)]  # all-ones words: carries through every limb
    rows += [[1024 * 1024 * M32] * 4 + [0], [1024 * M32] * 5]
    xs = [0, 1, 2, 3, (1 << 128) - 1, ONE + 1]  # zero, the smallest value 2^-128, ...
    xs.append((0x20000000000725 << 64) | 0x63ca828dd5f4b3b2)  # rounds differently in the previous f64 formula
    for k in range(-127, 62):  # around 0.5, 1 and every power of two
        base = 1 << (128 + k)
        for d in (1, 2, 3, 1 << 40, (1 << 74) - 1, 1 << 74, (1 << 74) + 1):
            xs += [base - d, base + d] if d < base else [base + d]
    for ip in (2 ** 53, 2 ** 53 + 1, 2 ** 54 + 3, 2 ** 60 + 7, 2 ** 62):  # integer parts past 2^53: ties and halves
        xs += [ip * ONE, ip * ONE + (1 << 127), ip * ONE + (1 << 127) + 1, ip * ONE + (1 << 127) - 1, ip * ONE + 1]
    rows += ints_to_limbs(xs)
    return rows


def test_conversion_is_correctly_rounded(N):
    gm = N.Model([b"a"], [-1.0], device=0)
    rows = conversion_cases()
    want = nearest([l0 + (l1 << 32) + (l2 << 64) + (l3 << 96) + (l4 << 128) for l0, l1, l2, l3, l4 in rows])
    assert_same_bits(convert(N, gm, rows), want)


def test_expected_counts_f64_is_the_rounded_exact_sum(N, random_cases):
    """tgx_expected_counts returns the nearest f64 to the oracle's exact sum; tgx_expected_counts_dev adds that value
    to what d_expected held (+=)."""
    import torch
    for i, (toks, scores, blob, off, snip, want) in enumerate(random_cases):
        gm = N.Model(toks, scores, device=0)
        ex, rc, *_ = gm.expected_counts(blob, off, snippet_len=snip)
        assert rc == 0
        assert_same_bits(ex, nearest(want), i)
        prefill = np.random.default_rng(i).uniform(-3.0, 1e6, len(toks))
        d_ex = torch.from_numpy(prefill.copy()).cuda()
        d_text, d_off = to_dev(blob, off)
        rc, bad, _ = gm.expected_counts_dev(d_text.data_ptr(), d_off.data_ptr(), len(off) - 1, int(off[-1]),
                                            d_ex.data_ptr(), snippet_len=snip)
        assert rc == 0
        assert_same_bits(d_ex.cpu().numpy(), prefill + nearest(want), i)
