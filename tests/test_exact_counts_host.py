"""The oracle's exact E-step sums (CPU only).

The CUDA E-step keeps every count as the exact sum of its contributions, each truncated to 2^-128 (192-bit fixed
point, include/tokengeex_b200.h).  The oracle keeps the same sums beside its f64 ones (run_e_step_fixed), so the GPU
tests can compare counts bit for bit.  Pinned here: those sums equal sum(floor(c * 2^128)) computed in Python integers
from the oracle's own list of contributions, they do not depend on the thread count or on sharding, and they describe
the same lattice as the f64 E-step.
"""
import math
import random
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import counts_rel_err, fixed_point_samples, rand_samples, rand_vocab

ONE = 1 << 128  # a count of 1.0 in the fixed-point scale


def floor_scaled(c: float) -> int:
    n, d = c.as_integer_ratio()
    return (n << 128) // d


def python_exact(om, samples, snip, dropout=0.0, seed=0, byte_base=0):
    """sum(floor(c * 2^128)) per token over the contributions of every snippet, from marginal_contributions."""
    X = [0] * om.V
    pos = byte_base
    for s in samples:
        for o in range(0, len(s), snip):
            z, cs = om.marginal_contributions(s[o:o + snip], dropout, seed, pos + o)
            assert math.isfinite(z) and z != 0.0
            for i, c in cs:
                X[i] += floor_scaled(c)
        pos += len(s)
    return X


def to_f64(X):
    return np.array([float(Fraction(x, ONE)) for x in X])


@pytest.mark.parametrize("snip", [7, 64, 81920])
@pytest.mark.parametrize("complete,int_scores", [(True, False), (True, True), (False, False), (False, True)])
def test_fixed_sums_equal_python_integer_sums(snip, complete, int_scores):
    rng = random.Random(hash((snip, complete, int_scores)) & 0xFFFF)
    for it in range(6):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(5, 40), max_len=rng.randrange(1, 8),
                                  complete=complete, int_scores=int_scores)
        om = O.OracleModel(toks, scores)
        samples = rand_samples(rng, b"abcd", rng.randrange(1, 40), 1, 300)
        if not complete:  # plus text the vocabulary covers; then only the samples with a path
            samples = fixed_point_samples(om, samples + [t * rng.randrange(1, 20) for t in toks[:3]], snip,
                                          limit=math.inf)
        blob, off = O.pack_samples(samples)
        X, rc, bad = om.run_e_step_fixed(blob, off, max_sample_length=snip)
        assert rc == 0 and bad == -1
        exact = python_exact(om, samples, snip)
        assert X == [x % (1 << 192) for x in exact], (it, snip)
        if max(exact, default=0) < 1 << 192:
            ex, wrc, *_ = om.run_e_step(blob, off, max_sample_length=snip)
            assert wrc == 0 and counts_rel_err(to_f64(X), ex) < 1e-12


def test_dead_end_contributions_past_the_integer_word():
    """A position nothing begins at keeps beta = log 1 (src/lattice.rs:275-287), so a token ending there, off every
    path, can get a contribution far above 1.  The oracle's sums are then exact modulo 2^192; the device's
    accumulators hold contributions below 2^64 only."""
    om = O.OracleModel([b"a", b"ac", b"x"], [-1.0, -1.0, -1.0])
    s = b"ac" + b"x" * 200  # nothing begins at byte 1 ('c'): 'a' gets exp(-1 + 0 - z) with z = -201
    z, cs = om.marginal_contributions(s)
    assert z == -201.0 and cs[0] == (0, math.exp(200.0))
    assert math.isfinite(z) and max(c for _, c in cs) > 2.0 ** 64
    assert fixed_point_samples(om, [s], 81920) == [] and fixed_point_samples(om, [s], 81920, math.inf) == [s]
    blob, off = O.pack_samples([s])
    X, rc, _ = om.run_e_step_fixed(blob, off)
    assert rc == 0 and X == [x % (1 << 192) for x in python_exact(om, [s], 81920)]


def test_single_path_contributions_are_one():
    """One segmentation per sample (single-byte vocabulary, integer scores): every contribution is exactly 1.0, so a
    count is exactly its number of occurrences."""
    toks = [b"a", b"b", b"c"]
    om = O.OracleModel(toks, [-1.0, -2.0, -3.0])
    samples = [b"abcabc", b"a" * 500, b"cb" * 90, b"c"]
    for s in samples:
        z, cs = om.marginal_contributions(s)
        assert z == -float(sum(b - 96 for b in s)) and all(c == 1.0 for _, c in cs)
    blob, off = O.pack_samples(samples)
    for snip in (7, 64, 81920):
        X, rc, _ = om.run_e_step_fixed(blob, off, max_sample_length=snip)
        want = [sum(s.count(t) for s in samples) * ONE for t in toks]
        assert rc == 0 and X == want == python_exact(om, samples, snip)


def test_exact_ties_integer_scores():
    """Integer scores with exact ties: 'aa' as one token or as two has the same score."""
    om = O.OracleModel([b"a", b"aa", b"b", b"ab"], [-2.0, -4.0, -3.0, -5.0])
    samples = [b"aa", b"aaaa", b"aab" * 30, b"ab" * 50]
    blob, off = O.pack_samples(samples)
    X, rc, _ = om.run_e_step_fixed(blob, off)
    assert rc == 0 and X == python_exact(om, samples, 81920)
    ex = om.run_e_step(blob, off)[0]
    assert counts_rel_err(to_f64(X), ex) < 1e-12


@pytest.mark.parametrize("p", [0.3, 0.7])
def test_keyed_dropout_fixed_sums(p):
    rng = random.Random(int(p * 10))
    for it in range(4):
        toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=rng.randrange(8, 50), max_len=rng.randrange(2, 9),
                                  int_scores=(it % 2 == 1))
        om = O.OracleModel(toks, scores)
        samples = rand_samples(rng, b"abcd", 30, 1, 200)
        blob, off = O.pack_samples(samples)
        seed, base = [(11, 0), (2 ** 62 + 5, 123456)][it % 2]
        for snip in (64, 81920):
            X, rc, _ = om.run_e_step_fixed(blob, off, p, seed, keyed=True, byte_base=base, max_sample_length=snip)
            assert rc == 0
            assert X == python_exact(om, samples, snip, p, seed, base), (it, snip)
            ex, wrc, *_ = om.run_e_step_dropout(blob, off, p, seed, keyed=True, byte_base=base, max_sample_length=snip)
            assert wrc == 0 and counts_rel_err(to_f64(X), ex) < 1e-12
            X0 = om.run_e_step_fixed(blob, off, max_sample_length=snip)[0]
            assert X != X0  # the draw changes the lattice


@pytest.mark.parametrize("dropout", [0.0, 0.3])
def test_fixed_sums_independent_of_threads_and_shards(dropout):
    """Integer sums: any thread count (chunking and merge order) and any split of the corpus into shards with their
    byte bases give the same integers."""
    rng = random.Random(5)
    toks, scores = rand_vocab(rng, alphabet=b"abcd", n_tok=60, max_len=6)
    om = O.OracleModel(toks, scores)
    samples = rand_samples(rng, b"abcd", 200, 1, 400)
    blob, off = O.pack_samples(samples)
    whole, rc, _ = om.run_e_step_fixed(blob, off, dropout, 9, max_sample_length=100)
    assert rc == 0
    for threads in (2, 3, 8):
        assert om.run_e_step_fixed(blob, off, dropout, 9, threads=threads, max_sample_length=100)[0] == whole
    S = len(off) - 1
    for cuts in ([S // 2], [1, S - 1], [S // 3, 2 * S // 3]):
        total = [0] * om.V
        for lo, hi in zip([0] + cuts, cuts + [S]):
            b = blob[int(off[lo]):int(off[hi])]
            o = (off[lo:hi + 1] - off[lo]).astype(np.uint64)
            part, rc, _ = om.run_e_step_fixed(b, o, dropout, 9, byte_base=int(off[lo]), max_sample_length=100)
            assert rc == 0
            total = [x + y for x, y in zip(total, part)]
        assert total == whole, cuts
