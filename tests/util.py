"""Shared helpers for the test-suite (seeded vocabularies / corpora)."""
import functools
import random

import numpy as np


def rand_vocab(rng, alphabet=b"abc", n_tok=12, max_len=4, complete=True, int_scores=False):
    n_possible = sum(len(alphabet) ** l for l in range(1, max_len + 1))
    n_tok = min(n_tok, n_possible)
    toks = set()
    if complete:
        toks |= {bytes([c]) for c in alphabet}
    while len(toks) < n_tok:
        toks.add(bytes(rng.choice(alphabet) for _ in range(rng.randrange(1, max_len + 1))))
    toks = sorted(toks)
    rng.shuffle(toks)
    if int_scores:  # many exact ties (SURVEY H2)
        scores = [-float(rng.randrange(2, 6)) for _ in toks]
    else:
        scores = [-(rng.random() * 6 + 0.5) for _ in toks]
    return toks, scores


def rand_samples(rng, alphabet, n, lo, hi):
    return [bytes(rng.choice(alphabet) for _ in range(rng.randrange(lo, hi))) for _ in range(n)]


@functools.lru_cache(maxsize=4)
def synth_setup(kind: int, seed: int, nbytes: int, vocab_size: int, max_len: int):
    """(blob, off, tokens, scores, keep) — cached per session."""
    from tokengeex_b200 import synth
    blob, off = synth.corpus(kind, seed, nbytes)
    toks, sc, kp = synth.vocab(blob, off, seed, vocab_size, max_len, 0.05)
    return blob, off, toks, sc, kp


def estep_cfg(m, g):
    """E-step kernel set of a device Model.  g = lanes per snippet of the lane-group kernels (lane-per-snippet kernels
    off); g = 0: every snippet below the long threshold runs one lane each (fb_*_lane_kernel), the rest a warp each."""
    if g in (0, -2, -3):  # 0: split form, lane kernels that walk the trie (the default); -2: the lane kernels over the
        m.set_option(17, 1 << 30)  # match stream; -3: no beta array (fused backward + counts on the lane-group kernels)
        m.set_option(2, 4)
        m.set_option(19, {0: 1, -2: 2, -3: 0}[g])
    else:
        m.set_option(17, 0)
        m.set_option(2, g)


def fixed_point_samples(om, samples, snip, limit=2.0 ** 64):
    """The samples whose every snippet has a path (z normal, so the E-step reports no error) and whose contributions
    are all below `limit`.  The device's 192-bit accumulators hold contributions below 2^64; only a lattice with
    positions nothing begins at (incomplete vocabularies: beta = log 1 there) can have larger ones."""
    import math
    out = []
    for s in samples:
        ok = True
        for o in range(0, len(s), snip):
            z, cs = om.marginal_contributions(s[o:o + snip])
            ok = ok and math.isfinite(z) and z != 0.0 and all(c < limit for _, c in cs)
        if ok:
            out.append(s)
    return out


def split_ids(ids: np.ndarray, id_off: np.ndarray):
    return [ids[int(id_off[i]):int(id_off[i + 1])].tolist() for i in range(len(id_off) - 1)]


# The kernels accumulate expected counts in fixed point with 2^-128 resolution (exact, order-independent sums: see
# include/tokengeex_b200.h), so a count is compared relatively where it is large enough to be resolved and absolutely
# below that (the M-step's only threshold is 0.5: src/prune.rs:132).
COUNT_RESOLVED = 1e-18
COUNT_ABS = 1e-27


def counts_rel_err(got: np.ndarray, want: np.ndarray) -> float:
    """max relative error over the counts >= COUNT_RESOLVED; asserts the rest agree to COUNT_ABS and that tokens the
    oracle never counts stay exactly zero."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    big = want >= COUNT_RESOLVED
    small = ~big
    assert np.all(np.abs(got[small] - want[small]) <= COUNT_ABS), float(np.abs(got[small] - want[small]).max())
    assert np.all(got[want == 0] == 0)
    return float(np.max(np.abs(got[big] - want[big]) / want[big])) if big.any() else 0.0
