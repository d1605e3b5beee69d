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


# ----------------------------------------------------------------------------- the whole byte range
# Alphabets beyond 'a'..'d': NUL (label 0 lands a child on its parent's base; the text is padded with zero bytes past
# the blob's end), bytes with the high bit set (sign / mask slips when a kernel pulls a byte out of a word), 0xFF (the
# far end of a 256-slot block) and CR / LF next to them.
BYTE_ALPHABETS = {
    "all": bytes(range(256)),
    "edges": bytes([0x00, 0x01, 0x7F, 0x80, 0xFE, 0xFF]),
    "high": bytes(range(0x80, 0x100)),
    "nul_a": b"\x00a",
    "crlf": b"\r\n\x00\xffa",
}


def byte_edge_tokens():
    """Hand-placed tokens: ending in NUL, only NUL (up to 16 bytes), starting with NUL, runs of 0xFF up to 16 bytes, and
    b"a" next to b"a\\x00" (same bytes but one, different length)."""
    toks = [b"x", b"x\x00", b"x\x00\x00", b"\x00x", b"\x00\xff", b"\xff\x00", b"a", b"a\x00", b"\x00a\x00"]
    toks += [b"\x00" * k for k in range(1, 17)] + [b"\xff" * k for k in range(1, 17)]
    return toks


def byte_vocab(rng, alphabet, n_tok=40, max_len=6, complete=True, int_scores=False, edges=True, long=False):
    """rand_vocab over `alphabet`, plus byte_edge_tokens (edges) and a few tokens longer than 16 bytes (long: the
    lane-group kernels then take every sample)."""
    toks, scores = rand_vocab(rng, alphabet=alphabet, n_tok=n_tok, max_len=max_len, complete=complete,
                              int_scores=int_scores)
    extra = byte_edge_tokens() if edges else []
    if long:
        extra += [alphabet[:1] * 17, b"\x00" * 24, bytes(rng.choice(alphabet) for _ in range(21))]
    have = set(toks)
    extra = [t for t in dict.fromkeys(extra) if t not in have]
    for t in extra:
        toks.append(t)
        scores.append(-float(rng.randrange(2, 6)) if int_scores else -(rng.random() * 6 + 0.5))
    return toks, scores


def byte_samples(rng, alphabet, toks, n=40, hi=200):
    """Random samples over the alphabet, NUL-heavy ones, runs of vocabulary tokens (long matches), NUL / 0xFF runs and
    an empty sample."""
    out = rand_samples(rng, alphabet, n, 0, hi)
    nul_heavy = b"\x00" * 6 + alphabet
    out += rand_samples(rng, nul_heavy, 10, 1, hi)
    out += [b"".join(rng.choice(toks) for _ in range(rng.randrange(1, 30))) for _ in range(12)]
    out += [b"\x00" * k for k in (1, 2, 15, 16, 17, 33)] + [b"\xff" * k for k in (1, 16, 17, 40)] + [b""]
    rng.shuffle(out)
    return out


@functools.lru_cache(maxsize=2)
def wide_vocab(seed=7, n_long=3000):
    """All 256 single bytes, all 65 536 two-byte strings and n_long random longer tokens (3..16 bytes): a root with 256
    children, depth-1 nodes with 256 children each (the second trie level does not fit the shared-memory stage), every
    entry of the two-byte walk table used, ids of 65 536 and above.  Scores from a small integer set for a quarter of
    the tokens (exact ties)."""
    rng = random.Random(seed)
    toks = [bytes([b]) for b in range(256)] + [bytes([a, b]) for a in range(256) for b in range(256)]
    longs = set()
    while len(longs) < n_long:
        longs.add(bytes(rng.randrange(256) for _ in range(rng.randrange(3, 17))))
    toks += sorted(longs)
    scores = [-float(rng.randrange(3, 7)) if rng.random() < 0.25 else -(rng.random() * 8 + 1.0) for _ in toks]
    return tuple(toks), tuple(scores)


def wide_samples(rng, toks, n=60, hi=400):
    """Random bytes over the full range, runs of the wide vocabulary's longer tokens, NUL and 0xFF runs."""
    longs = [t for t in toks if len(t) > 2]
    out = rand_samples(rng, bytes(range(256)), n, 0, hi)
    out += [b"".join(rng.choice(longs) for _ in range(rng.randrange(1, 40))) for _ in range(n // 2)]
    out += [b"\x00" * 37, b"\xff" * 41, b"\x00\xff" * 30, b"\xff\x00" * 3 + b"\xff"]
    rng.shuffle(out)
    return out


# code points of the mixed-script corpus: ASCII, two-byte UTF-8 (U+0080..U+07FF), Cyrillic, CJK, four-byte emoji
MIXED_RANGES = [(0x21, 0x7E), (0x80, 0x7FF), (0x400, 0x4FF), (0x4E00, 0x9FFF), (0x1F300, 0x1FAFF)]
MIXED_SINGLES = ["\ufffd", "\U0010ffff", "\u0080", "\u07ff", "\u0800", "\uffff", "\U00010000"]


def mixed_script_samples(seed, n=400, max_words=60):
    """Seeded UTF-8 samples: words drawn from a per-script lexicon (so that a vocabulary learns multi-byte tokens),
    separated by spaces, newlines and CRLF, with U+FFFD, U+10FFFF and the UTF-8 length boundaries sprinkled in."""
    rng = random.Random(seed)
    lexicon = []
    for lo, hi in MIXED_RANGES:
        for _ in range(40):
            lexicon.append("".join(chr(rng.randint(lo, hi)) for _ in range(rng.randrange(1, 7))))
    lexicon += MIXED_SINGLES
    out = []
    for _ in range(n):
        words = [rng.choice(lexicon) for _ in range(rng.randrange(1, max_words))]
        out.append("".join(w + rng.choice([" ", " ", " ", "\n", "\r\n", "\t"]) for w in words).encode("utf-8"))
    return out


@functools.lru_cache(maxsize=2)
def mixed_script_setup(seed=5, n=400, vocab_size=3000, max_len=16):
    """(samples, tokens, scores): the mixed-script corpus, a vocabulary learnt from it by synth.vocab, and the 256
    single bytes that the vocabulary lacks (every byte string then has a path)."""
    from tokengeex_b200 import synth
    samples = mixed_script_samples(seed, n)
    lens = np.fromiter(map(len, samples), np.uint64, len(samples))
    off = np.zeros(len(samples) + 1, np.uint64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b"".join(samples), np.uint8).copy()
    toks, sc, kp = synth.vocab(blob, off, seed, vocab_size, max_len, 0.05)
    toks = list(toks)
    sc = [float(x) for x in sc]
    have = set(toks)
    for b in range(256):
        if bytes([b]) not in have:
            toks.append(bytes([b]))
            sc.append(-14.0)
    return tuple(samples), tuple(toks), tuple(sc)


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
