"""Rows a1/a2 on the host: the product's double-array trie (csrc/trie_build.cpp, the structure every kernel walks)
against the oracle's restatement of the reference's pointer trie (src/trie.rs), through
tgx_model_common_prefix_search — no device needed.  Random vocabularies with duplicates (last id wins, Q1), empty
tokens (never yielded), all 256 byte values, tokens up to the 64-byte limit; and the builder's density."""
import random

import numpy as np
import pytest

from oracle import oracle as O
from tokengeex_b200 import _native as N


def _rand_vocab(rng, alphabet, n_tok, max_len, dup_frac=0.1):
    toks = [bytes(rng.choice(alphabet) for _ in range(rng.randrange(0 if rng.random() < 0.02 else 1, max_len + 1)))
            for _ in range(n_tok)]
    for _ in range(int(n_tok * dup_frac)):
        toks.append(rng.choice(toks))  # duplicates: the later id must win
    rng.shuffle(toks)
    return toks, [-(rng.random() * 8 + 0.1) for _ in toks]


@pytest.mark.parametrize("alphabet,n_tok,max_len", [(b"ab", 40, 6), (b"abcdefgh", 400, 8), (bytes(range(256)), 3000, 5),
                                                    (b"xyz", 300, 64), (bytes(range(200, 256)), 500, 16)])
def test_double_array_matches_pointer_trie(alphabet, n_tok, max_len):
    rng = random.Random(n_tok * 131 + max_len)
    toks, scores = _rand_vocab(rng, alphabet, n_tok, max_len)
    hm, om = N.Model(toks, scores, device=None), O.OracleModel(toks, scores)
    info = hm.info()
    assert info.max_token_len == max(map(len, toks))
    queries = [rng.choice(toks) + bytes(rng.choice(alphabet) for _ in range(rng.randrange(0, 8))) for _ in range(600)]
    queries += [bytes(rng.choice(alphabet) for _ in range(rng.randrange(0, 70))) for _ in range(600)] + [b""]
    for q in queries:
        assert hm.common_prefix_search(q) == om.common_prefix_search(q), q


def test_double_array_is_dense_and_byte_complete():
    rng = random.Random(9)
    toks = [bytes([b]) for b in range(255)]  # generate's byte tokens (0xFF absent, Q19)
    toks += list({bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz_ (){};=\n") for _ in range(rng.randrange(2, 17)))
                  for _ in range(20000)})
    hm = N.Model(toks, [-1.0 - (i % 97) * 0.01 for i in range(len(toks))], device=None)
    info = hm.info()
    n_nodes = len({t[:k] for t in toks for k in range(1, len(t) + 1)}) + 1
    assert n_nodes <= info.trie_slots <= 1.25 * n_nodes + 512  # the bitmap allocator packs the slots (DESIGN §1 a2)
    ids, lens = hm.common_prefix_search(bytes([0xFF]))
    assert ids == [] and lens == []
    assert hm.common_prefix_search(b"\x00")[0] == [0]


def test_rebuild_keeps_the_layout_for_a_subset_and_builds_afresh_otherwise():
    """tgx_model_rebuild with a SUBSET of the vocabulary the array was built for (what the EM loop hands over after every
    M-step and every prune step, src/prune.rs:48,53) rewrites terminals / ids / scores in place (retarget_double_array):
    common_prefix_search equals the oracle's on the new vocabulary — new ids, new scores, the tokens that went never
    yielded — for every share that is kept; below 45 % of the built size, with a token the array has no node for, or
    with option 45 = 0 the array is built afresh."""
    rng = random.Random(5)
    alpha = b"abcdefgh"
    toks = sorted({bytes(rng.choice(alpha) for _ in range(rng.randrange(1, 13))) for _ in range(6000)} | {bytes([c]) for c in alpha})
    sc = [-(rng.random() * 8 + 0.1) for _ in toks]
    hm = N.Model(toks, sc, device=None)
    slots0, built = hm.info().trie_slots, len(toks)
    for frac in (0.9, 0.7, 0.5, 0.3):
        keep = [i for i in range(len(toks)) if rng.random() < frac or len(toks[i]) == 1]
        t2, s2 = [toks[i] for i in keep], [sc[i] - 0.5 for i in keep]
        hm.rebuild(t2, s2)
        om = O.OracleModel(t2, s2)
        for _ in range(1500):
            q = rng.choice(toks) + bytes(rng.choice(alpha) for _ in range(rng.randrange(0, 6)))
            assert hm.common_prefix_search(q) == om.common_prefix_search(q), (frac, q)
        kept_layout = hm.info().trie_slots == slots0
        assert kept_layout == (len(t2) * 1000 >= built * 450), (frac, len(t2), built)
        if not kept_layout:
            slots0, built = hm.info().trie_slots, len(t2)
        toks, sc = t2, s2
    t3, s3 = toks + [b"zzzz", toks[0]], sc + [-1.0, -0.25]  # a new token, and a duplicate (the last id wins)
    hm.rebuild(t3, s3)
    om = O.OracleModel(t3, s3)
    for q in (b"zzzzab", toks[0] + b"a", toks[5]):
        assert hm.common_prefix_search(q) == om.common_prefix_search(q)
    hm.set_option(45, 0)
    with pytest.raises(N.TgxError) as ei:  # 11 is not an option key: refused like any unknown key
        hm.set_option(11, 0)
    assert ei.value.code == N.TGX_ERR_INVALID
    hm.rebuild(t3[:-3], s3[:-3])
    om = O.OracleModel(t3[:-3], s3[:-3])
    for q in (toks[0] + b"a", toks[7], b"zzzz"):
        assert hm.common_prefix_search(q) == om.common_prefix_search(q)


def test_failed_rebuild_leaves_the_model_as_it_was():
    """tgx_model_rebuild rewrites the array in place for a subset, but only after every token has been walked to its
    slot and every score checked: a vocabulary it refuses (a non-finite score; a token beyond 64 bytes after a miss)
    leaves the old vocabulary answering (include/tokengeex_b200.h: "On failure the model is unchanged")."""
    rng = random.Random(9)
    alpha = b"abcdef"
    toks = sorted({bytes(rng.choice(alpha) for _ in range(rng.randrange(1, 10))) for _ in range(4000)} | {bytes([c]) for c in alpha})
    sc = [-(rng.random() * 8 + 0.1) for _ in toks]
    hm = N.Model(toks, sc, device=None)
    om = O.OracleModel(toks, sc)
    queries = [rng.choice(toks) + bytes(rng.choice(alpha) for _ in range(rng.randrange(0, 5))) for _ in range(500)]
    before = [hm.common_prefix_search(q) for q in queries]
    assert before == [om.common_prefix_search(q) for q in queries]
    sub = [i for i in range(len(toks)) if i % 5 or len(toks[i]) == 1]
    bad_scores = [sc[i] for i in sub]
    bad_scores[len(sub) // 2] = float("inf")  # in the middle of a subset that would otherwise keep the layout
    with pytest.raises(N.TgxError):
        hm.rebuild([toks[i] for i in sub], bad_scores)
    assert [hm.common_prefix_search(q) for q in queries] == before
    with pytest.raises(N.TgxError):
        hm.rebuild([toks[i] for i in sub] + [b"x" * 65], [sc[i] for i in sub] + [-1.0])
    assert [hm.common_prefix_search(q) for q in queries] == before
    assert hm.info().vocab_size == len(toks)
    hm.rebuild([toks[i] for i in sub], [sc[i] for i in sub])  # and the same subset with good scores goes through
    om2 = O.OracleModel([toks[i] for i in sub], [sc[i] for i in sub])
    assert [hm.common_prefix_search(q) for q in queries] == [om2.common_prefix_search(q) for q in queries]
