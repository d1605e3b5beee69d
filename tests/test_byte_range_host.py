"""The oracle over the whole byte range (CPU): NUL, bytes above 0x7F and 0xFF, pinned against the brute-force
enumerator, and the host walk of the device's double-array against the oracle's trie.  The device tests on these bytes
(tests/test_gpu_byte_range.py) take the oracle as their reference."""
import random

import numpy as np
import pytest

from oracle import oracle as O
from tests import bruteforce as BF
from tests.util import (BYTE_ALPHABETS, MIXED_SINGLES, byte_samples, byte_vocab, mixed_script_samples,
                        mixed_script_setup, rand_samples, wide_samples, wide_vocab)


@pytest.mark.parametrize("name", list(BYTE_ALPHABETS))
def test_oracle_encode_and_marginal_vs_bruteforce(name):
    """Tiny vocabularies over the byte alphabets with the hand-placed NUL / 0xFF tokens: Viterbi under the first-wins
    tie rule, NoPath, and (where every byte of the text is a token) the marginals, against every enumerated
    segmentation."""
    alphabet = BYTE_ALPHABETS[name]
    small = alphabet if len(alphabet) <= 6 else bytes([0x00, 0x80, 0xFF]) + alphabet[-3:]
    rng = random.Random(40 + len(alphabet))
    for it in range(60):
        complete = it % 3 != 2
        toks, scores = byte_vocab(rng, small, n_tok=rng.randrange(4, 14), max_len=4, complete=complete,
                                  int_scores=(it % 2 == 0))
        om = O.OracleModel(toks, scores)
        texts = rand_samples(rng, small + b"x", 6, 0, 10)
        texts += [b"\x00" * rng.randrange(1, 9), b"x\x00", b"x", b"a\x00\x00", b"\xff" * rng.randrange(1, 9)]
        for text in texts:
            want = BF.viterbi_first_wins(text, toks, scores)
            if want is None:
                with pytest.raises(O.NoPath) as ei:
                    om.encode(text, 0.0)
                assert (ei.value.pos, ei.value.length) == (len(text), len(text))
                continue
            assert om.encode(text, 0.0) == want, (it, text)
            # (the marginals of a lattice with dead ends keep log 1 there, src/lattice.rs:275-287: not a sum over paths)
            if not text or any(bytes([c]) not in toks for c in text):
                continue
            logz, ex = BF.marginals(text, toks, scores)
            z, got = om.marginal(text, literal=True)
            assert abs(z - logz) < 1e-12, (it, text)
            assert np.allclose(got, ex, rtol=1e-11, atol=1e-14), (it, text)


def test_oracle_nopath_on_nul_without_nul_tokens():
    """NUL in the text and no token with a NUL in it: NoPath at the sample's length, and no match of any token across
    the NUL."""
    toks = [bytes([b]) for b in range(0x80, 0x100)] + [b"\x80\x81", b"\xff\xff"]
    om = O.OracleModel(toks, [-3.0] * 128 + [-4.0, -5.0])
    for text in (b"\x00", b"\x80\x00", b"\x00\x80", b"\xff\x00\xff", b"\x80\x81" * 5 + b"\x00"):
        with pytest.raises(O.NoPath) as ei:
            om.encode(text, 0.0)
        assert (ei.value.pos, ei.value.length) == (len(text), len(text))
        assert BF.viterbi_first_wins(text, toks, [-3.0] * 128 + [-4.0, -5.0]) is None
    assert om.common_prefix_search(b"\x00\x80") == ([], [])


def common_prefix_everywhere(hm, om, text):
    for i in range(len(text)):
        assert hm.common_prefix_search(text[i:]) == om.common_prefix_search(text[i:]), (i, text[i:i + 16])


def test_common_prefix_search_wide_vocabulary():
    """The host walk of the double-array (a host-only Model) and the oracle's trie yield the same (id, length) lists
    from every start of the wide vocabulary's texts: 256-way fan-out at the root and at depth 1, NUL and 0xFF."""
    from tokengeex_b200 import _native as N
    toks, scores = wide_vocab()
    hm = N.Model(list(toks), list(scores), device=None)
    om = O.OracleModel(list(toks), list(scores))
    rng = random.Random(8)
    for text in wide_samples(rng, toks, n=20, hi=120):
        common_prefix_everywhere(hm, om, text)


@pytest.mark.parametrize("name", list(BYTE_ALPHABETS))
def test_common_prefix_search_byte_vocabularies(name):
    """The same over the byte alphabets, with and without the NUL tokens: a NUL probe from a root whose base is 0
    lands on the root's own slot, which must read as empty."""
    from tokengeex_b200 import _native as N
    alphabet = BYTE_ALPHABETS[name]
    rng = random.Random(60 + len(alphabet))
    for it in range(6):
        toks, scores = byte_vocab(rng, alphabet, n_tok=rng.randrange(10, 200), max_len=rng.randrange(2, 17),
                                  complete=(it % 2 == 0), edges=(it % 3 != 2))
        if it % 3 == 2:  # no token with a NUL in it
            keep = [i for i, t in enumerate(toks) if 0 not in t]
            toks, scores = [toks[i] for i in keep], [scores[i] for i in keep]
        hm = N.Model(toks, scores, device=None)
        om = O.OracleModel(toks, scores)
        for text in byte_samples(rng, alphabet + b"\x00", toks, n=8, hi=60):
            common_prefix_everywhere(hm, om, text)


def test_generators_are_deterministic():
    rng1, rng2 = random.Random(3), random.Random(3)
    for name, alphabet in BYTE_ALPHABETS.items():
        v1 = byte_vocab(rng1, alphabet, complete=False, int_scores=True, long=True)
        v2 = byte_vocab(rng2, alphabet, complete=False, int_scores=True, long=True)
        assert v1 == v2, name
        assert byte_samples(rng1, alphabet, v1[0]) == byte_samples(rng2, alphabet, v2[0]), name
    assert wide_samples(random.Random(4), wide_vocab()[0]) == wide_samples(random.Random(4), wide_vocab()[0])
    assert mixed_script_samples(9) == mixed_script_samples(9)
    s = mixed_script_setup()
    mixed_script_setup.cache_clear()
    assert mixed_script_setup() == s
    toks, _ = wide_vocab()
    assert len(toks) == len(set(toks)) == 256 + 65536 + 3000
    texts = b"".join(s[0]).decode("utf-8")
    assert all(c in texts for c in MIXED_SINGLES)
    assert all(bytes([b]) in s[1] for b in range(256))
