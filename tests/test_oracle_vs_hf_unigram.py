"""Weak secondary cross-check of the oracle (SURVEY §8c): HuggingFace `tokenizers`' Unigram model is the upstream the
reference's Viterbi was "imported and modified from" (src/model.rs:1-2, src/lattice.rs:1-2).  It steps over chars and
has unk handling, so it is not an oracle — but on text whose every char is in the vocabulary its best segmentation,
including the choice among exactly tied paths, must be the reference's (smallest start wins, SURVEY Q3).

HF's ids for every case are stored in tests/golden/hf_unigram_ids.json (tools/make_hf_golden.py), so the oracle is
checked against them whether or not `tokenizers` is installed; where it is, HF must still give the stored ids."""
import json
import os
import random

import pytest

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hf_unigram_ids.json")
CHARS = ["abcd", "你好世界"]


def _hf(toks, scores):
    from tokenizers import Tokenizer, models
    # the unk token is a char that never occurs (HF fuses consecutive unk ids)
    return Tokenizer(models.Unigram([(t.decode(), s) for t, s in zip(toks, scores)] + [("⁇", -100.0)],
                                    unk_id=len(toks), byte_fallback=False))


def _vocab(rng, chars, n_tok, max_len, int_scores):
    toks = set(chars)
    n_tok = min(n_tok, sum(len(chars) ** l for l in range(1, max_len + 1)))
    while len(toks) < n_tok:
        toks.add("".join(rng.choice(chars) for _ in range(rng.randrange(1, max_len + 1))))
    toks = sorted(toks)
    rng.shuffle(toks)
    scores = [-float(rng.randrange(2, 6)) if int_scores else -(rng.random() * 6 + 0.5) for _ in toks]
    return [t.encode() for t in toks], scores


def cases(chars):
    """→ (tokens, scores, 40 texts) per vocabulary of the comparison, drawn from a generator seeded by `chars`."""
    rng = random.Random(len(chars[0].encode()))
    for it in range(30):
        toks, scores = _vocab(rng, chars, rng.randrange(6, 60), rng.randrange(2, 6), int_scores=(it % 2 == 0))
        if max(len(t) for t in toks) > 64:
            continue
        yield toks, scores, ["".join(rng.choice(chars) for _ in range(rng.randrange(1, 60))) for _ in range(40)]


@pytest.mark.parametrize("chars", CHARS)
def test_oracle_encode_equals_hf_unigram(chars):
    with open(GOLDEN) as f:
        golden = json.load(f)[chars]
    try:
        import tokenizers  # noqa: F401
        live = True
    except ImportError:
        live = False
    n = 0
    for it, ((toks, scores, texts), want) in enumerate(zip(cases(chars), golden, strict=True)):
        om, hf = O.OracleModel(toks, scores), _hf(toks, scores) if live else None
        for s, ids in zip(texts, want, strict=True):
            if hf is not None:
                assert hf.encode(s).ids == ids, ("HF differs from the stored ids", it, s)
            assert om.encode(s.encode(), 0.0) == ids, (it, s)
            n += 1
    assert n >= 1000
