#!/usr/bin/env python
"""Writes tests/golden/hf_unigram_ids.json: the ids HuggingFace `tokenizers`' Unigram model gives for every case of
tests/test_oracle_vs_hf_unigram.py, one line per vocabulary (needs `tokenizers`; stored from version 0.22.2).

    python tools/make_hf_golden.py            # rewrites the golden file
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import tokenizers  # noqa: E402

from tests.test_oracle_vs_hf_unigram import CHARS, GOLDEN, _hf, cases  # noqa: E402


def main():
    parts = []
    for chars in CHARS:
        rows = []
        for toks, scores, texts in cases(chars):
            hf = _hf(toks, scores)
            rows.append(json.dumps([hf.encode(s).ids for s in texts], separators=(",", ":")))
        parts.append(json.dumps(chars, ensure_ascii=False) + ":[\n" + ",\n".join(rows) + "\n]")
    with open(GOLDEN, "w", encoding="utf-8") as f:
        f.write("{" + ",\n".join(parts) + "}\n")
    print(GOLDEN, os.path.getsize(GOLDEN), "bytes, tokenizers", tokenizers.__version__)


if __name__ == "__main__":
    main()
