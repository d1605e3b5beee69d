"""File → token ids: today's host path against corpus.encode_file, on one GPU.

Writes a seeded NUL-separated synthetic corpus (kind 3, 131k-token vocabulary: the benchmark's configuration) under
--out, then times, after a warm-up and with the corpus file in the page cache (it has just been written and read):
  (a) cli.load_sources + _native.pack + Model.encode_batch + writing the arrays;
  (b) corpus.encode_file.
The tokenizer is passed as an object (encode_file then neither parses its JSON nor hashes its file).
Reports GB/s of input for both (and the time of the untimed first call), the device ms per GB of the split kernels (tgx_model_last_stat 11) and of the whole
tgx_encode_corpus call, whether both paths wrote the same bytes, and the card's name and power limit.

    python tools/bench_encode_corpus.py --out /tmp/bench_corpus [--gb 1.0] [--runs 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tokengeex_b200 import _native as N  # noqa: E402
from tokengeex_b200 import cli, corpus, synth  # noqa: E402
from tokengeex_b200.tokenizer import Tokenizer  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gb", type=float, default=1.0)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    nbytes = int(a.gb * 1e9)
    blob, off = synth.corpus(3, a.seed, nbytes)
    toks, sc, _ = synth.vocab(blob, off, a.seed, 131072, 16, 0.05)
    lens = np.diff(off).astype(np.int64)
    S = len(lens)
    data = np.zeros(int(off[-1]) + S - 1, np.uint8)
    data[np.arange(int(off[-1]), dtype=np.int64) + np.repeat(np.arange(S, dtype=np.int64), lens)] = blob[:int(off[-1])]
    src = os.path.join(a.out, "corpus.bin")
    data.tofile(src)
    tj = os.path.join(a.out, "tokenizer.json")
    Tokenizer(toks, sc).save(tj)
    del blob, off, data
    size = os.path.getsize(src)

    def path_a(prefix):
        samples = cli.load_sources([f"c:{src}"], [], "train")[0].processed_samples
        b, o = N.pack(samples)
        ids, id_off, _, _, rc, _ = model.encode_batch(b, o)
        assert rc == 0
        ids.astype(np.uint32).tofile(prefix + ".ids")
        id_off.tofile(prefix + ".idx")

    tok = Tokenizer.from_file(tj)
    model = N.Model(toks, sc, device=0)

    def path_b(prefix):
        corpus.encode_file(tok, src, prefix, dtype="uint32", dropout_seed=0)

    res = {"card": card(), "input_bytes": size, "page_cache": "the corpus file is read once before the timed runs"}
    with open(src, "rb") as f:  # into the page cache
        while f.read(1 << 26):
            pass
    for name, fn in (("a_load_sources_pack_encode_batch", path_a), ("b_corpus_encode_file", path_b)):
        t0 = time.perf_counter()
        fn(os.path.join(a.out, name))  # warm-up (path b pins its window buffers here; the timed runs reuse them)
        res[name] = {"first_call_seconds": time.perf_counter() - t0}
        ts = []
        for _ in range(a.runs):
            t0 = time.perf_counter()
            fn(os.path.join(a.out, name))
            ts.append(time.perf_counter() - t0)
        res[name].update({"seconds": ts, "GB_per_s": [size / t / 1e9 for t in ts]})
    same = all(open(os.path.join(a.out, f"a_load_sources_pack_encode_batch.{e}"), "rb").read()
               == open(os.path.join(a.out, f"b_corpus_encode_file.{e}"), "rb").read() for e in ("ids", "idx"))
    res["outputs_identical"] = same
    # device time of one tgx_encode_corpus call over the whole image from pinned memory
    buf = N.pinned_empty(size)
    with open(src, "rb") as f:
        f.readinto(memoryview(buf))
    m = tok._dev(0.0)
    ids_out = N.pinned_empty((size + 1) * 4).view(np.uint32)
    calls = []
    for _ in range(a.runs + 1):
        t0 = time.perf_counter()
        ids, id_off, rc, _, _ = m.encode_corpus(buf, ids_out=ids_out)
        calls.append((time.perf_counter() - t0, m.stat(11)))
        assert rc == 0
    calls = calls[1:]
    gb = size / 1e9
    res["encode_corpus_call_pinned"] = {"ms_per_GB_call": [c[0] * 1e3 / gb for c in calls],
                                        "ms_per_GB_split_kernels": [c[1] / gb for c in calls],
                                        "GB_per_s": [gb / c[0] for c in calls]}
    print(json.dumps(res, indent=1))
    with open(os.path.join(a.out, "result.json"), "w") as f:
        json.dump(res, f, indent=1)
    for e in ("ids", "idx", "json"):
        for name in ("a_load_sources_pack_encode_batch", "b_corpus_encode_file"):
            p = os.path.join(a.out, f"{name}.{e}")
            if os.path.exists(p):
                os.remove(p)
    os.remove(src)


if __name__ == "__main__":
    main()
