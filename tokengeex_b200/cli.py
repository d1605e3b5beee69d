"""`tokengeex prune` on the GPU hot path: the caller side of the EM pruning loop.

Mirrors the reference's command line for this one sub-command (/root/reference/src/cli.rs:65-86 arguments,
:455-494 `prune_cmd`) and its corpus loader (`load_sources`, :237-314):

    python -m tokengeex_b200.cli prune -i in.json -o out.json -v 65536 \\
        --train code:./data/train/code.bin:0.5 --train zh:./data/train/zh.bin \\
        --dropout 0.0 --shrink-factor 0.8 --em-subiters 2

`encode` pretokenizes one corpus file to token ids on disk (tokengeex_b200/corpus.py):

    python -m tokengeex_b200.cli encode -i tokenizer.json --input corpus.bin -o out/prefix --separator "<eos>"

A source is `name:path[:proportion]`; the file holds samples separated by NUL bytes (docs/DATASET.md:69); every
sample must be valid UTF-8; empty samples are dropped; `floor(count * proportion)` samples are taken from the front;
the tokenizer's processors are applied and samples that became empty are dropped.  The reference then shuffles the
samples with an unseeded RNG (:370-379), which only changes the order of f64 additions in the E-step; here the
order is the file order unless --shuffle-seed is given.

--dropout defaults to 0.01 like the reference (src/cli.rs:687): every multi-byte match of the E-step lattice is dropped
with that probability (src/model.rs:48-50).  The reference draws from an unseeded thread RNG; here the draw is keyed
(seed, byte offset in the corpus, token length: include/tokengeex_b200.h, tgx_model_set_dropout), fresh per run unless
--dropout-seed is given, and independent of the number of GPUs.  --dropout 0.0 (the benchmark configurations) runs
the faster default E-step kernels.  Under torchrun (WORLD_SIZE > 1) every rank
loads the same sources, keeps a byte-balanced shard of the samples and all-reduces the count vectors (dist.py).
"""
from __future__ import annotations

import argparse
import logging
import os
import random
import sys
from dataclasses import dataclass
from typing import List, Optional, Sequence

log = logging.getLogger("tokengeex_b200.cli")


@dataclass
class Source:
    """`struct Source` of src/cli.rs: one training file after loading."""
    name: str
    processed_samples: List[bytes]
    total_samples: int
    total_bytes: int
    processed_total_bytes: int


def parse_source(spec: str):
    """`{name}:{path}[:{proportion}]` (src/cli.rs:240-256)."""
    pieces = spec.split(":")
    if len(pieces) < 2 or len(pieces) > 3:
        raise ValueError(f"Invalid source format: {spec!r}. Expected to be formatted as {{name}}:{{path}}")
    proportion = 1.0
    if len(pieces) == 3:
        try:
            proportion = float(pieces[2])
        except ValueError:
            raise ValueError(f"Invalid proportion {pieces[2]!r} in source {spec!r}") from None
    return pieces[0], pieces[1], proportion


def load_sources(sources: Sequence[str], processors=(), mode: str = "train") -> List[Source]:
    """src/cli.rs:237-314.  `processors`: objects with `.preprocess(str) -> str` (tokenizer._Processor)."""
    out = []
    for spec in sources:
        name, path, proportion = parse_source(spec)
        with open(path, "rb") as f:
            contents = f.read()
        samples = []
        for piece in contents.split(b"\x00"):
            if not piece:
                continue
            try:
                samples.append(piece.decode("utf-8"))
            except UnicodeDecodeError as e:
                raise ValueError(f"Sample in {path!r} is not valid UTF-8: {e}") from None
        total_bytes = sum(len(s.encode("utf-8")) for s in samples)
        take = int(len(samples) * proportion)  # `as usize`: truncation
        processed = []
        for s in samples[:max(take, 0)]:
            for p in processors:
                s = p.preprocess(s)
            if s:
                processed.append(s.encode("utf-8"))
        src = Source(name, processed, len(samples), total_bytes, sum(len(s) for s in processed))
        log.info("Loaded %d/%d samples from %r %s source (%.2fMB)", len(processed), len(samples), name, mode,
                 src.processed_total_bytes / 1e6)
        out.append(src)
    return out


def prune_cmd(input: str, output: str, vocab_size: int, train: Sequence[str], dropout: float = 0.0,
              shrink_factor: float = 0.8, em_subiters: int = 1, device: Optional[int] = None,
              shuffle_seed: Optional[int] = None, dropout_seed: Optional[int] = None):
    """src/cli.rs:455-494.  Returns the PruneReport of the run."""
    from . import _native as N
    from . import dist
    from .prune import ModelVocabularyPruner, Vocab
    from .tokenizer import Tokenizer

    if not (0.0 <= dropout < 1.0):
        raise ValueError("--dropout must be in [0, 1)")
    log.info("Pruning vocabulary input=%r output=%r vocab_size=%d dropout=%s shrink_factor=%s em_subiters=%d", input,
             output, vocab_size, dropout, shrink_factor, em_subiters)
    tok = Tokenizer.from_file(input)
    initial = tok.base_vocab_size()
    sources = load_sources(train, tok._processors, "train")
    samples = [s for src in sources for s in src.processed_samples]
    if shuffle_seed is not None:
        random.Random(shuffle_seed).shuffle(samples)

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", os.environ.get("TGX_DEVICE", "0")))
    allreduce = None
    n_global = len(samples)
    blob, off = N.pack(samples)
    byte_base = 0
    if world > 1:
        import torch
        import torch.distributed as td
        if not td.is_initialized():
            backend = os.environ.get("TGX_DIST_BACKEND", "nccl")
            if backend == "nccl":
                torch.cuda.set_device(device)
            td.init_process_group(backend)
        byte_base = int(off[dist.shard_ranges(off, world)[rank][0]])
        blob, off, _ = dist.take_shard(blob, off, rank, world)  # byte-balanced contiguous sample range
        if dropout > 0.0 and dropout_seed is None:  # one seed for the job: rank 0's
            box = [random.SystemRandom().getrandbits(63)]
            td.broadcast_object_list(box, src=0)
            dropout_seed = box[0]
        allreduce = dist.Collective(device=f"cuda:{device}" if td.get_backend() == "nccl" else None)
    pruner = ModelVocabularyPruner(vocab_size, shrink_factor, em_subiters, dropout, device=device, allreduce=allreduce,
                                   n_samples_global=n_global, dropout_seed=dropout_seed, byte_base=byte_base)
    vocab, report = pruner.prune(Vocab(list(tok._tokens), tok._scores.copy(), tok._keep.copy()), blob, off)
    log.info("Pruned vocabulary from=%d to=%d mem=%.2fMB", initial, len(vocab), sum(len(t) for t in vocab.tokens) / 1e6)
    if rank == 0:
        Tokenizer(vocab.tokens, vocab.scores, vocab.keep, tok._processors, tok.special_tokens()).save(output)
        log.info("Saved pruned vocabulary to %r", output)
    return report


def encode_cmd(input: str, source: str, output: str, separator: Optional[str] = None, dtype: str = "auto",
               dropout: float = 0.0, dropout_seed: Optional[int] = None, device: Optional[int] = None,
               window_bytes: Optional[int] = None) -> dict:
    """Pretokenizes a NUL-separated corpus file into OUTPUT.{ids,idx,json} (tokengeex_b200/corpus.py)."""
    import time

    from . import corpus

    if device is None:
        device = int(os.environ.get("TGX_DEVICE", "0"))
    log.info("Encoding corpus input=%r source=%r output=%r separator=%r dtype=%s dropout=%s", input, source, output,
             separator, dtype, dropout)
    t0 = time.perf_counter()
    meta = corpus.encode_file(input, source, output, separator=separator, dtype=None if dtype == "auto" else dtype,
                              dropout=dropout, dropout_seed=dropout_seed, device=device,
                              window_bytes=window_bytes or corpus.DEFAULT_WINDOW_BYTES)
    dt = time.perf_counter() - t0
    size = meta["source"]["bytes"]
    log.info("Encoded %d samples into %d %s ids from %r (%.2fMB) in %.2fs (%.2f GB/s)", meta["n_samples"],
             meta["n_ids"], meta["dtype"], source, size / 1e6, dt, size / dt / 1e9 if dt > 0 else 0.0)
    return meta


def main(argv: Optional[Sequence[str]] = None) -> int:
    ap = argparse.ArgumentParser(prog="tokengeex_b200", description=__doc__.split("\n\n")[0])
    sub = ap.add_subparsers(dest="cmd", required=True)
    pr = sub.add_parser("prune", help="prune a vocabulary with EM on the GPU (src/cli.rs:65-86)")
    pr.add_argument("-i", "--input", required=True, help="input tokenizer JSON")
    pr.add_argument("-o", "--output", required=True, help="output tokenizer JSON")
    pr.add_argument("-v", "--vocab-size", type=int, required=True)
    pr.add_argument("--train", action="append", default=[], metavar="NAME:PATH[:PROPORTION]")
    pr.add_argument("--dropout", type=float, default=0.01, help="E-step dropout in [0, 1) (src/cli.rs:687)")
    pr.add_argument("--dropout-seed", type=int, default=None, help="seed of the keyed dropout draw (default: fresh)")
    pr.add_argument("--shrink-factor", type=float, default=0.8)
    pr.add_argument("--em-subiters", type=int, default=1)
    pr.add_argument("--device", type=int, default=None)
    pr.add_argument("--shuffle-seed", type=int, default=None)
    en = sub.add_parser("encode", help="tokenize a NUL-separated corpus file into token ids on the GPU")
    en.add_argument("-i", dest="tokenizer", required=True, help="tokenizer JSON")
    en.add_argument("--input", dest="source", required=True, help="corpus file: samples separated by NUL bytes")
    en.add_argument("-o", "--output", required=True, help="output prefix: PREFIX.ids, PREFIX.idx, PREFIX.json")
    en.add_argument("--separator", default=None, metavar="TOKEN", help="token appended after every sample")
    en.add_argument("--dtype", choices=("auto", "uint16", "uint32"), default="auto")
    en.add_argument("--dropout", type=float, default=0.0, help="dropout in [0, 1) (default 0.0: plain encoding)")
    en.add_argument("--dropout-seed", type=int, default=None, help="seed of the keyed dropout draw (default: fresh)")
    en.add_argument("--device", type=int, default=None)
    en.add_argument("--window-bytes", type=int, default=None, help="bytes read per window (default 2 GiB)")
    args = ap.parse_args(argv)
    logging.basicConfig(level=logging.INFO, format="%(asctime)s %(levelname)s %(message)s")
    if args.cmd == "encode":
        encode_cmd(args.tokenizer, args.source, args.output, args.separator, args.dtype, args.dropout, args.dropout_seed,
                   args.device, args.window_bytes)
        return 0
    if not args.train:
        ap.error("at least one --train source is required")
    prune_cmd(args.input, args.output, args.vocab_size, args.train, args.dropout, args.shrink_factor, args.em_subiters,
              args.device, args.shuffle_seed, args.dropout_seed)
    return 0


if __name__ == "__main__":
    sys.exit(main())
