#!/usr/bin/env python
"""bench.py — headline benchmark of the tokengeex_b200 hot path.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs bench_outputs         # also write the last timed step's ids there (*.npy)

A "step" is one encode_batch pass over one batch of synthetic input (BASELINE.json
configs[1]: 1 GB synthetic multi-language code corpus, 131k Unigram vocab, crlf processor,
token ids bit-exact).  With N > 1 (torchrun, one rank per GPU) every rank encodes its own
1 GB shard of the code+Chinese mix (configs[2]); samples are independent, so there is no
data-path collective and scaling is weak.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark leaves nothing in it

VOCAB_SIZE = 131072
MAX_TOKEN_LEN = 16
VOCAB_SAMPLE_BYTES = 96_000_000
FORWARD_KERNEL_NAME = "viterbi_pair_kernel<2, 1, 960>"  # forward pass 2 (batches below 600 MiB)
TEAM_KERNEL_NAME = "viterbi_team_kernel<16>"  # forward pass 3: the consumer of the match stream
SIDE_KERNEL_NAME = "viterbi_pair_kernel<2, 2, 800> (samples >= 64 KiB, side stream, beside the teams)"
METRIC = "encode_input_throughput"
UNIT = "MB/s"


_JSON_OUT = None  # see main(): the original stdout when NCCL may write to descriptor 1


def emit_json(line: dict) -> None:
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def env_int(k, d):
    return int(os.environ.get(k, d))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def build_vocab(synth, n_gpus=1):
    """Identical on every rank: built from a fixed common sample of the workload's corpus kind (multi-language code
    at N = 1, configs[1]; code+Chinese mix at N > 1, configs[2])."""
    if n_gpus == 1:
        blob, off = synth.corpus(synth.KIND_MULTILANG, 2, VOCAB_SAMPLE_BYTES)
        toks, sc, kp = synth.vocab(blob, off, 2, VOCAB_SIZE, MAX_TOKEN_LEN, 0.05)
    else:
        blob, off = synth.corpus(synth.KIND_CODE_CJK, 3, VOCAB_SAMPLE_BYTES)
        toks, sc, kp = synth.vocab(blob, off, 3, VOCAB_SIZE, MAX_TOKEN_LEN, 0.05)
    return toks, sc, kp


def workload(synth, n_gpus, rank, nbytes, out=None):
    if n_gpus == 1:
        kind, seed, name = synth.KIND_MULTILANG, 2, "encode_batch 1GB multi-language code, 131k vocab (configs[1])"
    else:
        kind, seed, name = synth.KIND_CODE_CJK, 3 + 1000 * rank, "encode 1GB/GPU shard of code+Chinese mix, 131k vocab (configs[2])"
    blob, off = synth.corpus(kind, seed, nbytes, out=out)
    return blob, off, name


DUMP_BYTES = 60_000_000  # data --dump-outputs writes at most (the id offsets take at most half of it)


def dump_outputs(path, torch, d_ids, d_id_off, S):
    """What the last timed step handed its caller (ids u32[T], id_off u64[S+1]), as .npy files in `path`:
      id_off.npy  float64[S+1]  every sample's first token; the last entry is T
      rows.npy    float64[k]    a sample of the samples, drawn in an order fixed by seed 0 for as long as the three
                                files stay within DUMP_BYTES, ascending
      ids.npy     float32[.]    the ids of those samples, concatenated in that order (ids < 2^24: exact)"""
    id_off = d_id_off.cpu().numpy()
    order = np.random.default_rng(0).permutation(S)
    cost = np.cumsum(4 * (id_off[order + 1] - id_off[order]) + 8)
    rows = np.sort(order[:int(np.searchsorted(cost, DUMP_BYTES - 8 * id_off.size, side="right"))])
    n = id_off[rows + 1] - id_off[rows]
    idx = np.arange(int(n.sum()), dtype=np.int64) + np.repeat(id_off[rows] - (np.cumsum(n) - n), n)
    ids = d_ids[torch.from_numpy(idx).to(d_ids.device)].cpu().numpy().view(np.uint32)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "id_off.npy"), id_off.astype(np.float64))
    np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(path, "ids.npy"), ids.astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """The timed region starts here: stop() reports the samples taken from now on (nvidia-smi needs a few hundred
        milliseconds to deliver its first line, so it is started during the warm-up)."""
        self.n0 = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[getattr(self, "n0", 0):]
        during = bool(rows)
        if not rows:  # a timed region shorter than the sampling period: the warm-up steps ran the same kernels
            rows = self.rows[-3:]
        self.samples_from = "timed region" if during else "warm-up steps of the same workload (timed region shorter than the sampling period)"
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_from": self.samples_from}


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path, restated (oracle port; the Rust
    crate cannot be built in this image), all host threads, bounded sample per step."""
    if rank != 0:
        return
    from oracle import oracle as O
    from tokengeex_b200 import synth
    threads = synth.n_threads()
    toks, sc, kp = build_vocab(synth, args.gpus)
    om = O.OracleModel(toks, sc)
    blob, off, name = workload(synth, args.gpus, 0, min(args.bytes, 256_000_000))
    # calibrate: ~8 MB, then size one step to ~8 s
    k = int(np.searchsorted(off, 8_000_000))
    t = time.perf_counter()
    om.encode_batch(blob, off[:k + 1], crlf=True, threads=threads)
    rate = int(off[k]) / (time.perf_counter() - t)
    step_bytes = int(min(int(off[-1]), max(8_000_000, rate * 8.0)))
    k = int(np.searchsorted(off, step_bytes))
    o = off[:k + 1]
    nb = int(o[-1])
    for _ in range(args.warmup):
        om.encode_batch(blob, o, crlf=True, threads=threads)
    times, tokens = [], 0
    for _ in range(args.steps):
        t = time.perf_counter()
        r = om.encode_batch(blob, o, crlf=True, threads=threads)
        times.append(time.perf_counter() - t)
        tokens = int(r[1][-1])
    dt = sum(times)
    mbps = nb * args.steps / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": mbps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 scores / u32 ids",
            "data": "synthetic", "tokens_per_s": tokens * args.steps / dt,
            "config": {"workload": name, "vocab": len(toks), "max_token_len": MAX_TOKEN_LEN, "processor": "crlf",
                       "sample_bytes_per_step": nb},
            "cpu_baseline": {"value": mbps, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"first {nb} bytes ({k} samples) of the workload per step, oracle "
                                       "encode_batch (C++ restatement of the Rust rayon path)"},
            "e2e": {"value": mbps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


PRUNE_VOCAB = 500_000
PRUNE_VOCAB_SAMPLE_BYTES = 200_000_000


def run_prune_iter(args, rank, world, local, torch, dist, N, synth):
    """One EM iteration of `tokengeex prune` (BASELINE.json configs[3]): E-step (forward-backward expected counts,
    src/prune.rs:64-120) -> M-step -> model rebuild -> frequency pass -> prune_vocab selection (src/prune.rs:23-57),
    over a code+Chinese corpus of args.prune_bytes in total, sharded by sample across the ranks, 500k initial
    vocabulary, one all-reduce of the count vector per pass.  Seconds are wall clock around synchronised regions,
    max over ranks."""
    from tokengeex_b200 import prune as P
    dev = torch.device("cuda", local)
    # the vocabulary is built once (rank 0) and broadcast: identical on every rank
    if rank == 0:
        vb, vo = synth.corpus(synth.KIND_CODE_CJK, 4, PRUNE_VOCAB_SAMPLE_BYTES)
        toks, sc, kp = synth.vocab(vb, vo, 4, PRUNE_VOCAB, MAX_TOKEN_LEN, 0.05)
        del vb, vo
        tb, to = N.pack(toks)
        hdr = torch.tensor([len(toks), len(tb)], dtype=torch.int64, device=dev)
    else:
        hdr = torch.zeros(2, dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(hdr, 0)
    V, nb = int(hdr[0]), int(hdr[1])
    if rank == 0:
        t_tb, t_to = torch.from_numpy(tb[:nb].copy()).to(dev), torch.from_numpy(to.view(np.int64).copy()).to(dev)
        t_sc, t_kp = torch.from_numpy(np.ascontiguousarray(sc)).to(dev), torch.from_numpy(np.ascontiguousarray(kp)).to(dev)
    else:
        t_tb = torch.empty(nb, dtype=torch.uint8, device=dev)
        t_to = torch.empty(V + 1, dtype=torch.int64, device=dev)
        t_sc = torch.empty(V, dtype=torch.float64, device=dev)
        t_kp = torch.empty(V, dtype=torch.uint8, device=dev)
    if world > 1:
        for t in (t_tb, t_to, t_sc, t_kp):
            dist.broadcast(t, 0)
        tb, to = t_tb.cpu().numpy(), t_to.cpu().numpy().view(np.uint64)
        toks = [tb[int(to[i]):int(to[i + 1])].tobytes() for i in range(V)]
        sc, kp = t_sc.cpu().numpy(), t_kp.cpu().numpy()
    del t_tb, t_to, t_sc, t_kp
    vocab = P.Vocab(list(toks), np.asarray(sc, np.float64), np.asarray(kp, np.uint8))

    # ONE corpus (seed 4) for every N: rank r generates and keeps its byte-balanced shard of it (dist.shard_ranges), so
    # the all-reduced counts, the frequencies and the pruned vocabulary of an N-GPU run are the 1-GPU run's
    blob, off, first_sample, n_samples = synth.corpus_shard(synth.KIND_CODE_CJK, 4, args.prune_bytes, rank, world)
    S, NB = len(off) - 1, int(off[-1])
    coll = None
    if world > 1:
        from tokengeex_b200.dist import Collective
        coll = Collective(device=f"cuda:{local}")
    pr = P.ModelVocabularyPruner(65536, 0.8, 2, 0.0, device=local, allreduce=coll, n_samples_global=n_samples)
    d = pr._upload(blob, off)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(fn):
        sync()
        t = time.perf_counter()
        r = fn()
        sync()
        dt = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return r, float(dt[0])

    model, t_build0 = timed(lambda: N.Model(vocab.tokens, vocab.scores, device=local))
    pr.run_e_step(model, blob, off, d)  # warm-up: workspaces are allocated on the first call
    # same for the frequency pass (back lengths, marks: ~8 GB of cudaMalloc the EM loop pays once, not per iteration)
    d_wfr = torch.zeros(max(model.V, 1), dtype=torch.int64, device=dev)
    model.token_frequencies_dev(d["text"].data_ptr(), d["off"].data_ptr(), d["S"], d["N"], False, d_wfr.data_ptr())
    del d_wfr
    expected, t_e = timed(lambda: pr.run_e_step(model, blob, off, d))
    e_dev_ms, fwd_ms, bwd_ms, e_match_ms = model.stat(4), model.stat(2), model.stat(3), model.stat(7)
    t_allreduce_e = pr.last_allreduce_s
    expected2 = pr.run_e_step(model, blob, off, d)  # a second run: the counts are bit-identical (integer accumulation)
    counts_reproducible = bool(np.array_equal(np.asarray(expected).view(np.uint64), np.asarray(expected2).view(np.uint64)))
    del expected2
    # property (i) at the full size (SURVEY Appendix A): every byte of the corpus is covered by exactly one token on
    # every path of its snippet, so sum over ids of expected[id] * len(id) == corpus bytes (all ranks, after the
    # all-reduce) — checked on the counts of the timed E-step itself
    tok_len = np.array([len(t) for t in vocab.tokens], np.float64)
    total_bytes = coll.sum_int(NB) if coll is not None else NB
    covered = float(np.dot(np.asarray(expected, np.float64), tok_len))
    cover_err = abs(covered - total_bytes) / total_bytes
    new_vocab, t_m = timed(lambda: pr.run_m_step(vocab, expected))

    def rebuild():  # *model = Model::from(vocab): new trie, same handle and workspaces
        model.rebuild(new_vocab.tokens, new_vocab.scores, packed=new_vocab.packed())  # (as ModelVocabularyPruner.prune does)
        return model
    model2, t_rebuild = timed(rebuild)
    rep = P.PruneReport()
    pruned, t_prune = timed(lambda: pr.prune_vocab(model2, new_vocab, blob, off, rep, d))
    t_freq, t_sel = rep.freq_s[-1], rep.select_s[-1]
    out = {"workload": f"EM prune iteration, {args.prune_bytes} B code+Chinese corpus sharded x{world}, "
                       f"{len(vocab)} initial vocab, max_token_len {MAX_TOKEN_LEN} (configs[3])",
           "unit": "s", "iter_s": t_e + t_m + t_rebuild + t_prune,
           "e_step_s": t_e, "m_step_s": t_m, "model_rebuild_s": t_rebuild, "freq_pass_s": t_freq,
           "prune_select_s": t_sel, "vocab_after_m_step": len(new_vocab), "vocab_after_prune": len(pruned),
           "e_step_device_ms": e_dev_ms, "fb_forward_ms": fwd_ms, "fb_backward_ms": bwd_ms, "match_ms": e_match_ms,
           "allreduce_e_step_s": t_allreduce_e, "allreduce_freq_s": rep.allreduce_s[-1] if rep.allreduce_s else 0.0,
           "corpus": "ONE corpus (kind code+Chinese, seed 4) whatever the number of ranks; rank r holds shard r of it",
           "n_samples_total": int(n_samples), "first_sample_of_rank0": int(first_sample),
           "counts_bit_identical_between_two_runs": counts_reproducible,
           # identical for every N (the driver's N = 1, 2, 4, 8 lines can be compared field by field)
           "expected_counts_sha256": hashlib.sha256(np.ascontiguousarray(expected, np.float64).tobytes()).hexdigest()[:16],
           "frequencies_sha256": hashlib.sha256(np.ascontiguousarray(pr.last_freq).tobytes()).hexdigest()[:16],
           "pruned_vocab_sha256": hashlib.sha256(b"\0".join(pruned.tokens)).hexdigest()[:16],
           "audit": [float(x) for x in rep.audits[-1]] if rep.audits else None,
           "e_step_input_MBps": args.prune_bytes / t_e / 1e6,
           "property_sum_expected_len_eq_bytes_rel_err": cover_err, "property_holds_1e-9": bool(cover_err < 1e-9),
           "bytes_per_gpu": NB, "samples_per_gpu": S,
           "roofline": None, "cpu_baseline": None}
    peak, peak_src = measured_peak()
    alg = NB + 8 * (S + 1) + 8 * len(vocab)
    out["roofline"] = {"bound": "hbm", "achieved": alg / (e_dev_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": alg / (e_dev_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes": alg,
                       "kernel": "fb_split_lane_kernel<false> + fb_contrib_kernel<false> (snippets below the warp threshold) + "
                                 "fb_forward_kernel<32> / fb_backward_kernel<32, true> (whole E-step, device ms)"}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        threads = synth.n_threads()
        om = O.OracleModel(vocab.tokens, vocab.scores)
        k = int(np.searchsorted(off, 2_000_000))
        t = time.perf_counter()
        om.run_e_step(blob, off[:k + 1], threads=threads)
        rate = int(off[k]) / (time.perf_counter() - t)
        k = int(np.searchsorted(off, min(NB, max(2_000_000, rate * 10.0))))
        o = off[:k + 1]
        t = time.perf_counter()
        want = om.run_e_step(blob, o, threads=threads)[0]
        dt = time.perf_counter() - t
        chk = N.Model(vocab.tokens, vocab.scores, device=local)
        got = chk.expected_counts(blob[:max(int(o[-1]), 1)], o)[0]
        chk.close()
        nz = want > 0
        rel = float(np.max(np.abs(got[nz] - want[nz]) / want[nz])) if nz.any() else 0.0
        out["cpu_baseline"] = {"max_rel_diff_vs_gpu": rel, "within_1e-9": bool(rel < 1e-9),"e_step_input_MBps": int(o[-1]) / dt / 1e6, "unit": "MB/s", "cores": threads, "kind": "port",
                               "sample": f"first {int(o[-1])} bytes ({k} samples) of the same corpus, oracle run_e_step "
                                         "(C++ restatement of src/prune.rs:64-120, rayon-like chunking)",
                               "e_step_s_extrapolated": args.prune_bytes / (int(o[-1]) / dt)}
    model2.close()
    return out


def run_prune_schedule(args, rank, world, local, torch, dist, N, synth):
    """BASELINE.json configs[4]: the full prune schedule (src/prune.rs:23-57, docs/RECIPES.md:44-52) — 500k -> 65k
    tokens, shrink 0.8, two EM sub-iterations per step, dropout 0.0 — over ONE corpus of args.schedule_bytes sharded over
    the ranks, run TWICE: wall seconds, sizes after every step, the margin audit, and whether both runs end in the same
    vocabulary (they must: the counts are integer sums)."""
    from tokengeex_b200 import prune as P
    dev = torch.device("cuda", local)
    vb, vo = synth.corpus(synth.KIND_CODE_CJK, 4, PRUNE_VOCAB_SAMPLE_BYTES)  # (deterministic: identical on every rank)
    toks, sc, kp = synth.vocab(vb, vo, 4, PRUNE_VOCAB, MAX_TOKEN_LEN, 0.05)
    del vb, vo
    vocab = P.Vocab(list(toks), np.asarray(sc, np.float64), np.asarray(kp, np.uint8))
    blob, off, first_sample, n_samples = synth.corpus_shard(synth.KIND_CODE_CJK, 4, args.schedule_bytes, rank, world)
    coll = None
    if world > 1:
        from tokengeex_b200.dist import Collective
        coll = Collective(device=f"cuda:{local}")
    runs = []
    for rep_i in range(args.schedule_runs):
        pr = P.ModelVocabularyPruner(65536, 0.8, 2, 0.0, device=local, allreduce=coll, n_samples_global=n_samples)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        final, rep = pr.prune(vocab, blob, off)
        torch.cuda.synchronize()
        wt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(wt, op=dist.ReduceOp.MAX)
        runs.append({"wall_s": float(wt[0]), "final_vocab": len(final),
                     "final_vocab_sha256": hashlib.sha256(b"\0".join(final.tokens)).hexdigest()[:16],
                     "vocab_sizes": rep.vocab_sizes, "e_step_s": round(sum(rep.e_step_s), 3),
                     "m_step_s": round(sum(rep.m_step_s), 3), "freq_pass_s": round(sum(rep.freq_s), 3),
                     "prune_select_s": round(sum(rep.select_s), 3), "rebuild_s": round(sum(rep.rebuild_s), 3),
                     "allreduce_s": round(sum(rep.allreduce_s), 3), "e_steps": len(rep.e_step_s),
                     "m_step_margins": rep.m_margins,
                     "cut_audit": [{"exact_loss_tie_at_cut": bool(a[5]), "loss_gap_at_cut": float(a[6]),
                                    "silently_dropped": int(a[2]), "candidates": int(a[4])} for a in rep.audits]})
    return {"workload": f"full prune schedule {len(vocab)} -> 65536 tokens, shrink 0.8, 2 EM sub-iterations, dropout 0.0, "
                        f"{args.schedule_bytes} B code+Chinese corpus (seed 4) sharded x{world} (configs[4])",
            "runs": runs, "runs_end_in_the_same_vocabulary": len({r["final_vocab_sha256"] for r in runs}) == 1,
            "n_samples_total": int(n_samples)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--bytes", type=int, default=1_000_000_000, help="input bytes per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-prune", action="store_true", help="skip the EM prune-iteration measurement")
    ap.add_argument("--prune-bytes", type=int, default=4_000_000_000, help="total corpus bytes of the prune iteration")
    ap.add_argument("--schedule-bytes", type=int, default=0,
                    help="also run the full prune schedule (configs[4]) over a corpus of this many bytes in total")
    ap.add_argument("--schedule-runs", type=int, default=2)
    ap.add_argument("--only-schedule", action="store_true", help="skip the encode benchmark and the prune iteration")
    ap.add_argument("--chunk-bytes", type=int, default=0, help="bytes per chunk of the pipelined host entry point")
    ap.add_argument("--g-short", type=int, default=0)
    ap.add_argument("--long-threshold", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ids and id offsets of the last timed encode step (rank 0's) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.only_schedule):
        ap.error("--dump-outputs writes the native encode step's outputs: not with --impl reference / --only-schedule")

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from tokengeex_b200 import _native as N
    from tokengeex_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the native arm)")
    torch.cuda.set_device(local)
    numa_node = None
    if world > 1 and not os.environ.get("TGX_NO_NUMA_BIND"):
        from tokengeex_b200.dist import bind_to_gpu_numa_node
        numa_node = bind_to_gpu_numa_node(local)  # host buffers next to this rank's GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it.  NCCL writes its log to file descriptor 1, which has to carry exactly
        # one JSON line: from here on descriptor 1 IS stderr (so the communicator lines stay visible to whoever captures
        # the run) and the JSON line goes out through a private copy of the original stdout.
        global _JSON_OUT
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()

    if args.only_schedule:
        sched = run_prune_schedule(args, rank, world, local, torch, dist, N, synth)
        if rank == 0:
            emit_json({"metric": "prune_schedule_wall_s", "unit": "s", "n_gpus": world, "higher_is_better": False,
                       "value": min(r["wall_s"] for r in sched["runs"]), "prune_schedule": sched})
        if world > 1:
            dist.destroy_process_group()
        return

    toks, sc, kp = build_vocab(synth, world)
    model = N.Model(toks, sc, device=local)
    if args.g_short:
        model.set_option(0, args.g_short)
    if args.long_threshold:
        model.set_option(1, args.long_threshold)
    if args.chunk_bytes:
        model.set_option(7, args.chunk_bytes)
    info = model.info()

    # pinned host input (also the source of the e2e H2D copies)
    h_text = N.pinned_empty(args.bytes)
    blob, off, wname = workload(synth, world, rank, args.bytes, out=h_text)
    S, NB = len(off) - 1, int(off[-1])
    if args.dump_outputs and 16 * (S + 1) > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: the id offsets of {S} samples take more than half of {DUMP_BYTES} bytes")

    d_text = torch.from_numpy(blob).cuda()
    d_off = torch.from_numpy(off.view(np.int64)).cuda()
    d_ids = torch.empty(NB + 4, dtype=torch.int32, device="cuda")
    d_id_off = torch.empty(S + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()

    def step_dev():
        tot, rc, bad = model.encode_batch_dev(d_text.data_ptr(), d_off.data_ptr(), S, NB, True, d_ids.data_ptr(),
                                              NB + 4, d_id_off.data_ptr())
        assert rc == 0, "NoPath in benchmark corpus"
        return tot

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()  # (nvidia-smi delivers its first line after a few hundred milliseconds: started with the warm-up)
    for _ in range(max(args.warmup, 3)):
        tokens = step_dev()
    if rank == 0:  # a few more untimed steps until the sampler is alive (the timed region may be shorter than its period)
        t_w = time.perf_counter()
        while clocks.proc and not clocks.rows and time.perf_counter() - t_w < 2.0:
            tokens = step_dev()
    launches = int(model.stat(0))
    torch.cuda.synchronize()
    barrier()
    clocks.mark()
    dev_ms, vit_ms, back_ms, emit_ms, match_ms, allfwd_ms, side_ms = [], [], [], [], [], [], []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tokens = step_dev()
        dev_ms.append(model.stat(4))
        vit_ms.append(model.stat(1))
        back_ms.append(model.stat(5))
        emit_ms.append(model.stat(6))
        match_ms.append(model.stat(7))
        allfwd_ms.append(model.stat(8))
        side_ms.append(model.stat(9))
    fwd_algo = int(model.stat(10))
    torch.cuda.synchronize()
    barrier()
    wall = time.perf_counter() - t0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, d_ids, d_id_off, S)

    # max over ranks of the device time of the K steps
    tsum = torch.tensor([sum(dev_ms), wall, float(NB), float(tokens), sum(vit_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = tsum.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ttot = tsum.clone()
        dist.all_reduce(ttot, op=dist.ReduceOp.SUM)
        dev_total_ms, wall_max = float(tmax[0]), float(tmax[1])
        bytes_all, tokens_all = float(ttot[2]), float(ttot[3])
    else:
        dev_total_ms, wall_max, bytes_all, tokens_all = sum(dev_ms), wall, float(NB), float(tokens)
    ms_per_step = dev_total_ms / args.steps
    value = bytes_all / (ms_per_step * 1e-3) / 1e6

    # roofline of the dominant kernel (the Viterbi kernel launches), this rank
    peak, peak_src = measured_peak()
    alg_bytes = NB + 4 * tokens + 16 * (S + 1)
    # The forward pass by the algorithm the library picked for this batch (tgx_model_last_stat 10): the pair-CTA kernel
    # alone (2), or match_kernel, then the lane teams over the match stream with the pair-CTA kernel of the longest
    # samples beside them on a stream of its own (3; 0 = the row consumer).  The roofline is quoted for the longest one.
    if fwd_algo == 3:
        fwd_kernels = {"match2_kernel": float(np.mean(match_ms)), TEAM_KERNEL_NAME: float(np.mean(vit_ms)),
                       SIDE_KERNEL_NAME: float(np.mean(side_ms))}
        forward_ms = float(np.mean(allfwd_ms))
    elif fwd_algo == 0:
        fwd_kernels = {"viterbi_rows_kernel": float(np.mean(vit_ms)), "match2_kernel": float(np.mean(match_ms))}
        forward_ms = sum(fwd_kernels.values())
    else:
        fwd_kernels = {FORWARD_KERNEL_NAME: float(np.mean(vit_ms))}
        forward_ms = float(np.mean(vit_ms))
    # (the pair-CTA kernel of the longest samples runs BESIDE the teams on a few SMs and sees 8 % of the bytes: it is
    # listed, but the roofline of the whole batch's bytes is quoted for the longer of the two kernels that see them all)
    dom_kernel = max((k for k in fwd_kernels if k != SIDE_KERNEL_NAME), key=fwd_kernels.get)
    vit = fwd_kernels[dom_kernel] * 1e-3
    achieved = alg_bytes / vit / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            ent = tj.get("kernels", {}).get(dom_kernel)
            if ent:  # DRAM bytes of that kernel per input byte (ncu --set full capture named in the file) x this launch
                traffic = float(ent["dram_bytes_per_input_byte"]) * NB
                traffic_src = ent.get("source")
        except Exception:
            traffic = None

    # e2e: the C-ABI host call, pinned host buffers, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        h_ids = N.pinned_empty(4 * (int(tokens) + 16)).view(np.uint32)  # token count known from the device pass
        for _ in range(2):
            r = model.encode_batch(blob, off, crlf=True, ids_out=h_ids)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = model.encode_batch(blob, off, crlf=True, ids_out=h_ids)
        torch.cuda.synchronize()
        barrier()
        e_wall = time.perf_counter() - t0
        ew = torch.tensor([e_wall], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ew, op=dist.ReduceOp.MAX)
        e2e = {"value": bytes_all * args.steps / float(ew[0]) / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": NB + 8 * (S + 1),
               "d2h_bytes_per_step": int(4 * r[0].size + 8 * (S + 1) + 12 * S),
               "ms_per_step": 1e3 * float(ew[0]) / args.steps,
               "buffers": "pinned host memory (tgx_host_alloc) for text in and ids out"}
        # What the host side alone allows: the step's H2D and D2H bytes copied between the same pinned buffers and the
        # device on two streams, no kernel at all — at N ranks every rank does this at once, so the figure is the
        # ceiling the box's host memory / PCIe path sets for `e2e` whatever the kernels do.  (No collective inside:
        # a failure here is recorded, never fatal.)
        co_ms = float("nan")
        try:
            n_ids = int(r[0].size)
            t_in, t_out = torch.from_numpy(blob), torch.from_numpy(h_ids.view(np.int32))[:n_ids]
            d_out = d_ids[:n_ids]
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
            reps = max(2, args.steps // 2)
            for i in range(reps + 1):  # the first pass is a warm-up
                if i == 1:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                with torch.cuda.stream(s_in):
                    d_text.copy_(t_in, non_blocking=True)
                with torch.cuda.stream(s_out):
                    t_out.copy_(d_out, non_blocking=True)
            torch.cuda.synchronize()
            co_ms = 1e3 * (time.perf_counter() - t0) / reps
            e2e["copy_only"] = {"pinned_host_buffers": bool(t_in.is_pinned() and t_out.is_pinned())}
        except Exception as ex:  # noqa: BLE001
            e2e["copy_only"] = {"error": repr(ex)[:200]}
        cw = torch.tensor([co_ms if co_ms == co_ms else -1.0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(cw, op=dist.ReduceOp.MAX)
        if float(cw[0]) > 0 and "error" not in e2e["copy_only"]:
            e2e["copy_only"].update({"ms_per_step": float(cw[0]), "value": bytes_all / (float(cw[0]) * 1e-3) / 1e6,
                                     "unit": UNIT, "what": "H2D of the text + D2H of the ids alone, both directions at "
                                     "once, max over ranks: the ceiling of e2e on this host"})
        # the same call with ordinary (pageable) caller memory, as a Rust Vec or Python bytes would hand it over
        pg_text = np.array(blob, copy=True)
        pg_ids = np.empty(int(tokens) + 16, np.uint32)
        model.encode_batch(pg_text, off, crlf=True, ids_out=pg_ids)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(1, args.steps // 2)):
            r = model.encode_batch(pg_text, off, crlf=True, ids_out=pg_ids)
        torch.cuda.synchronize()
        barrier()
        pw = torch.tensor([(time.perf_counter() - t0) / max(1, args.steps // 2)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(pw, op=dist.ReduceOp.MAX)
        e2e["pageable"] = {"value": bytes_all / float(pw[0]) / 1e6, "unit": UNIT, "ms_per_step": 1e3 * float(pw[0]),
                           "buffers": "pageable numpy arrays for text in and ids out"}
        del pg_text, pg_ids
        # and through the drop-in Python surface: tokengeex.Tokenizer.encode_batch(List[str], dropout) -> List[List[int]]
        # (bindings/python/src/lib.rs:51-59) on a bounded sample; str -> utf-8 and ids -> Python lists included
        if rank == 0:
            import tokengeex  # the drop-in module name (re-exports tokengeex_b200.tokenizer.Tokenizer)
            from tokengeex_b200.tokenizer import _Processor
            tk = tokengeex.Tokenizer(toks, sc, kp, processors=[_Processor("crlf")], device=local)
            if tk is not None:
                k = int(np.searchsorted(off, 64_000_000))
                raw = blob[:int(off[k])].tobytes()
                texts = [raw[int(off[i]):int(off[i + 1])].decode("utf-8") for i in range(k)]
                tk.encode_batch(texts[:64], 0.0)
                t0 = time.perf_counter()
                out = tk.encode_batch(texts, 0.0)
                dt = time.perf_counter() - t0
                e2e["tokenizer_encode_batch"] = {"value": int(off[k]) / dt / 1e6, "unit": UNIT, "ms": 1e3 * dt,
                                                 "sample": f"{k} samples, {int(off[k])} bytes as List[str] -> List[List[int]]",
                                                 "tokens": int(sum(len(x) for x in out))}
                del texts, out, raw

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        threads = synth.n_threads()
        om = O.OracleModel(toks, sc)
        k = int(np.searchsorted(off, 8_000_000))
        t = time.perf_counter()
        om.encode_batch(blob, off[:k + 1], crlf=True, threads=threads)
        rate = int(off[k]) / (time.perf_counter() - t)
        k = int(np.searchsorted(off, min(NB, max(8_000_000, rate * 12.0))))
        o = off[:k + 1]
        t = time.perf_counter()
        r = om.encode_batch(blob, o, crlf=True, threads=threads)
        dt = time.perf_counter() - t
        # parity on the sample, while we are here
        ok = bool(np.array_equal(r[0], d_ids[:int(r[1][-1])].cpu().numpy().view(np.uint32)))
        cpu = {"value": int(o[-1]) / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"first {int(o[-1])} bytes ({k} samples) of the same corpus, oracle encode_batch "
                         "(C++ restatement of the Rust rayon path)", "ids_match_gpu": ok}

    # every rank: the device ids of a seeded sample of ITS shard against the oracle (bit-exact), min over ranks
    sampled = None
    if not args.no_cpu_baseline:
        from oracle import oracle as O
        om_s = O.OracleModel(toks, sc)
        h_idoff = d_id_off.cpu().numpy().view(np.uint64)
        rs = np.random.RandomState(1234 + rank)
        lens_s = np.diff(off.astype(np.int64))
        pick = set(rs.choice(S, size=min(S, 150), replace=False).tolist()) | set(np.argsort(lens_s)[-2:].tolist())
        ok_s = True
        for i in sorted(pick):
            a, b = int(h_idoff[i]), int(h_idoff[i + 1])
            got = d_ids[a:b].cpu().numpy().view(np.uint32).tolist()
            ok_s = ok_s and got == om_s.encode(O.crlf(blob[int(off[i]):int(off[i + 1])].tobytes()), 0.0)
        okt = torch.tensor([1 if ok_s else 0], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        sampled = {"ids_match_oracle": bool(int(okt[0])), "samples_per_rank": len(pick),
                   "what": "seeded sample of every rank's shard + its two longest samples, oracle encode (bit-exact)"}
        del om_s

    prune_iter = None
    if not args.no_prune:
        del d_text, d_ids, d_id_off, d_off, blob, h_text
        if not args.no_e2e:
            del h_ids
        model.close()
        torch.cuda.empty_cache()
        prune_iter = run_prune_iter(args, rank, world, local, torch, dist, N, synth)

    prune_schedule = None
    if args.schedule_bytes:
        torch.cuda.empty_cache()
        prune_schedule = run_prune_schedule(args, rank, world, local, torch, dist, N, synth)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64 scores / u32 ids", "data": "synthetic",
                "tokens_per_s": tokens_all / (ms_per_step * 1e-3),
                "wall_ms_per_step": 1e3 * wall_max / args.steps,
                "config": {"workload": wname, "vocab": len(toks), "max_token_len": MAX_TOKEN_LEN,
                           "processor": "crlf", "bytes_per_gpu": NB, "samples_per_gpu": S,
                           "l2": "inputs (1 GB/GPU) larger than L2; no flush needed",
                           "trie_slots": int(info.trie_slots), "parallelism": f"sample-sharded x{world}, no collective",
                           "host_numa_node_rank0": numa_node, "host_threads_rank0": synth.n_threads()},
                "gpu_launches": launches * args.steps,
                "clocks": clk,
                "e2e": e2e,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                             "peak_source": peak_src,
                             "kernel": dom_kernel + " (the longest kernel of the forward pass; CUDA events on its own stream)",
                             "algorithmic_bytes": alg_bytes, "kernel_ms": vit * 1e3,
                             "forward_algo": fwd_algo,
                             "forward_kernels_ms": fwd_kernels,
                             "forward_pass_ms": forward_ms,
                             "frac_of_whole_forward_pass": alg_bytes / (forward_ms * 1e-3) / 1e9 / peak,
                             "frac_of_whole_step": alg_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                             "step_breakdown_ms": {"forward": forward_ms, "backtrack": float(np.mean(back_ms)),
                                                   "emit": float(np.mean(emit_ms)),
                                                   "crlf_sort_scan_other": ms_per_step - forward_ms -
                                                   float(np.mean(back_ms)) - float(np.mean(emit_ms))}},
                "cpu_baseline": cpu,
                "sampled_parity": sampled,
                "prune_iter": prune_iter, "prune_schedule": prune_schedule}
        emit_json(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
