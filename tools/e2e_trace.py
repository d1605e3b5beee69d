#!/usr/bin/env python
"""Developer probe: wall time of the pipelined host entry point (tgx_encode_batch, pinned host buffers) for several
forward passes and chunk sizes.  TGX_TRACE=1 prints the device timeline."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    import bench
    from tokengeex_b200 import _native as N, synth
    toks, sc, kp = bench.build_vocab(synth)
    m = N.Model(toks, sc, device=0)
    h_text = N.pinned_empty(1_000_000_000)
    blob, off, _ = bench.workload(synth, 1, 0, 1_000_000_000, out=h_text)
    NB = int(off[-1])
    h_ids = N.pinned_empty(4 * (NB // 2 + 16)).view(np.uint32)
    # argv: "algo:chunk_MiB[:key=value,...]" ...   (default: the shipped configuration and its neighbours)
    cfgs = sys.argv[1:] or ["2:352", "3:352", "3:176", "3:128"]
    for cfg in cfgs:
        parts = cfg.split(":")
        algo, ch = int(parts[0]), int(parts[1]) << 20
        m.set_option(3, algo)
        m.set_option(7, ch)
        if len(parts) > 2 and parts[2]:
            for kv in parts[2].split(","):
                k, v = kv.split("=")
                m.set_option(int(k), int(v))
        best = 1e9
        for i in range(4):
            t = time.perf_counter()
            m.encode_batch(blob, off, crlf=True, ids_out=h_ids)
            dt = time.perf_counter() - t
            if i:
                best = min(best, dt)
        print(f"algo {algo} chunk {ch >> 20} MiB {parts[2] if len(parts) > 2 else ''}: best {best * 1e3:.2f} ms  ({NB / best / 1e9:.2f} GB/s)", flush=True)


if __name__ == "__main__":
    main()
