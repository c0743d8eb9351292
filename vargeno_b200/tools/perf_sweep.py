"""Tuning helper: build the S1 workload once, then time the resident-input leg for several library variants
(environment knobs read by libvgb200.so at context creation / index upload).

    python -m vargeno_b200.tools.perf_sweep "" VGB_SHORTSCAN=0 VGB_SHORTSCAN=1 VGB_NO_TAIL_OVERLAP=1 ...   [--scale S] [--batch-reads B] [--steps K]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("variants", nargs="*", default=[""])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--batch-reads", type=int, default=2_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sub-rate", type=float, default=0.005)
    ap.add_argument("--lowq-prob", type=float, default=0.25)
    args = ap.parse_args()
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import workloads
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    from bench import REC_ID_WIDTH, rec_bytes

    t0 = time.time()
    wl = workloads.make_s1(scale=args.scale, sub_rate=args.sub_rate, lowq_prob=args.lowq_prob)
    print("workload built in %.1f s" % (time.time() - t0), flush=True)
    B, L = args.batch_reads, wl.read_len
    nb = args.steps + args.warmup
    bb = B * rec_bytes(L)
    for var in args.variants:
        env = dict(kv.split("=", 1) for kv in var.split(",") if kv)
        for k, v in env.items():
            os.environ[k] = v
        g = Genotyper(device=0, max_chunk_bytes=bb + 4096)
        g.upload_index(wl.index)
        h0, h1 = g.dalloc(wl.haps[0].size), g.dalloc(wl.haps[1].size)
        g.h2d(h0, wl.haps[0])
        g.h2d(h1, wl.haps[1])
        d = g.dalloc(nb * bb)
        g.synth_reads_device(h0, h1, wl.haps[0].size, wl.genome.starts, wl.genome.lengths, nb * B, L, wl.seed + 1000, 0, REC_ID_WIDTH,
                             wl.sub_rate, wl.lowq_prob, wl.lowq_chars, d, nb * bb)
        for i in range(args.warmup):
            g.submit_device(d + i * bb, bb)
        g.sync()
        s0 = g.stats()
        t = time.perf_counter()
        for i in range(args.warmup, nb):
            g.submit_device(d + i * bb, bb)
        g.sync()
        dt = time.perf_counter() - t
        s1 = g.stats()
        look = sum(s1[k] - s0[k] for k in ("exact_lookups", "nbr_query_lookups", "nbr_scan_reads"))
        print(json.dumps({"variant": var, "reads_per_s": args.steps * B / dt, "ms_per_step": dt / args.steps * 1e3,
                          "k_geno_ms": (s1["gpu_ms_geno"] - s0["gpu_ms_geno"]) / args.steps,
                          "framing_ms": (s1["gpu_ms_parse"] - s0["gpu_ms_parse"]) / args.steps,
                          "lookups_per_read": look / (s1["reads"] - s0["reads"]),
                          "placed": (s1["placed"] - s0["placed"]) / (s1["reads"] - s0["reads"])}), flush=True)
        for k in env:
            os.environ.pop(k, None)
        g.dfree(d)
        g.dfree(h0)
        g.dfree(h1)
        g.close()


if __name__ == "__main__":
    main()
