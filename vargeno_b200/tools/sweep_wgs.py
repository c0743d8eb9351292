"""Tuning helper at GRCh38 size: build the S2 index once, then time the resident-input leg on S2 and S3 reads for several
settings of the VGB_* kernel knobs (re-read by the library at vgb_reset_counts when VGB_RETUNE is set), and the S4 probe sets.

    python -m vargeno_b200.tools.sweep_wgs "" VGB_SHORTSCAN=1 VGB_NO_WIDE=1 ...   [--scale S] [--steps K]
(VGB200_LIB=<other build of libvgb200.so> selects a compile-time variant, one process per variant.)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("variants", nargs="*", default=[""])
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--batch-reads", type=int, default=2_000_000)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--probe", action="store_true")
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    os.environ["VGB_RETUNE"] = "1"
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    import bench
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import device_workloads as dw

    B = args.batch_reads
    bb = B * bench.rec_bytes()
    nb = args.steps + args.warmup
    g = Genotyper(device=0, max_chunk_bytes=bb + 4096)
    t0 = time.time()
    wl = bench.build_workload(g, "s2", args.scale)
    print("workload built in %.1f s" % (time.time() - t0), flush=True)
    sets = {}
    for name in ("s2", "s3"):
        d = g.dalloc(nb * bb)
        sub, lowq = bench.READ_SETS[name]
        dw.synth_batch(g, wl, d, nb * B, 0, sub, lowq, bench.LOWQ_CHARS, bench.REC_ID_WIDTH)
        sets[name] = d
    for var in args.variants:
        env = dict(kv.split("=", 1) for kv in var.split(",") if kv)
        for k, v in env.items():
            os.environ[k] = v
        out = {"variant": var, "tag": args.tag}
        for name, d in sets.items():
            g.reset()
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
            out[name] = {"reads_per_s": args.steps * B / dt, "k_geno_ms": (s1["gpu_ms_geno"] - s0["gpu_ms_geno"]) / args.steps,
                         "framing_ms": (s1["gpu_ms_parse"] - s0["gpu_ms_parse"]) / args.steps, "placed": s1["placed"] - s0["placed"]}
        print(json.dumps(out), flush=True)
        for k in env:
            os.environ.pop(k, None)
    if args.probe:
        rs = g.random_sector_bench(32 << 30, 1 << 30, 3)
        for mode, name in ((0, "misses"), (1, "hits"), (2, "half")):
            ms, found = g.probe_bench(1 << 28, mode, 11, 10)
            print(json.dumps({"probe": name, "ms": ms, "g_lookups_per_s": 2 * (1 << 28) / ms / 1e6, "found": found,
                              "frac_of_random_sector_rate": 2 * (1 << 28) / (ms * 1e-3) * 32 / 1e9 / rs, "random_sector_gbs": rs}), flush=True)
    g.close()


if __name__ == "__main__":
    main()
