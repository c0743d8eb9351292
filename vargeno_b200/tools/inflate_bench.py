"""Device-side inflate measured alone: S1-like FASTQ text made on the device and compressed by zlib at two levels, either as BGZF
pushed through vgb_submit_bgzf (k_inflate_bgzf), or (--mode gzip) as one single gzip stream pushed through vgb_submit_gzip in
pieces (the sub-stream pipeline of csrc/vgb_gzip.cu), or (--mode bam) as unaligned BAM of the same reads at zlib level 1 pushed
through vgb_submit_bam (members inflated, records framed and converted on the device, csrc/vgb_bam.cu).  Prints the rate at which text comes out of the inflate + framing kernels
(vgb_stats.gpu_ms_parse: CUDA events around both) and the wall-clock rate of the whole submit loop.  --profile adds one
repetition under torch.profiler and prints the CUDA time of each kernel (the window chain's share of a round is read there).

    python -m vargeno_b200.tools.inflate_bench [--mode bgzf|gzip|bam] [--reads 4000000] [--chunk-mb 256] [--levels 1,6] [--profile]
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np


def _members(args):
    from vargeno_b200.tools import bgzf
    data, level, block = args
    return b"".join(bgzf.member(data[a:a + block], level) for a in range(0, len(data), block))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--chunk-mb", type=int, default=256, help="inflated bytes per vgb_submit_bgzf call")
    ap.add_argument("--levels", default="1,6")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--mode", choices=("bgzf", "gzip", "bam"), default="bgzf")
    ap.add_argument("--piece-mb", type=int, default=64, help="--mode gzip: compressed bytes per vgb_submit_gzip call")
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    import torch

    import bench
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import bgzf
    from vargeno_b200.tools import device_workloads as dw

    rb = bench.rec_bytes()
    own = args.chunk_mb << 20
    with Genotyper(device=0, max_chunk_bytes=own + (1 << 20)) as g:
        wl = dw.build_s1(g, scale=0.25)
        d = g.dalloc(args.reads * rb)
        dw.synth_batch(g, wl, d, args.reads, 0, 0.005, 0.25, bench.LOWQ_CHARS, bench.REC_ID_WIDTH)
        text = g.d2h(d, args.reads * rb).tobytes()
        g.dfree(d)
        if args.mode == "bam":
            _bam_mode(g, text, args)
            return
        if args.mode == "gzip":
            for level in (int(x) for x in args.levels.split(",")):
                _gzip_mode(g, text, level, args)
            return
        for level in (int(x) for x in args.levels.split(",")):
            t0 = time.time()
            span = 65280 * 256
            with mp.Pool(max(1, (os.cpu_count() or 2) - 1)) as pool:
                buf = b"".join(pool.imap(_members, [(text[a:a + span], level, 65280) for a in range(0, len(text), span)])) + bgzf.EOF_MEMBER
            t_comp = time.time() - t0
            mem, plan = bgzf.plan_chunks(bgzf.scan(buf), own)
            chunks = []
            for k, (o0, i0, i1, ov) in enumerate(plan):
                comp, tab = bgzf.chunk_arrays(buf, mem, o0, i1)
                pin = torch.empty(comp.size, dtype=torch.uint8, pin_memory=True).numpy()
                pin[:] = comp
                chunks.append((pin, tab, ov, k + 1 == len(plan)))
            best = None
            for rep in range(args.repeats + 1):
                g.reset()
                s0 = g.stats()
                t0 = time.perf_counter()
                for pin, tab, ov, last in chunks:
                    g.submit_bgzf(pin, tab, ov, last)
                g.sync()
                dt = time.perf_counter() - t0
                s1 = g.stats()
                ms_parse = s1["gpu_ms_parse"] - s0["gpu_ms_parse"]
                assert s1["reads"] - s0["reads"] == args.reads, (s1["reads"], args.reads)
                if rep and (best is None or ms_parse < best[0]):
                    best = (ms_parse, dt, s1["gpu_ms_geno"] - s0["gpu_ms_geno"])
            print(json.dumps({"zlib_level": level, "text_bytes": len(text), "bgzf_bytes": len(buf), "ratio": len(text) / len(buf), "members": len(mem),
                              "chunks": len(chunks), "compress_s": round(t_comp, 1), "inflate_plus_framing_ms": best[0], "geno_ms": best[2],
                              "inflate_text_gb_per_s": len(text) / (best[0] * 1e-3) / 1e9, "wall_s": best[1],
                              "wall_text_gb_per_s": len(text) / best[1] / 1e9, "wall_reads_per_s": args.reads / best[1]}), flush=True)


def _gzip_mode(g, text, level, args):
    import subprocess

    import torch
    t0 = time.time()
    comp = subprocess.run(["gzip", "-%d" % level, "-c"], input=text, stdout=subprocess.PIPE, check=True).stdout
    t_comp = time.time() - t0
    piece = min(args.piece_mb << 20, g.max_chunk_bytes)
    pin = torch.empty(len(comp), dtype=torch.uint8, pin_memory=True).numpy()
    pin[:] = np.frombuffer(comp, dtype=np.uint8)
    n_reads = text.count(b"\n") // 4
    best = None
    for rep in range(args.repeats + 1):
        g.reset()
        t0 = time.perf_counter()
        calls = g.submit_gzip(pin, piece)
        g.sync()
        dt = time.perf_counter() - t0
        s1 = g.stats()
        assert s1["reads"] == n_reads, (s1["reads"], n_reads)
        if rep and (best is None or s1["gpu_ms_parse"] < best[0]):
            best = (s1["gpu_ms_parse"], dt, s1["gpu_ms_geno"])
    rec = {"mode": "gzip", "gzip_level": level, "text_bytes": len(text), "gzip_bytes": len(comp), "ratio": len(text) / len(comp), "calls": calls,
           "compress_s": round(t_comp, 1), "inflate_plus_framing_ms": best[0], "geno_ms": best[2],
           "inflate_text_gb_per_s": len(text) / (best[0] * 1e-3) / 1e9, "wall_s": best[1], "wall_text_gb_per_s": len(text) / best[1] / 1e9,
           "wall_reads_per_s": n_reads / best[1]}
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        g.reset()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            g.submit_gzip(pin, piece)
            g.sync()
        ker = {}
        for e in prof.events():
            if e.device_type.name == "CUDA":
                ker[e.name] = ker.get(e.name, 0.0) + e.device_time / 1e3
        gz = {k: v for k, v in ker.items() if "k_gz_" in k}
        rec["kernel_ms"] = {k.split("(")[0]: round(v, 3) for k, v in sorted(ker.items(), key=lambda x: -x[1])[:12]}
        rec["window_chain_share_of_gzip_kernels"] = sum(v for k, v in gz.items() if "k_gz_window" in k) / max(1e-9, sum(gz.values()))
    print(json.dumps(rec), flush=True)


def _bam_mode(g, text, args):
    """uBAM of the reads (level 1, bgzip-sized members); wall-clock reads/s of the submit loop (the BAM kernels are not inside
    gpu_ms_parse), and the share of 64 KiB tiles the chain walks again (tools/bam.repair_share, the same check as the device)"""
    import torch

    from vargeno_b200.tools import bam, bgzf
    t0 = time.time()
    raw = bam.ubam_fixed(text)
    span = 65280 * 256
    with mp.Pool(max(1, (os.cpu_count() or 2) - 1)) as pool:
        buf = b"".join(pool.imap(_members, [(raw[a:a + span], 1, 65280) for a in range(0, len(raw), span)])) + bgzf.EOF_MEMBER
    t_comp = time.time() - t0
    calls = []
    for comp, tab in g.bam_calls(buf, args.chunk_mb << 20):
        pin = torch.empty(comp.size, dtype=torch.uint8, pin_memory=True).numpy()
        pin[:] = comp
        calls.append((pin, np.ascontiguousarray(tab, dtype="<u4")))
    n_reads = text.count(b"\n") // 4
    best = None
    for rep in range(args.repeats + 1):
        g.reset()
        t0 = time.perf_counter()
        for k, (pin, tab) in enumerate(calls):
            g.submit_bam_call(pin, tab, k == 0, k + 1 == len(calls))
        g.sync()
        dt = time.perf_counter() - t0
        s1 = g.stats()
        assert s1["reads"] == n_reads, (s1["reads"], n_reads)
        if rep and (best is None or dt < best[0]):
            best = (dt, s1["gpu_ms_parse"], s1["gpu_ms_geno"])
    tiles, repaired = bam.repair_share(raw[:64 << 20])
    print(json.dumps({"mode": "bam", "zlib_level": 1, "text_bytes": len(text), "bam_bytes": len(raw), "bgzf_bytes": len(buf), "calls": len(calls),
                      "compress_s": round(t_comp, 1), "wall_s": best[0], "wall_reads_per_s": n_reads / best[0], "wall_text_gb_per_s": len(text) / best[0] / 1e9,
                      "framing_ms": best[1], "geno_ms": best[2], "tiles_first_64MiB": tiles, "tiles_repaired": repaired,
                      "repair_share": repaired / max(1, tiles)}), flush=True)


if __name__ == "__main__":
    main()
