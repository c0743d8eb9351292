"""The drop-in's real end to end: `vargeno-b200 geno` on FASTQ FILES (plain text, BGZF, single-stream gzip), wall clock of the
read loop as the program reports it (index load excluded, reported separately), on 1..N GPUs of this box.

    python -m vargeno_b200.tools.cli_e2e [--reads 64000000] [--gpus 1,8] [--dir /dev/shm/vgb_e2e] [--workload s1]

Everything is made on this box: the S1 index (device builder -> the five files), the reads (device generator -> a file in
tmpfs, i.e. the page-cache case a warm run sees), the BGZF copy (multi-process zlib level 1, like `bgzip -@`), and a
single-stream `gzip -1` copy of the first 2 GB, run inflated on the device (vgb_submit_gzip, first GPU only) and, for comparison,
through host zlib (VGB_HOST_INFLATE=1), and an unaligned BAM copy of the first 2 GB (the same reads, zlib level 1, one file: one
GPU; --skip-bam leaves it out).  Prints one JSON object per run."""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import time

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=64_000_000)
    ap.add_argument("--gpus", default="1")
    ap.add_argument("--dir", default="/dev/shm/vgb_e2e")
    ap.add_argument("--chunk-mb", type=int, default=512)
    ap.add_argument("--skip-gzip", action="store_true")
    ap.add_argument("--skip-bam", action="store_true")
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    import bench
    from vargeno_b200 import build as vb
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import bgzf, synth
    from vargeno_b200.tools import device_workloads as dw
    from vargeno_b200.tools import index_builder as ib

    vb.build()
    os.makedirs(args.dir, exist_ok=True)
    prefix, fq, vcf = (os.path.join(args.dir, x) for x in ("s1", "reads.fq", "snp.vcf"))
    rb = bench.rec_bytes()
    t0 = time.time()
    with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:
        wl = dw.build_s1(g, keep_host=True)
        ib.write_index(wl.host_index, prefix)
        gobj = synth.Genome(wl.names, [wl.host_genome[s:s + l] for s, l in zip(wl.starts, wl.lens)])
        synth.write_vcf(gobj, wl.host_snps, vcf)
        B = 8_000_000
        d = g.dalloc(B * rb)
        with open(fq, "wb") as f:
            for first in range(0, args.reads, B):
                n = min(B, args.reads - first)
                dw.synth_batch(g, wl, d, n, first, 0.005, 0.25, bench.LOWQ_CHARS, bench.REC_ID_WIDTH)
                g.d2h(d, n * rb).tofile(f)
        g.dfree(d)
    size = os.path.getsize(fq)
    print(json.dumps({"section": "setup", "reads": args.reads, "fastq_bytes": size, "seconds": round(time.time() - t0, 1), "dir": args.dir,
                      "cpus": os.cpu_count()}), flush=True)
    t0 = time.time()
    bgz = fq + ".bgzf.gz"
    bgzf.compress_file(fq, bgz, procs=max(1, (os.cpu_count() or 2) - 1))
    print(json.dumps({"section": "bgzf written", "bytes": os.path.getsize(bgz), "ratio": size / os.path.getsize(bgz), "seconds": round(time.time() - t0, 1)}), flush=True)
    gz, n_small = None, 0
    if not args.skip_gzip:
        gz = fq + ".single.gz"
        n_small = min(size, (2_000_000_000 // rb) * rb)
        with open(fq, "rb") as f, open(gz, "wb") as o:
            p = subprocess.Popen(["gzip", "-1", "-c"], stdin=subprocess.PIPE, stdout=o)
            left = n_small
            while left:
                blk = f.read(min(left, 1 << 26))
                p.stdin.write(blk)
                left -= len(blk)
            p.stdin.close()
            p.wait()
    ubam, n_bam = None, 0
    if not args.skip_bam:
        from vargeno_b200.tools import bam
        ubam = fq + ".bam"
        n_bam = min(size, (2_000_000_000 // rb) * rb)
        with open(fq, "rb") as f:
            raw = bam.ubam_fixed(f.read(n_bam))
        with open(ubam + ".raw", "wb") as f:
            f.write(raw)
        del raw
        bgzf.compress_file(ubam + ".raw", ubam, procs=max(1, (os.cpu_count() or 2) - 1))
        os.remove(ubam + ".raw")

    def run(tag, path, gpus, n_reads, extra_env=None):
        out = os.path.join(args.dir, "out.vcf")
        env = dict(os.environ)
        env.update(extra_env or {})
        t = time.time()
        p = subprocess.run([vb.HOST_BIN, "geno", prefix, path, vcf, out, "--gpus", str(gpus), "--chunk-mb", str(args.chunk_mb), "--verbose"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
        wall = time.time() - t
        info = None
        for line in p.stderr.splitlines():
            if line.startswith("{"):
                info = json.loads(line)
        rec = {"section": "run", "input": tag, "gpus": gpus, "rc": p.returncode, "wall_s": round(wall, 2), "file_bytes": os.path.getsize(path)}
        if info:
            rec.update({"reads": info["reads"], "placed": info["placed"], "load_s": info["load_s"], "reads_s": info["reads_s"],
                        "reads_per_s": info["reads_per_s"], "text_gb_per_s": info["reads"] * rb / info["reads_s"] / 1e9, "calls": info["calls"]})
        else:
            rec["stderr"] = p.stderr[-500:]
        print(json.dumps(rec), flush=True)
        return open(out, "rb").read() if p.returncode == 0 else None

    for gpus in [int(x) for x in args.gpus.split(",")]:
        a = run("plain text (tmpfs)", fq, gpus, args.reads)
        b = run("BGZF, inflated on the device", bgz, gpus, args.reads)
        print(json.dumps({"section": "check", "gpus": gpus, "bgzf_vcf_identical_to_plain": a is not None and a == b}), flush=True)
        if gpus == 1:
            run("BGZF, inflated on the host by zlib (sequential reader)", bgz, gpus, args.reads, {"VGB_HOST_INFLATE": "1"}) if size <= 8_000_000_000 else None
            if gz:
                d = run("single-stream gzip, first 2 GB, inflated on the device", gz, gpus, 0)
                h = run("single-stream gzip, first 2 GB, inflated on the host by zlib", gz, gpus, 0, {"VGB_HOST_INFLATE": "1"})
                chk = {"section": "check", "gpus": gpus, "gzip_device_vcf_identical_to_host_zlib": d is not None and d == h}
                if n_small == size:
                    chk["gzip_device_vcf_identical_to_plain"] = d is not None and d == a
                print(json.dumps(chk), flush=True)
            if ubam:
                run("unaligned BAM, first 2 GB of reads, inflated and converted on the device", ubam, gpus, 0)
    shutil.rmtree(args.dir, ignore_errors=True)


if __name__ == "__main__":
    main()
