"""A cohort end to end: `vargeno-b200 geno-samples` over a sample sheet against the same samples as separate `vargeno-b200 geno`
processes run back to back, on 1..N GPUs of this box.  What it shows is the fixed cost per sample that geno-samples removes: the
index load (open, upload, re-layout, pinned buffers) happens once per GPU instead of once per sample.

    python -m vargeno_b200.tools.cohort_e2e [--samples 16] [--reads 8000000] [--gpus 1,8] [--dir /dev/shm/vgb_cohort]

Everything is made on this box: the S1 index (device builder -> the five files), and K samples of synthetic reads from the device
generator, one seed each, written to tmpfs (the page-cache case a warm run sees) as plain text and as BGZF (multi-process zlib
level 1, like `bgzip -@`).  For each GPU count and format it runs (a) geno-samples over the sheet and (b) K geno processes, checks
that (a) and (b) wrote identical VCFs, and prints one JSON object per run with the per-sample load / read-loop / VCF-write times.
The GPU's name and power limit are read in the same run and printed first."""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import time


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    return [l.strip() for l in q.stdout.splitlines() if l.strip()]


def verbose_lines(stderr):
    return [json.loads(l) for l in stderr.splitlines() if l.startswith("{")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--reads", type=int, default=8_000_000, help="reads per sample")
    ap.add_argument("--gpus", default="", help="comma list of GPU counts; default 1 and every GPU of the box")
    ap.add_argument("--dir", default="/dev/shm/vgb_cohort")
    ap.add_argument("--chunk-mb", type=int, default=512)
    ap.add_argument("--formats", default="plain,bgzf")
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    import bench
    from vargeno_b200 import build as vb
    from vargeno_b200.geno import Genotyper
    from vargeno_b200.tools import bgzf, synth
    from vargeno_b200.tools import device_workloads as dw
    from vargeno_b200.tools import index_builder as ib

    gpus = gpu_info()
    if not gpus:
        raise SystemExit("cohort_e2e: no GPU found (nvidia-smi lists none)")
    counts = [int(x) for x in args.gpus.split(",")] if args.gpus else sorted({1, len(gpus)})
    print(json.dumps({"section": "gpus", "nvidia_smi": gpus}), flush=True)

    vb.build()
    os.makedirs(args.dir, exist_ok=True)
    prefix, vcf = os.path.join(args.dir, "s1"), os.path.join(args.dir, "snp.vcf")
    rb = bench.rec_bytes()
    names = ["S%02d" % k for k in range(args.samples)]
    plain = {n: os.path.join(args.dir, n + ".fq") for n in names}
    t0 = time.time()
    with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:
        wl = dw.build_s1(g, keep_host=True)
        ib.write_index(wl.host_index, prefix)
        gobj = synth.Genome(wl.names, [wl.host_genome[s:s + l] for s, l in zip(wl.starts, wl.lens)])
        synth.write_vcf(gobj, wl.host_snps, vcf)
        B = 8_000_000
        d = g.dalloc(B * rb)
        for k, n in enumerate(names):
            with open(plain[n], "wb") as f:
                for first in range(0, args.reads, B):
                    m = min(B, args.reads - first)
                    g.synth_reads_device(wl.hap0_d, wl.hap1_d, wl.genome_len, wl.starts, wl.lens, m, wl.read_len, wl.seed + 1000 + k, first,
                                         bench.REC_ID_WIDTH, 0.005, 0.25, bench.LOWQ_CHARS, d, m * rb)
                    g.d2h(d, m * rb).tofile(f)
        g.dfree(d)
    print(json.dumps({"section": "setup", "samples": args.samples, "reads_per_sample": args.reads, "fastq_bytes_per_sample": os.path.getsize(plain[names[0]]),
                      "seconds": round(time.time() - t0, 1), "dir": args.dir, "cpus": os.cpu_count()}), flush=True)
    inputs = {}
    if "plain" in args.formats:
        inputs["plain"] = plain
    if "bgzf" in args.formats:
        t0 = time.time()
        inputs["bgzf"] = {n: p + ".gz" for n, p in plain.items()}
        for n in names:
            bgzf.compress_file(plain[n], inputs["bgzf"][n], procs=max(1, (os.cpu_count() or 2) - 1))
        print(json.dumps({"section": "bgzf written", "bytes": sum(os.path.getsize(p) for p in inputs["bgzf"].values()),
                          "seconds": round(time.time() - t0, 1)}), flush=True)

    def read_dir(d):
        return {n: open(os.path.join(d, n + ".vcf"), "rb").read() for n in names if os.path.exists(os.path.join(d, n + ".vcf"))}

    for fmt, files in inputs.items():
        sheet = os.path.join(args.dir, "samples_%s.tsv" % fmt)
        with open(sheet, "w") as f:
            f.write("".join("%s\t%s\n" % (n, files[n]) for n in names))
        for n_gpu in counts:
            common = ["--gpus", str(n_gpu), "--chunk-mb", str(args.chunk_mb), "--verbose"]
            # (a) one geno-samples process
            out_a = os.path.join(args.dir, "out_a")
            shutil.rmtree(out_a, ignore_errors=True)
            t = time.time()
            p = subprocess.run([vb.HOST_BIN, "geno-samples", prefix, sheet, vcf, out_a] + common, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            wall = time.time() - t
            info = verbose_lines(p.stderr)
            summary = next((x for x in info if "total_s" in x), {})
            rec = {"section": "run", "mode": "geno-samples", "format": fmt, "gpus": n_gpu, "rc": p.returncode, "wall_s": round(wall, 3),
                   "load_s": summary.get("load_s"), "total_s": summary.get("total_s"), "failed": summary.get("failed"),
                   "per_sample": [{k: x[k] for k in ("name", "gpu", "reads", "reads_s", "write_s", "ok")} for x in info if "name" in x]}
            if p.returncode:
                rec["stderr"] = p.stderr[-800:]
            print(json.dumps(rec), flush=True)
            a = read_dir(out_a)
            # (b) one geno process per sample, back to back
            out_b = os.path.join(args.dir, "out_b")
            shutil.rmtree(out_b, ignore_errors=True)
            os.makedirs(out_b)
            per, rcs, t = [], [], time.time()
            for n in names:
                ts = time.time()
                q = subprocess.run([vb.HOST_BIN, "geno", prefix, files[n], vcf, os.path.join(out_b, n + ".vcf")] + common, stdout=subprocess.PIPE,
                                   stderr=subprocess.PIPE, text=True)
                wall_s = time.time() - ts
                x = (verbose_lines(q.stderr) or [{}])[-1]
                rcs.append(q.returncode)
                # geno reports no write time: what is left of the process's wall time after load and read loop (start-up included)
                left = wall_s - x["load_s"] - x["reads_s"] if "load_s" in x else None
                per.append({"name": n, "rc": q.returncode, "reads": x.get("reads"), "load_s": x.get("load_s"), "reads_s": x.get("reads_s"),
                            "rest_s": round(left, 3) if left is not None else None, "wall_s": round(wall_s, 3)})
            wall = time.time() - t
            print(json.dumps({"section": "run", "mode": "geno x %d" % len(names), "format": fmt, "gpus": n_gpu, "rc": max(rcs, key=abs),
                              "wall_s": round(wall, 3), "load_s_sum": round(sum(x["load_s"] or 0 for x in per), 3), "per_sample": per}), flush=True)
            b = read_dir(out_b)
            print(json.dumps({"section": "check", "format": fmt, "gpus": n_gpu, "vcfs": len(a),
                              "identical": len(a) == len(names) and a == b}), flush=True)
    shutil.rmtree(args.dir, ignore_errors=True)


if __name__ == "__main__":
    main()
