"""The output VCF at GRCh38 size: the device writer (vgb_vcf_template + vgb_vcf_write) against the host path it replaces
(`vargeno-b200 vcf-rewrite`: calls_to_map + rewrite_vcf) and `gzip -1` of that output, on the same box.

    python -m vargeno_b200.tools.vcf_write_bench [--records 12000000] [--repeats 3] [--dir DIR]

The index is S1 (tools/device_workloads.build_s1: 1 M sites on a chr22-shaped contig, built on the GPU).  The synthetic VCF puts
records-per-site = ceil(records / sites) dbSNP-style lines on every site, so every record is written (a site shared by several
records calls all of them).  Every site is called (a random genotype, a random confidence), GQ comes from the C library's log as on
the command line.  It prints one JSON object: the GPU's name and power limit, the template parse + upload, the per-sample device
write as .vcf and as .vcf.gz (callback that drops the bytes: device work and the copy back), the host rewrite and gzip -1, and the
size of the BGZF output against tools/bgzf.compress(level=1) of the same text.  The device output is checked against the host's,
byte for byte, and the BGZF output must inflate to it."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

T0 = time.time()


def log(msg):
    print("[%7.1f s] %s" % (time.time() - T0, msg), file=sys.stderr, flush=True)


def inflate_members(buf):
    """a BGZF file inflated member by member (gzip.decompress copies the rest of the buffer for every member)"""
    from vargeno_b200.tools import bgzf
    mv = memoryview(buf)
    return b"".join(zlib.decompress(mv[off + poff:off + size - 8], -15) for off, size, poff, _ in bgzf.scan(buf))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    return q.stdout.splitlines()[0].strip() if q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=12_000_000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--dir", default="")
    a = ap.parse_args()
    from vargeno_b200 import _lib
    from vargeno_b200 import build as vb
    from vargeno_b200.geno import Genotyper, site_gq
    from vargeno_b200.tools import bgzf, device_workloads
    vb.build()
    res = {"gpu": gpu_info()}
    tmp = tempfile.TemporaryDirectory(prefix="vgb_vcf_", dir=a.dir or None)
    d = tmp.name
    with Genotyper(device=0) as g:
        device_workloads.build_s1(g)
        log("index built")
        pos = g.sites()["pos"]
        n = pos.size
        per = -(-a.records // n)
        t0 = time.time()
        name = g.chr_names[0]
        lines = []
        for i, p in enumerate(pos.tolist()):
            for k in range(per):
                lines.append("%s\t%d\trs%d\tA\tC\t.\tPASS\tRS=%d;RSPOS=%d;dbSNPBuildID=150;SAO=0;VC=SNV;CAF=0.9%d,0.0%d;COMMON=1\n"
                             % (name, p, 1000 * i + k, 1000 * i + k, p, k % 10, 9 - k % 10))
        vcf = ("##fileformat=VCFv4.0\n##source=vcf_write_bench\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n" + "".join(lines)).encode()
        del lines
        log("VCF made")
        res.update({"records": n * per, "sites": int(n), "vcf_bytes": len(vcf), "make_vcf_s": round(time.time() - t0, 2)})
        rng = np.random.default_rng(5)
        gt = rng.integers(1, 4, n).astype(np.uint8)
        conf = rng.uniform(1e-9, 1.0, n)
        gq = site_gq(gt, conf)
        t0 = time.time()
        g.vcf_template(vcf)
        res["template_s"] = round(time.time() - t0, 3)
        drop = _lib.WRITE_FN(lambda user, p, k: 0)
        for bz in (0, 1):
            ts = []
            for _ in range(a.repeats + 1):
                t0 = time.time()
                g._ck(g.L.vgb_vcf_write(g.h, _lib.ptr(gt), _lib.ptr(gq), n, bz, drop, None, None))
                ts.append(time.time() - t0)
            res["device_write_%s_s" % ("vcf_gz" if bz else "vcf")] = [round(x, 4) for x in ts[1:]]
        log("device writes timed")
        plain = g.vcf_write(gt, gq)
        packed = g.vcf_write(gt, gq, bgzf=True)
    res["vcf_out_bytes"] = len(plain)
    res["vcf_gz_bytes"] = len(packed)
    # the host path on the same calls
    vcf_path, calls, prefix, out = (os.path.join(d, x) for x in ("in.vcf", "calls.tsv", "ix", "host.vcf"))
    open(vcf_path, "wb").write(vcf)
    with open(prefix + ".chrlens", "w") as f:
        f.write("%s %d\n" % (name, int(g.chr_lens[0])))
    with open(calls, "w") as f:
        f.write("".join("%d %d %s\n" % (p, x, c.hex()) for p, x, c in zip(pos.tolist(), gt.tolist(), conf.tolist())))
    log("host inputs written")
    t0 = time.time()
    subprocess.check_call([vb.HOST_BIN, "vcf-rewrite", prefix, calls, vcf_path, out])
    res["host_vcf_rewrite_s"] = round(time.time() - t0, 2)
    t0 = time.time()
    with open(out + ".gz", "wb") as f:
        subprocess.check_call(["gzip", "-1", "-c", out], stdout=f)
    res["host_gzip_1_s"] = round(time.time() - t0, 2)
    log("host path timed")
    host = open(out, "rb").read()
    res["device_equals_host"] = plain == host
    res["bgzf_inflates_to_host"] = inflate_members(packed) == host
    log("outputs compared")
    t0 = time.time()
    ref = len(bgzf.compress(host, level=1))
    res["zlib1_bgzf_bytes"] = ref
    res["zlib1_bgzf_s"] = round(time.time() - t0, 2)
    res["size_vs_zlib1"] = round(len(packed) / ref, 4)
    print(json.dumps(res), flush=True)
    tmp.cleanup()
    if not (res["device_equals_host"] and res["bgzf_inflates_to_host"]):
        raise SystemExit("device output differs from the host's")


if __name__ == "__main__":
    main()
