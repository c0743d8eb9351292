"""The output VCF written on the device (vgb_vcf_template / vgb_vcf_write, csrc/vgb_vcf.cu) and the device BGZF writer
(vgb_deflate_bgzf, csrc/vgb_deflate.cuh -- the same source tests/test_deflate_host.py checks on the CPU).  `geno ... out.vcf.gz`
must inflate to the golden VCF, `geno-samples --bgzf` must write for each sample what `geno` writes for it alone, a VCF error that
depends on a sample's calls must fail that sample only, and BGZF text from the device must read back through vgb_submit_bgzf."""
import gzip
import os
import subprocess
import threading
import zlib

import numpy as np
import pytest

from oracle import oracle as orc
from vargeno_b200 import build as vb
from vargeno_b200.tools import bgzf
from vargeno_b200.tools import index_builder as ib

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=60).stdout
    except Exception:
        return 0
    return sum(1 for l in out.splitlines() if l.startswith("GPU "))


def _prefix(cache, name, tmp_path):
    prefix = str(tmp_path / "ix")
    if name == "ucscA":                 # the golden ucscA VCF comes from the index built from the UCSC table
        p = subprocess.run([vb.HOST_BIN, "index", cache.dataset(name).fasta, cache.dataset(name).txt, prefix, "--no-lite"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert p.returncode == 0, p.stderr
    else:
        ib.write_index(cache.index(name), prefix)
    return prefix


def _members_ok(buf):
    mem = bgzf.scan(buf)
    assert buf.endswith(bgzf.EOF_MEMBER)
    assert all(size <= 65536 and isize <= 65280 for _, size, _, isize in mem)


@pytest.mark.parametrize("gpus", [1, 2])
@pytest.mark.parametrize("name", ["s0", "advA", "advB", "ucscA"])
def test_geno_vcf_gz_inflates_to_the_reference_vcf(cache, name, gpus, tmp_path):
    if gpus > _gpu_count():
        pytest.skip("needs %d GPUs" % gpus)
    vb.build()
    ds = cache.dataset(name)
    prefix = _prefix(cache, name, tmp_path)
    out = str(tmp_path / "out.vcf.gz")
    p = subprocess.run([vb.HOST_BIN, "geno", prefix, ds.fastq, ds.vcf, out, "--gpus", str(gpus), "--chunk-mb", "1"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr
    buf = open(out, "rb").read()
    _members_ok(buf)
    assert gzip.decompress(buf) == open(os.path.join(GOLD, name + ".out.vcf"), "rb").read()


def _sheet(tmp_path, rows):
    path = str(tmp_path / "samples.tsv")
    with open(path, "w") as f:
        for n, r in rows:
            f.write("%s\t%s\n" % (n, r))
    return path


def test_geno_samples_bgzf_is_what_geno_writes(cache, tmp_path):
    vb.build()
    ds = cache.dataset("advA")
    prefix = _prefix(cache, "advA", tmp_path)
    text = open(ds.fastq, "rb").read()
    lines = text.split(b"\n")
    half = str(tmp_path / "half.fq")
    open(half, "wb").write(b"\n".join(lines[:len(lines) // 8 * 4]) + b"\n")
    reads = {"whole": ds.fastq, "half": half}
    out_dir = str(tmp_path / "out")
    gpus = min(2, max(1, _gpu_count()))
    p = subprocess.run([vb.HOST_BIN, "geno-samples", prefix, _sheet(tmp_path, reads.items()), ds.vcf, out_dir, "--bgzf", "--gpus", str(gpus)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr
    assert sorted(os.listdir(out_dir)) == ["half.vcf.gz", "whole.vcf.gz"]
    for name, r in reads.items():
        one = str(tmp_path / (name + ".vcf.gz"))
        q = subprocess.run([vb.HOST_BIN, "geno", prefix, r, ds.vcf, one], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert q.returncode == 0, q.stderr
        got = open(os.path.join(out_dir, name + ".vcf.gz"), "rb").read()
        assert got == open(one, "rb").read()
        _members_ok(got)
    assert gzip.decompress(open(os.path.join(out_dir, "whole.vcf.gz"), "rb").read()) == open(os.path.join(GOLD, "advA.out.vcf"), "rb").read()


def test_sample_dependent_vcf_error_fails_only_its_sample(cache, tmp_path):
    """GT declared, sample columns, no GT in FORMAT: an error only once a record is called.  A sample of one all-N read calls
    nothing and gets a header-only VCF; the advA reads call sites and fail with rewrite_vcf's message."""
    vb.build()
    ds = cache.dataset("advA")
    prefix = _prefix(cache, "advA", tmp_path)
    vcf = str(tmp_path / "gt.vcf")
    with open(ds.vcf, "rb") as f, open(vcf, "wb") as o:
        for line in f:
            if line.startswith(b"##"):
                o.write(line)
            elif line.startswith(b"#"):
                o.write(b'##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n' + line.rstrip(b"\n") + b"\tFORMAT\tS1\n")
            else:
                o.write(line.rstrip(b"\n") + b"\tDP\t7\n")
    quiet = str(tmp_path / "quiet.fq")
    open(quiet, "wb").write(b"@q\n" + b"N" * 100 + b"\n+\n" + b"I" * 100 + b"\n")
    out_dir = str(tmp_path / "out")
    p = subprocess.run([vb.HOST_BIN, "geno-samples", prefix, _sheet(tmp_path, [("loud", ds.fastq), ("quiet", quiet)]), vcf, out_dir],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 1
    assert "sample loud: header declares GT but FORMAT has none" in p.stderr
    assert sorted(os.listdir(out_dir)) == ["quiet.vcf"]
    assert open(os.path.join(out_dir, "quiet.vcf"), "rb").read() == b"".join(
        l for l in open(vcf, "rb").read().splitlines(True) if l.startswith(b"#")).replace(
        b"#CHROM", b'##FORMAT=<ID=GQ,Number=1,Type=Integer,Description="Genotype Quality">\n#CHROM')
    q = subprocess.run([vb.HOST_BIN, "geno", prefix, ds.fastq, vcf, str(tmp_path / "loud.vcf")], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert q.returncode == 1 and "header declares GT but FORMAT has none" in q.stderr


def test_api_vcf_write_plain_and_bgzf(cache):
    """Genotyper.vcf_write from the golden calls: plain text equal to the golden VCF, BGZF inflating to it; a second context gets
    the template by vgb_vcf_template_copy"""
    from vargeno_b200.geno import Genotyper, site_gq
    gold = np.load(os.path.join(GOLD, "advB.npz"))
    ix = cache.index("advB")
    vcf = open(cache.dataset("advB").vcf, "rb").read()
    want = open(os.path.join(GOLD, "advB.out.vcf"), "rb").read()
    with Genotyper(device=0) as g:
        g.upload_index(ix)
        g.vcf_template(vcf)
        sites = g.sites()
        assert np.array_equal(sites["pos"], gold["sites"]["pos"])
        gt = np.zeros(g.n_sites, np.uint8)
        conf = np.zeros(g.n_sites)
        for i, s in enumerate(gold["sites"]):
            if s["ref"] != s["alt"]:
                gt[i], conf[i] = orc.call(int(s["ref_cnt"]), int(s["alt_cnt"]), int(s["ref_freq"]), int(s["alt_freq"]))
        gq = site_gq(gt, conf)
        assert g.vcf_write(gt, gq) == want
        buf = g.vcf_write(gt, gq, bgzf=True)
        _members_ok(buf)
        assert gzip.decompress(buf) == want
        with Genotyper(device=min(1, _gpu_count() - 1)) as h:
            h.upload_index(ix)
            h.vcf_template_copy(g)
            assert h.vcf_write(gt, gq) == want


def test_deflate_bgzf_of_fastq_reads_back_through_submit_bgzf(cache):
    """vgb_deflate_bgzf of advA's FASTQ text (host text, and the same text from device memory) fed back through vgb_submit_bgzf:
    the oracle's per-read results"""
    from vargeno_b200.geno import Genotyper
    ix = cache.index("advA")
    text = open(cache.dataset("advA").fastq, "rb").read()
    o = orc.Oracle(ix)
    want = o.process_fastq(np.frombuffer(text, dtype=np.uint8))
    o.close()
    with Genotyper(device=0, trace=True, max_chunk_bytes=1 << 22) as g:
        g.upload_index(ix)
        buf = g.deflate_bgzf(text)
        d = g.dalloc(len(text))
        g.h2d(d, np.frombuffer(text, dtype=np.uint8))
        assert g.deflate_bgzf((d, len(text))) == buf
        g.dfree(d)
        _members_ok(buf)
        assert gzip.decompress(buf) == text
        assert len(buf) <= 1.10 * len(bgzf.compress(text, level=1))
        g.submit_bgzf_file(buf, 1_000_000)
        g.sync()
        got = g.read_results()
    assert got.size == want.size
    for f in ("flags", "freq", "n_ref", "n_snp", "passes", "ctx_hash"):
        assert np.array_equal(got[f], want[f]), f


def test_deflate_bgzf_over_several_rounds():
    """text of three rounds and a bit (a round is 1024 blocks of 65280 bytes), and empty text"""
    from vargeno_b200.geno import Genotyper
    rng = np.random.default_rng(7)
    words = [b"chr%d\t%d\trs%d\tA\tC\t.\tPASS\tAF=0.%d\n" % (i % 23, i * 37, i, i % 97) for i in range(20000)]
    text = b"".join(words[int(k)] for k in rng.integers(0, len(words), 5_400_000))
    with Genotyper(device=0) as g:
        buf = g.deflate_bgzf(text)
        assert g.deflate_bgzf(b"") == bgzf.EOF_MEMBER
        assert g.deflate_bgzf(text[:1000], eof=False)[-28:] != bgzf.EOF_MEMBER
    assert len(text) > 3 * 1024 * 65280
    _members_ok(buf)
    assert gzip.decompress(buf) == text


def test_geno_reads_the_vcf_from_a_fifo(cache, tmp_path):
    """a VCF that is not a regular file (a FIFO, as `<(zcat snps.vcf.gz)` gives) is read to its end, not taken as empty"""
    vb.build()
    ds = cache.dataset("s0")
    prefix = _prefix(cache, "s0", tmp_path)
    fifo = str(tmp_path / "snps.fifo")
    os.mkfifo(fifo)
    data = open(ds.vcf, "rb").read()

    def feed():
        with open(fifo, "wb") as f:
            f.write(data)
    t = threading.Thread(target=feed)
    t.start()
    out = str(tmp_path / "out.vcf")
    p = subprocess.run([vb.HOST_BIN, "geno", prefix, ds.fastq, fifo, out], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    t.join()
    assert p.returncode == 0, p.stderr
    assert open(out, "rb").read() == open(os.path.join(GOLD, "s0.out.vcf"), "rb").read()


def _inflate_members(buf):
    mv = memoryview(buf)
    return b"".join(zlib.decompress(mv[off + poff:off + size - 8], -15) for off, size, poff, _ in bgzf.scan(buf))


def test_vcf_write_over_several_rounds_matches_vcf_rewrite(cache, tmp_path):
    """an output VCF of more than two rounds (a round is 1024 x 65280 bytes): records that straddle round boundaries, GT / GQ
    replaced in a sample column, against `vargeno-b200 vcf-rewrite` on the same calls; BGZF must inflate to the same bytes"""
    from vargeno_b200.geno import Genotyper, site_gq
    vb.build()
    ix = cache.index("advA")
    with Genotyper(device=0) as g:
        g.upload_index(ix)
        pos = g.sites()["pos"]
        cum = np.concatenate([[0], np.cumsum(ix.chr_lens)[:-1]])
        n = pos.size
        per = -(-1_600_000 // n)
        lines = [b"##fileformat=VCFv4.2\n", b'##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n',
                 b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\n"]
        for i, p in enumerate(pos.tolist()):
            c = int(np.searchsorted(cum, p, side="left")) - 1      # the contig whose range holds p (1-based positions)
            c = max(c, 0)
            name, rel = ix.chr_names[c].encode(), p - int(cum[c])
            for k in range(per):
                lines.append(b"%s\t%d\trs%d\tA\tC\t.\tPASS\tINFO=%s\tDP:GT:AD\t%d:0|1:%d,%d\tx\n"
                             % (name, rel, i * 1000 + k, b"x" * ((i * 7 + k * 13) % 90), k, i, k % 17))
        vcf = b"".join(lines)
        rng = np.random.default_rng(11)
        gt = np.where(rng.random(n) < 0.9, rng.integers(1, 4, n), 0).astype(np.uint8)
        conf = rng.uniform(1e-9, 1.0, n)
        g.vcf_template(vcf)
        plain = g.vcf_write(gt, site_gq(gt, conf))
        packed = g.vcf_write(gt, site_gq(gt, conf), bgzf=True)
    assert len(plain) > 2 * 1024 * 65280
    prefix = str(tmp_path / "ix")
    with open(prefix + ".chrlens", "w") as f:
        for nm, l in zip(ix.chr_names, ix.chr_lens):
            f.write("%s %d\n" % (nm, l))
    calls = str(tmp_path / "calls.tsv")
    with open(calls, "w") as f:
        f.write("".join("%d %d %s\n" % (p, x, c.hex()) for p, x, c in zip(pos.tolist(), gt.tolist(), conf.tolist())))
    vin, out = str(tmp_path / "in.vcf"), str(tmp_path / "host.vcf")
    open(vin, "wb").write(vcf)
    p = subprocess.run([vb.HOST_BIN, "vcf-rewrite", prefix, calls, vin, out], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr
    host = open(out, "rb").read()
    assert plain == host
    _members_ok(packed)
    assert _inflate_members(packed) == host
