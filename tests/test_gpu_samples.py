"""Many samples on one context (vgb_reset_sample) and `vargeno-b200 geno-samples`.

One index upload serves a sequence of samples in every input format.  After each sample the per-read results, the pileup
counters and the read count must be the oracle's for exactly that sample's reads: nothing of an earlier sample may leak into a
later one, also when the earlier one was a gzip stream or a BAM file abandoned half way, or an input that failed.  Through the
command line, every sample's VCF must be the file `geno` writes for it alone."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from oracle import oracle as orc
from vargeno_b200 import build as vb
from vargeno_b200.tools import bam, bgzf

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _gz(data, level=6):
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    return c.compress(data) + c.flush()


def _halves(text):
    lines = text.split(b"\n")
    assert lines[-1] == b""
    cut = (len(lines) - 1) // 8 * 4                  # a record boundary near the middle
    return b"\n".join(lines[:cut]) + b"\n", b"\n".join(lines[cut:])


@pytest.fixture(scope="module")
def adva(cache):
    ix = cache.index("advA")                       # mixed read lengths 31..250, N and lower case in reads
    text = open(cache.dataset("advA").fastq, "rb").read()
    return ix, text


def _oracle(ix, text):
    o = orc.Oracle(ix)
    want = o.process_fastq(np.frombuffer(text, dtype=np.uint8))
    sites = o.sites()
    o.close()
    return want, sites


def _check(g, ix, text):
    want, sites = _oracle(ix, text)
    g.sync()
    got = g.read_results()
    r, a = g.pileup()
    st = g.stats()
    assert got.size == want.size
    for f in ("flags", "freq", "n_ref", "n_snp", "passes", "ctx_hash"):
        bad = np.flatnonzero(got[f] != want[f])
        assert bad.size == 0, "%s differs for %d reads, first %s" % (f, bad.size, bad[:5])
    assert np.array_equal(r, sites["ref_cnt"]) and np.array_equal(a, sites["alt_cnt"])
    assert st["reads"] == want.size == text.count(b"\n") // 4


def test_samples_in_sequence_on_one_index_upload(adva):
    from vargeno_b200._lib import VGB_E_ARG, VgbError
    from vargeno_b200.geno import Genotyper
    ix, text = adva
    h1, h2 = _halves(text)
    full_bam = bam.write(bam.from_reads(bam.fastq_reads(text), aligned=True, extra_every=7, seed=3), level=1)
    with Genotyper(device=0, trace=True, max_chunk_bytes=1 << 20) as g:
        g.upload_index(ix)
        g.submit(h1)                                           # first half, plain
        _check(g, ix, h1)
        g.reset_sample()
        g.submit_gzip(_gz(h2), 40_000)                         # second half, single-stream gzip in small pieces
        _check(g, ix, h2)
        g.reset_sample()
        comp = _gz(text)
        g.submit_gzip(comp[:300_000], 300_000, first=True, last=False)   # a stream abandoned mid-way
        g.reset_sample()
        with pytest.raises(VgbError) as e:                     # the abandoned stream is gone: nothing to continue
            g.submit_gzip(comp[300_000:400_000], 100_000, first=False, last=True)
        assert e.value.code == VGB_E_ARG
        g.reset_sample()
        g.submit_gzip(_gz(h2), 40_000)                         # a new gzip stream: none of the abandoned stream's text in front
        _check(g, ix, h2)
        g.reset_sample()
        g.submit_bam(full_bam, 1 << 20)                        # the full set, aligned-style BAM
        _check(g, ix, text)
        g.reset_sample()
        calls = g.bam_calls(full_bam, 1 << 19)
        assert len(calls) > 1
        g.submit_bam_call(*calls[0], first=True, last=False)  # a BAM file abandoned after its first call
        g.reset_sample()
        with pytest.raises(VgbError) as e:
            g.submit_bam_call(*calls[1], first=False, last=True)
        assert e.value.code == VGB_E_ARG
        g.reset_sample()
        g.submit_bam(full_bam, 1 << 20)                        # a new BAM file: no carried bytes, no "truncated file"
        _check(g, ix, text)
        g.reset_sample()
        g.submit_bgzf_file(bgzf.compress(h1, level=1), 1 << 19)   # the first half again, BGZF
        _check(g, ix, h1)
        g.reset_sample()
        bad = bytearray(_gz(h1))                               # a corrupt gzip sample fails on sync ...
        bad[len(bad) // 2] ^= 0x55
        g.submit_gzip(bytes(bad), 50_000)
        with pytest.raises(VgbError):
            g.sync()
        g.reset_sample()
        g.submit(h2)                                           # ... and the next sample is exact
        _check(g, ix, h2)


def _cli(*args):
    return subprocess.run([vb.HOST_BIN] + [str(a) for a in args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


@pytest.fixture(scope="module")
def cohort(cache, tmp_path_factory):
    from vargeno_b200.tools import index_builder as ib
    vb.build()
    d = tmp_path_factory.mktemp("cohort")
    ds = cache.dataset("advA")
    prefix = str(d / "ix")
    ib.write_index(cache.index("advA"), prefix)
    text = open(ds.fastq, "rb").read()
    h1, h2 = _halves(text)
    files = {
        "full": ("full.fq", text),
        "full_bam": ("full.bam", bam.write(bam.from_reads(bam.fastq_reads(text), aligned=True, extra_every=7, seed=3), level=1)),
        "h1_bgzf": ("h1.fq.bgz", bgzf.compress(h1, level=1)),
        "h2_bgzf": ("h2.fq.bgz", bgzf.compress(h2, level=1)),
        "h1_gz": ("h1.fq.gz", _gz(h1, 1)),
        "h2_gz": ("h2.fq.gz", _gz(h2, 6)),
    }
    reads = {}
    for name, (fn, data) in files.items():
        (d / fn).write_bytes(data)
        reads[name] = str(d / fn)
    reads["pair"] = "%s,%s" % (reads["h1_gz"], reads["h2_bgzf"])     # two files back to back, one sample
    want = {}
    for name, r in reads.items():
        out = d / ("geno_%s.vcf" % name)
        p = _cli("geno", prefix, r, ds.vcf, out, "--chunk-mb", "1")
        assert p.returncode == 0, p.stderr
        want[name] = out.read_bytes()
    gold = open(os.path.join(GOLD, "advA.out.vcf"), "rb").read()
    for name in ("full", "full_bam", "pair"):
        assert want[name] == gold
    sheet = d / "samples.tsv"
    sheet.write_text("# name\treads\n" + "".join("%s\t%s\n" % kv for kv in reads.items()))
    return d, prefix, ds, reads, want, sheet


def _geno_samples(cohort, sheet, out, *extra):
    d, prefix, ds, reads, want, _ = cohort
    return _cli("geno-samples", prefix, sheet, ds.vcf, out, "--chunk-mb", "1", "--verbose", *extra)


def test_cli_every_vcf_is_what_geno_writes(cohort, tmp_path):
    d, prefix, ds, reads, want, sheet = cohort
    out = tmp_path / "out"
    p = _geno_samples(cohort, sheet, out)
    assert p.returncode == 0, p.stderr
    assert sorted(os.listdir(out)) == sorted(n + ".vcf" for n in reads)
    for name in reads:
        assert (out / (name + ".vcf")).read_bytes() == want[name], name
    assert p.stdout.startswith("Time: ")
    assert '"samples": %d, "failed": 0' % len(reads) in p.stderr


def test_cli_two_gpus(cohort, tmp_path):
    from test_gpu_cli import _gpu_count
    if _gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    d, prefix, ds, reads, want, sheet = cohort
    out = tmp_path / "out"
    p = _geno_samples(cohort, sheet, out, "--gpus", "2")
    assert p.returncode == 0, p.stderr
    for name in reads:
        assert (out / (name + ".vcf")).read_bytes() == want[name], name
    assert '"gpus": 2' in p.stderr


def test_cli_a_failed_sample_fails_alone(cohort, tmp_path):
    d, prefix, ds, reads, want, _ = cohort
    bad = bytearray(open(reads["h1_gz"], "rb").read())
    bad[len(bad) // 2] ^= 0x55
    (tmp_path / "bad.fq.gz").write_bytes(bytes(bad))
    keep = ("full", "h2_gz", "full_bam")
    sheet = tmp_path / "samples.tsv"
    sheet.write_text("full\t%s\nbroken\t%s\nh2_gz\t%s\nfull_bam\t%s\n" % (reads["full"], tmp_path / "bad.fq.gz", reads["h2_gz"], reads["full_bam"]))
    out = tmp_path / "out"
    p = _geno_samples(cohort, sheet, out)
    assert p.returncode != 0
    assert "sample broken: " in p.stderr, p.stderr
    assert sorted(os.listdir(out)) == sorted(n + ".vcf" for n in keep)
    for name in keep:
        assert (out / (name + ".vcf")).read_bytes() == want[name], name
