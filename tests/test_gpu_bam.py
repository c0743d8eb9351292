"""BAM input on the device (vgb_submit_bam: BGZF members inflated by k_inflate_bgzf, records framed, chain-checked and converted
to FASTQ text by csrc/vgb_bam.cuh, which tests/test_bam_host.py checks on the CPU).  advA written as unaligned BAM and as
aligned-style BAM (half the reads reverse-complemented with flag 0x10, secondary and supplementary copies with other sequences
inserted) must give the oracle's per-read results on the original FASTQ, whatever the members and max_chunk_bytes; through the
command line, the golden VCF of the compiled reference."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from vargeno_b200 import build as vb
from vargeno_b200.tools import bam

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _bam(text, kind, members):
    reads = bam.fastq_reads(text)
    raw = bam.from_reads(reads, aligned=kind == "aligned", extra_every=7 if kind == "aligned" else 0, seed=3)
    return bam.write(raw, sizes=[97, 4000, 12345, 3]) if members == "tiny" else bam.write(raw, level=1)


@pytest.fixture(scope="module")
def adva(cache):
    ix = cache.index("advA")                       # mixed read lengths 31..250, N and lower case in reads
    text = open(cache.dataset("advA").fastq, "rb").read()
    o = orc.Oracle(ix)
    want = o.process_fastq(np.frombuffer(text, dtype=np.uint8))
    sites = o.sites()
    o.close()
    return ix, text, want, sites


@pytest.mark.parametrize("kind", ["ubam", "aligned"])
@pytest.mark.parametrize("members", ["bgzip", "tiny"])
@pytest.mark.parametrize("max_chunk", [1 << 20, "whole"])
def test_bam_gives_the_oracle_read_by_read(adva, kind, members, max_chunk):
    from vargeno_b200.geno import Genotyper
    ix, text, want, sites = adva
    buf = _bam(text, kind, members)
    if max_chunk == "whole":
        max_chunk = 2 * len(text) + (1 << 20)
    with Genotyper(device=0, trace=True, max_chunk_bytes=max_chunk) as g:
        g.upload_index(ix)
        calls = g.submit_bam(buf, max_chunk)
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
    if max_chunk == 1 << 20:
        assert calls > 4


def test_bad_bam_is_loud(cache):
    import struct

    from vargeno_b200._lib import VgbError
    from vargeno_b200.geno import Genotyper
    ix = cache.index("s0")
    text = open(cache.dataset("s0").fastq, "rb").read()[:400_000]
    text = text[:text.rfind(b"\n@") + 1]
    reads = bam.fastq_reads(text)
    raw = bam.from_reads(reads)
    starts, _ = bam.record_starts(raw)
    mid = starts[len(starts) // 2]
    small, big = bytearray(raw), bytearray(raw)
    small[mid:mid + 4] = struct.pack("<i", 20)
    big[mid:mid + 4] = struct.pack("<i", 2 << 20)
    long_read = bam.from_reads(reads[:5] + [(b"x", b"A" * 1500, b"I" * 1500)])
    for bad in (raw[:len(raw) * 2 // 3], raw[:10], b"BAM\x02" + raw[4:], bytes(small), bytes(big), long_read):
        with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:
            g.upload_index(ix)
            g.submit_bam(bam.write(bad, sizes=[30000]), 1 << 20)
            with pytest.raises(VgbError):
                g.sync()
    with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:      # the intact file, for contrast
        g.upload_index(ix)
        g.submit_bam(bam.write(raw, sizes=[30000]), 1 << 20)
        g.sync()
        assert g.stats()["reads"] == len(reads)


def _cli(prefix, reads, vcf, out, *extra):
    return subprocess.run([vb.HOST_BIN, "geno", prefix, reads, vcf, out, "--chunk-mb", "1"] + list(extra), stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True)


def _cli_setup(cache, tmp_path):
    from vargeno_b200.tools import index_builder as ib
    vb.build()
    ds = cache.dataset("advA")
    prefix = str(tmp_path / "ix")
    ib.write_index(cache.index("advA"), prefix)
    text = open(ds.fastq, "rb").read()
    cut = text.index(b"\n@", len(text) // 2) + 1
    one = tmp_path / "reads.bam"
    one.write_bytes(_bam(text, "aligned", "bgzip"))
    a, b = tmp_path / "a.bam", tmp_path / "b.bam"
    a.write_bytes(_bam(text[:cut], "ubam", "bgzip"))
    b.write_bytes(_bam(text[cut:], "aligned", "tiny"))
    gold = open(os.path.join(GOLD, "advA.out.vcf"), "rb").read()
    return ds, prefix, text, one, a, b, gold


def test_cli_bam_input_gives_the_reference_vcf(cache, tmp_path):
    ds, prefix, text, one, a, b, gold = _cli_setup(cache, tmp_path)
    out = str(tmp_path / "out.vcf")
    for reads in (str(one), "%s,%s" % (a, b)):
        p = _cli(prefix, reads, ds.vcf, out, "--verbose")
        assert p.returncode == 0, p.stderr
        assert open(out, "rb").read() == gold
    fq = tmp_path / "plain.fq"
    fq.write_bytes(text)
    p = _cli(prefix, "%s,%s" % (one, fq), ds.vcf, out)
    assert p.returncode != 0 and "mixes BAM" in p.stderr


def test_cli_bam_two_gpus(cache, tmp_path):
    from test_gpu_cli import _gpu_count
    if _gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    ds, prefix, text, one, a, b, gold = _cli_setup(cache, tmp_path)
    out = str(tmp_path / "out.vcf")
    p = _cli(prefix, "%s,%s" % (a, b), ds.vcf, out, "--gpus", "2")
    assert p.returncode == 0, p.stderr
    assert open(out, "rb").read() == gold
