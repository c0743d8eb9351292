"""Single-stream gzip FASTQ inflated on the device (vgb_submit_gzip: block finder, speculative decode, chain repair and window
resolution of csrc/vgb_gzip.cuh, which tests/test_inflate_gzip_host.py checks against zlib on the CPU), framed with the 32 KiB text
overlap: every record must be processed exactly once whatever the compression, the piece size and max_chunk_bytes.  Compared read
by read with the oracle, and through the command line with the golden VCF of the compiled reference."""
import gzip
import os
import subprocess
import zlib

import numpy as np
import pytest

from oracle import oracle as orc
from vargeno_b200 import build as vb

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _gz(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0):
    c = zlib.compressobj(level, zlib.DEFLATED, 31, 9, strategy)
    if not flush_every:
        return c.compress(data) + c.flush()
    parts = [c.compress(data[a:a + flush_every]) + c.flush(zlib.Z_SYNC_FLUSH) for a in range(0, len(data), flush_every)]
    return b"".join(parts) + c.flush()


def _compress(text, kind):
    if kind == "level1":
        return _gz(text, 1)
    if kind == "level6":
        return _gz(text, 6)
    if kind == "fixed":
        return _gz(text, 6, zlib.Z_FIXED)
    if kind == "sync_flush_128k":
        return _gz(text, 6, flush_every=128 << 10)
    cut = len(text) // 3 + 17                      # two members, cut inside a record
    return _gz(text[:cut], 1) + _gz(text[cut:], 9)


@pytest.fixture(scope="module")
def adva(cache):
    ix = cache.index("advA")                       # mixed read lengths 31..250, N and lower case in reads
    text = open(cache.dataset("advA").fastq, "rb").read()
    o = orc.Oracle(ix)
    want = o.process_fastq(np.frombuffer(text, dtype=np.uint8))
    sites = o.sites()
    o.close()
    return ix, text, want, sites


@pytest.mark.parametrize("kind", ["level1", "level6", "fixed", "sync_flush_128k", "two_members"])
@pytest.mark.parametrize("piece", [40_000, 1_000_000, "whole"])
def test_gzip_pieces_process_every_read_once(adva, kind, piece):
    from vargeno_b200.geno import Genotyper
    ix, text, want, sites = adva
    comp = _compress(text, kind)
    if piece == "whole":
        piece, max_chunk = len(comp), max(1 << 22, len(comp) + (1 << 16))
    else:
        max_chunk = 1 << 20                        # a few sub-streams per round: many rounds and calls
    with Genotyper(device=0, trace=True, max_chunk_bytes=max_chunk) as g:
        g.upload_index(ix)
        calls = g.submit_gzip(comp, piece)
        g.sync()
        got = g.read_results()
        r, a = g.pileup()
        st = g.stats()
    assert calls == -(-len(comp) // piece)
    assert got.size == want.size
    for f in ("flags", "freq", "n_ref", "n_snp", "passes", "ctx_hash"):
        bad = np.flatnonzero(got[f] != want[f])
        assert bad.size == 0, "%s differs for %d reads, first %s" % (f, bad.size, bad[:5])
    assert np.array_equal(r, sites["ref_cnt"]) and np.array_equal(a, sites["alt_cnt"])
    assert st["reads"] == want.size
    if max_chunk == 1 << 20:
        assert st["chunks"] > 2


def test_corrupt_truncated_isize_and_crc_are_loud(cache):
    from vargeno_b200._lib import VgbError
    from vargeno_b200.geno import Genotyper
    ix = cache.index("s0")
    text = open(cache.dataset("s0").fastq, "rb").read()[:400_000]
    text = text[:text.rfind(b"\n@") + 1]
    comp = _gz(text, 6)
    corrupt = bytearray(comp)
    corrupt[len(comp) // 2] ^= 0x55
    isize = bytearray(comp)
    isize[-1] ^= 0x01
    crc = bytearray(comp)
    crc[-8] ^= 0x01
    # the corrupt stream decodes to text of the right length (bits flipped inside base literals): the CRC32 check reports it
    for bad in (bytes(corrupt), comp[:len(comp) * 2 // 3], comp[:-4], bytes(isize), bytes(crc)):
        with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:
            g.upload_index(ix)
            g.submit_gzip(bad, 50_000)
            with pytest.raises(VgbError):
                g.sync()
    with Genotyper(device=0, max_chunk_bytes=1 << 20) as g:       # the intact stream, for contrast
        g.upload_index(ix)
        g.submit_gzip(comp + b"\0\0not gzip", 50_000)              # bytes behind the last member that are not one end the input
        g.sync()
        assert g.stats()["reads"] == text.count(b"\n") // 4


@pytest.mark.parametrize("chunk_mb", [1, 64])
def test_cli_gzip_input_gives_the_reference_vcf(cache, tmp_path, chunk_mb):
    """`vargeno-b200 geno` on a file written by gzip.open, and on two gzip files back to back, cut inside a record."""
    from vargeno_b200.tools import index_builder as ib
    vb.build()
    ds = cache.dataset("advA")
    prefix = str(tmp_path / "ix")
    ib.write_index(cache.index("advA"), prefix)
    text = open(ds.fastq, "rb").read()
    whole = tmp_path / "reads.fastq.gz"
    with gzip.open(whole, "wb") as f:
        f.write(text)
    out = str(tmp_path / "out.vcf")
    gold = open(os.path.join(GOLD, "advA.out.vcf"), "rb").read()
    p = subprocess.run([vb.HOST_BIN, "geno", prefix, str(whole), ds.vcf, out, "--chunk-mb", str(chunk_mb), "--verbose"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr
    assert open(out, "rb").read() == gold
    cut = len(text) // 2 + 23
    a, b = tmp_path / "a.fq.gz", tmp_path / "b.fq.gz"
    a.write_bytes(_gz(text[:cut], 1))
    b.write_bytes(_gz(text[cut:], 6, flush_every=100_000))
    p = subprocess.run([vb.HOST_BIN, "geno", prefix, "%s,%s" % (a, b), ds.vcf, out, "--chunk-mb", str(chunk_mb)], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr
    assert open(out, "rb").read() == gold
