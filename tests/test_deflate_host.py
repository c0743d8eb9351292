"""The device BGZF writer (vargeno_b200/csrc/vgb_deflate.cuh) compiled for the HOST with one lane: every member must inflate with
zlib to its input with the right CRC32 and ISIZE, the file must be walkable by tools/bgzf.scan and end with the EOF member, and on
VCF text the output must stay within 1.10 x of zlib level 1 in the same 65280-byte blocks.  The GPU runs the same source with 32
lanes (tests/test_gpu_vcf_out.py)."""
import ctypes as C
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from vargeno_b200.tools import bgzf

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("deflate") / "libdeflate_host.so")
    subprocess.check_call(["g++", "-O2", "-Wall", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "native", "deflate_host.cpp")])
    L = C.CDLL(so)
    L.vgb_host_deflate_bgzf.restype = C.c_ulonglong
    L.vgb_host_deflate_bgzf.argtypes = [C.c_char_p, C.c_ulonglong, C.c_uint, C.c_char_p, C.c_ulonglong]
    return L


def _bgzf(lib, data, block=65280):
    cap = len(data) + (len(data) // block + 1) * 64 + 64
    out = C.create_string_buffer(cap)
    n = lib.vgb_host_deflate_bgzf(data, len(data), block, out, cap)
    assert n > 0
    return out.raw[:n]


def _check_members(buf, data, block=65280):
    """every member on its own: BC subfield, raw DEFLATE that inflates to its slice, CRC32 and ISIZE"""
    mem = bgzf.scan(buf)
    assert buf.endswith(bgzf.EOF_MEMBER)
    at = 0
    for off, size, poff, isize in mem:
        if isize == 0:
            continue
        payload = buf[off + poff:off + size - 8]
        text = zlib.decompressobj(-15).decompress(payload)
        crc, isz = struct.unpack("<II", buf[off + size - 8:off + size])
        assert text == data[at:at + len(text)] and len(text) <= block
        assert isz == len(text) == isize and crc == zlib.crc32(text) & 0xFFFFFFFF
        assert size <= 65536
        at += len(text)
    assert at == len(data)
    assert gzip.decompress(buf) == data


def _fastq(n, seed):
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n):
        seq = "".join("ACGT"[j] for j in rng.integers(0, 4, 150))
        qual = "".join(chr(35 + int(q)) for q in np.minimum(40, rng.geometric(0.08, 150)))
        recs.append("@r%09d\n%s\n+\n%s\n" % (i, seq, qual))
    return "".join(recs).encode()


def _vcf_text():
    return b"".join(open(os.path.join(GOLD, n + ".out.vcf"), "rb").read() for n in ("s0", "advA", "advB", "ucscA"))


CASES = {
    "empty": b"",
    "one_byte": b"A",
    "block_exact": _fastq(400, 1)[:65280],
    "block_plus_one": _fastq(400, 1)[:65281],
    "fastq": _fastq(900, 2),
    "random": np.random.default_rng(3).integers(0, 256, 200000, dtype=np.uint8).tobytes(),
    "one_repeated_byte": b"N" * 300000,
    # a run that reaches the end of a block exactly, and one that crosses it
    "run_to_block_end": _fastq(100, 4)[:65280 - 3000] + b"A" * 3000 + b"C" * 100,
    "run_across_block_end": _fastq(100, 5)[:65000] + b"T" * 5000,
    "vcf": _vcf_text(),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_members_inflate_to_their_input(lib, name):
    data = CASES[name]
    _check_members(_bgzf(lib, data), data)


@pytest.mark.parametrize("block", [1, 7, 1000, 30000])
def test_small_blocks(lib, block):
    data = CASES["vcf"][:120000]
    _check_members(_bgzf(lib, data, block), data, block)


def test_golden_vcfs_each(lib):
    for n in ("s0", "advA", "advB", "ucscA"):
        data = open(os.path.join(GOLD, n + ".out.vcf"), "rb").read()
        _check_members(_bgzf(lib, data), data)


def test_vcf_size_within_bar_of_zlib_level_1(lib):
    data = CASES["vcf"] * 4
    ours, ref = len(_bgzf(lib, data)), len(bgzf.compress(data, level=1))
    assert ours <= 1.10 * ref, (ours, ref)


def test_random_bytes_are_stored(lib):
    """incompressible text: stored blocks, 5 bytes over the input per member plus header and trailer"""
    data = CASES["random"][:65280]
    buf = _bgzf(lib, data)
    assert len(buf) == 18 + 5 + 65280 + 8 + 28
