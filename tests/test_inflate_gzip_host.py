"""Single-stream gzip on the CPU: vargeno_b200/csrc/vgb_gzip.cuh (block finder, speculative decode with window markers, chain check
and repair, window resolution, members) compiled for the HOST with one lane and driven step by step (tests/native/gzip_host.cpp),
against zlib.  Sub-stream spacings go down to a few hundred bytes, where most finder hits are false or fall inside a block, so the
repair path decides the result.  The GPU runs the same source (tests/test_gpu_gzip.py)."""
import ctypes as C
import gzip
import os
import subprocess
import zlib

import numpy as np
import pytest

from test_inflate_host import CASES, _fastq

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("gzip") / "libgzip_host.so")
    subprocess.check_call(["g++", "-O2", "-Wall", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "native", "gzip_host.cpp")])
    L = C.CDLL(so)
    L.vgb_host_gz_block_start.argtypes = [C.c_char_p, C.c_ulonglong, C.c_ulonglong]
    L.vgb_host_gz_spec.argtypes = [C.c_char_p, C.c_ulonglong, C.c_ulonglong, C.c_char_p, C.c_uint, C.c_char_p, C.c_uint,
                                   C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
    L.vgb_host_gunzip.argtypes = [C.c_char_p, C.c_ulonglong, C.c_uint, C.c_uint, C.c_uint, C.c_char_p, C.c_ulonglong,
                                  C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    return L


def _gzip(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flush_every=0):
    c = zlib.compressobj(level, zlib.DEFLATED, 31, 9, strategy)
    if not flush_every:
        return c.compress(data) + c.flush()
    out = []
    for a in range(0, len(data), flush_every):
        out.append(c.compress(data[a:a + flush_every]) + c.flush(zlib.Z_SYNC_FLUSH))
    return b"".join(out) + c.flush()


def _gunzip(lib, comp, spacing, max_sub=64, slice_=1 << 16, cap=None):
    cap = cap or 64 * len(comp) + (1 << 20)
    out = C.create_string_buffer(cap)
    n = C.c_ulonglong()
    st = (C.c_ulonglong * 4)()
    rc = lib.vgb_host_gunzip(comp, len(comp), spacing, max_sub, slice_, out, cap, C.byref(n), st)
    return rc, out.raw[:n.value], list(st)


def _block_starts(raw):
    """Bit offsets of every block header of a raw DEFLATE stream, with its type, from a plain sequential parse."""
    bits = np.unpackbits(np.frombuffer(raw, dtype=np.uint8), bitorder="little")
    pos = 0

    def take(k):
        nonlocal pos
        v = int(sum(int(bits[pos + i]) << i for i in range(k)))
        pos += k
        return v

    LB = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
    LE = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
    DE = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
    ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]

    def table(lens):
        codes, code = {}, 0
        for ln in range(1, 16):
            for s, l in enumerate(lens):
                if l == ln:
                    codes[(ln, code)] = s
                    code += 1
            code <<= 1
        return codes

    def sym(t):
        code, ln = 0, 0
        while True:
            code = (code << 1) | take(1)
            ln += 1
            if (ln, code) in t:
                return t[(ln, code)]

    out = []
    while True:
        start = pos
        final, typ = take(1), take(2)
        out.append((start, typ))
        if typ == 0:
            pos = (pos + 7) & ~7
            ln = take(16)
            take(16)
            pos += 8 * ln
        else:
            if typ == 1:
                lt = table([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)
                dt = table([5] * 30)
            else:
                nl, nd, nc = take(5) + 257, take(5) + 1, take(4) + 4
                cl = [0] * 19
                for i in range(nc):
                    cl[ORDER[i]] = take(3)
                ct = table(cl)
                lens = []
                while len(lens) < nl + nd:
                    s = sym(ct)
                    if s < 16:
                        lens.append(s)
                    elif s == 16:
                        lens += [lens[-1]] * (3 + take(2))
                    elif s == 17:
                        lens += [0] * (3 + take(3))
                    else:
                        lens += [0] * (11 + take(7))
                lt, dt = table(lens[:nl]), table(lens[nl:])
            while True:
                s = sym(lt)
                if s == 256:
                    break
                if s > 256:
                    take(LE[s - 257])
                    take(DE[sym(dt)])
        if final:
            return out


def _raw(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    return c.compress(data) + c.flush()


STRATEGIES = [(1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FILTERED),
              (6, zlib.Z_RLE), (6, zlib.Z_HUFFMAN_ONLY), (0, zlib.Z_DEFAULT_STRATEGY)]
FQ = _fastq(1500, 11)                          # ~480 KB of reads: several blocks at every level


@pytest.mark.parametrize("level,strategy", STRATEGIES)
def test_finder_accepts_every_true_block_start(lib, level, strategy):
    raw = _raw(FQ, level, strategy)
    starts = _block_starts(raw)
    assert len(starts) > 1 or level == 0
    for bit, typ in starts:
        if typ in (0, 2):
            assert lib.vgb_host_gz_block_start(raw, len(raw), bit) == 1, (bit, typ)


@pytest.mark.parametrize("level,strategy", STRATEGIES[:6])
def test_marker_decode_from_each_true_start(lib, level, strategy):
    """Decoded from a true block start without its window, resolved with the true preceding 32 KiB: zlib's text, byte for byte."""
    raw = _raw(FQ, level, strategy)
    starts = _block_starts(raw)
    marks = 0
    for bit, typ in starts[1:]:
        # how much text the stream holds from this block on tells where the block's text begins in FQ
        out = C.create_string_buffer(len(FQ) + 1)
        n, m = C.c_uint(), C.c_uint()
        rc = lib.vgb_host_gz_spec(raw, len(raw), bit, FQ, 0, out, len(FQ) + 1, C.byref(n), C.byref(m))
        assert rc == -2 or rc == 0                       # -2: markers cannot be resolved without a window
        tail_len = n.value
        head = FQ[:len(FQ) - tail_len]
        rc = lib.vgb_host_gz_spec(raw, len(raw), bit, head, len(head), out, len(FQ) + 1, C.byref(n), C.byref(m))
        assert rc == 0 and out.raw[:n.value] == FQ[len(head):]
        marks += m.value
    assert marks > 0 or strategy in (zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE)       # RLE matches rarely reach across a block start


@pytest.mark.parametrize("spacing", [300, 1000, 4096, 32768])
@pytest.mark.parametrize("level,strategy", STRATEGIES)
def test_driver_equals_zlib_fastq(lib, spacing, level, strategy):
    comp = _gzip(FQ, level, strategy)
    rc, out, st = _gunzip(lib, comp, spacing)
    assert rc == 0 and out == FQ, st


@pytest.mark.parametrize("spacing", [300, 2048])
@pytest.mark.parametrize("name", sorted(CASES))
def test_driver_equals_zlib_cases(lib, name, spacing):
    data = CASES[name]
    for level in (1, 6, 9):
        comp = _gzip(data, level)
        rc, out, st = _gunzip(lib, comp, spacing, max_sub=7)
        assert rc == 0 and out == data, (level, st)


@pytest.mark.parametrize("spacing", [400, 8192])
def test_fixed_huffman_is_repaired(lib, spacing):
    comp = _gzip(FQ, 6, zlib.Z_FIXED)
    rc, out, st = _gunzip(lib, comp, spacing)
    assert rc == 0 and out == FQ


def test_stored_only_and_sync_flush_and_members(lib):
    for comp in (_gzip(FQ, 0), _gzip(FQ * 2, 6, flush_every=128 << 10), _gzip(FQ[:100000], 1) + _gzip(FQ[100000:], 9),
                 gzip.compress(FQ[:7]) + gzip.compress(b"") + gzip.compress(FQ[7:])):
        for spacing in (500, 16384):
            rc, out, st = _gunzip(lib, comp, spacing, max_sub=5)
            want = gzip.decompress(comp)
            assert rc == 0 and out == want, (spacing, st)


def test_header_fields_and_trailing_garbage(lib):
    body = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = body.compress(FQ[:50000]) + body.flush()
    hdr = bytes([0x1f, 0x8b, 8, 4 | 8 | 16 | 2, 0, 0, 0, 0, 0, 3]) + (5).to_bytes(2, "little") + b"xxxxx" + b"name\0" + b"comment\0" + b"\0\0"
    trailer = (zlib.crc32(FQ[:50000])).to_bytes(4, "little") + (50000).to_bytes(4, "little")
    comp = hdr + raw + trailer
    rc, out, _ = _gunzip(lib, comp + b"\0\0garbage", 1000)
    assert rc == 0 and out == FQ[:50000]


def test_many_rounds_and_small_slices(lib):
    comp = _gzip(FQ, 6)
    rc, out, st = _gunzip(lib, comp, 2048, max_sub=3, slice_=4096)
    assert rc == 0 and out == FQ and st[2] > 3


def test_errors_are_reported(lib):
    comp = _gzip(FQ, 6)
    rc, _, _ = _gunzip(lib, comp[:len(comp) // 2], 1000)                          # truncated inside a block
    assert rc == 2
    rc, _, _ = _gunzip(lib, comp[:-3], 1000)                                        # truncated trailer
    assert rc == 2
    bad = bytearray(comp)
    bad[-1] ^= 1                                                                     # ISIZE
    rc, _, _ = _gunzip(lib, bytes(bad), 1000)
    assert rc == 3
    bad = bytearray(comp)
    bad[len(comp) // 3] ^= 0x5A                                                     # corrupt DEFLATE data
    rc, out, _ = _gunzip(lib, bytes(bad), 1000)
    assert rc != 0
    rng = np.random.default_rng(9)
    for spacing in (300, 3000):
        for _ in range(20):
            junk = bytearray(comp[:20000])
            for i in rng.integers(10, len(junk), 5):
                junk[i] = int(rng.integers(0, 256))
            rc, out, _ = _gunzip(lib, bytes(junk), spacing)
            assert rc != 0


def test_crc32_is_checked(lib):
    """A corrupt stream can decode to text of the right length (flipped bits inside equal-length literal codes): only the member's
    CRC32 tells.  Checked for the CRC field itself and for corruption anywhere in the DEFLATE data that zlib rejects."""
    comp = _gzip(FQ, 6)
    bad = bytearray(comp)
    bad[-8] ^= 1                                                                     # CRC32 field
    rc, _, _ = _gunzip(lib, bytes(bad), 1000)
    assert rc == 5
    silent = 0
    for at in range(len(comp) // 4, len(comp) // 4 + 40):
        bad = bytearray(comp)
        bad[at] ^= 0x55
        try:
            zlib.decompress(bytes(bad), 31)
            continue                                                                 # still a valid stream (does not happen here)
        except zlib.error:
            pass
        rc, _, _ = _gunzip(lib, bytes(bad), 4096)
        assert rc != 0, at
        silent += rc == 5
    assert silent > 0                                                                # some of them decode to the right length
