"""BAM to FASTQ on the CPU: vargeno_b200/csrc/vgb_bam.cuh (header, record check, speculative tile starts, chain check and repair,
record list, round plan, conversion) compiled for the HOST and driven call by call with the unconsumed bytes carried over
(tests/native/bam_host.cpp), against the plain-Python contract of vargeno_b200/tools/bam.py.  Tiles go down to 64 bytes, where every
record crosses tiles and most tile starts are repaired.  The GPU runs the same source (tests/test_gpu_bam.py)."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

from vargeno_b200.tools import bam

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("bam") / "libbam_host.so")
    subprocess.check_call(["g++", "-O2", "-Wall", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "native", "bam_host.cpp")])
    L = C.CDLL(so)
    L.vgb_host_bam_check.argtypes = [C.c_char_p, C.c_uint, C.c_uint, C.c_int]
    L.vgb_host_bam_header.argtypes = [C.c_char_p, C.c_ulonglong, C.POINTER(C.c_ulonglong), C.POINTER(C.c_int)]
    L.vgb_host_bam_fastq.argtypes = [C.c_char_p, C.c_ulonglong, C.POINTER(C.c_ulonglong), C.c_uint, C.c_uint, C.c_ulonglong, C.c_uint,
                                     C.c_char_p, C.c_ulonglong, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    return L


def _reads(n, seed, max_len=250):
    """(name, seq, qual): lengths 0 .. max_len, N and lower case"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        ln = int(rng.integers(0, max_len + 1)) if i % 17 else 0 if i % 34 == 0 else 31
        seq = bytes(rng.choice(list(b"ACGTNacgt"), ln, p=[.22, .22, .22, .22, .02, .025, .025, .025, .025]).astype(np.uint8)) if ln else b""
        qual = bytes((33 + np.minimum(41, rng.geometric(0.08, ln))).astype(np.uint8))
        out.append((b"r%07d" % i, seq, qual))
    return out


def _expect(reads):
    return b"".join(b"@\n" + s.upper() + b"\n+\n" + q + b"\n" for _, s, q in reads if s)


def _run(lib, raw, cuts=None, tile=65536, max_header=1 << 20, round_cap=1 << 30):
    cuts = list(cuts) if cuts is not None else [len(raw)]
    cut_arr = (C.c_ulonglong * len(cuts))(*cuts)
    cap = 2 * len(raw) + 1024
    out = C.create_string_buffer(cap)
    n = C.c_ulonglong()
    st = (C.c_ulonglong * 6)()
    rc = lib.vgb_host_bam_fastq(raw, len(raw), cut_arr, len(cuts), tile, max_header, round_cap, out, cap, C.byref(n), st)
    return rc, out.raw[:n.value], list(st)


def _members(raw, sizes):
    """the uncompressed bytes and member ends of raw written as BGZF with member sizes `sizes` (cycled)"""
    got, ends = bam.inflate(bam.write(raw, sizes=sizes, level=1))
    assert got == raw
    return ends


def _fake_record():
    """a well-formed record, to hide inside names-free places (aux arrays) where the finder will take it for a record start"""
    return bam.record(b"fake", b"ACGTACGTAC", b"IIIIIIIIII", flag=0)


def _adversarial(n, seed):
    """aligned-style records whose aux payloads hold whole fake records and whose names look like headers"""
    rng = np.random.default_rng(seed)
    out = [bam.header([("chr1", 1000), ("chr2", 2000)])]
    fake = _fake_record()
    reads = _reads(n, seed)
    for i, (name, seq, qual) in enumerate(reads):
        payload = fake * int(rng.integers(1, 4)) + bytes(rng.integers(0, 3, int(rng.integers(0, 40)), dtype=np.uint8))
        aux = b"XBBC" + struct.pack("<i", len(payload)) + payload
        nm = b"!!!!" + name if i % 3 == 0 else name
        out.append(bam.record(nm, seq, qual, flag=0, ref_id=int(rng.integers(-1, 2)), pos=5, cigar=[(len(seq), 0)] if seq else [], aux=aux))
    return b"".join(out), reads


def test_python_contract_on_plain_reads():
    reads = _reads(300, 1)
    assert bam.to_fastq(bam.write(bam.from_reads(reads))) == _expect(reads)
    assert bam.to_fastq(bam.from_reads(reads, aligned=True, extra_every=3)) == _expect(reads)


@pytest.mark.parametrize("aligned", [False, True])
def test_check_accepts_every_true_record_start(lib, aligned):
    raw = bam.from_reads(_reads(400, 2), aligned=aligned, extra_every=5)
    for extra in (b"", _adversarial(100, 3)[0]):
        data = raw if not extra else extra
        starts, n_ref = bam.record_starts(data)
        assert starts
        for o in starts:
            assert lib.vgb_host_bam_check(data, len(data), o, n_ref) == 1, o
        assert lib.vgb_host_bam_check(data, len(data), starts[-1] + 1, n_ref) != 1


@pytest.mark.parametrize("tile", [64, 100, 1000, 4096, 65536])
@pytest.mark.parametrize("kind", ["ubam", "aligned", "adversarial"])
def test_pipeline_equals_contract(lib, kind, tile):
    if kind == "adversarial":
        raw, reads = _adversarial(300, 4)
    else:
        reads = _reads(600, 5)
        raw = bam.from_reads(reads, aligned=kind == "aligned", extra_every=4)
    want = _expect(reads)
    assert bam.to_fastq(raw) == want
    for cuts in ([len(raw)], _members(raw, [65280]), _members(raw, [97, 1500, 3, 40000, 777])):
        rc, out, st = _run(lib, raw, cuts, tile=tile)
        assert rc == 0 and out == want, (len(cuts), st)
        if tile <= 100:
            assert st[1] > 0                                          # repairs forced
    if kind == "adversarial" and tile == 65536:
        assert _run(lib, raw, tile=tile)[2][1] >= 0


def test_rounds(lib):
    reads = _reads(500, 6)
    raw = bam.from_reads(reads)
    want = _expect(reads)
    rc, out, st = _run(lib, raw, tile=512, round_cap=len(want) // 5)
    assert rc == 0 and out == want and st[4] >= 5
    rc, _, _ = _run(lib, raw, round_cap=len(want) // 20)                 # more than BAM_ROUNDS rounds
    assert rc == 7


def test_large_aux_crossing_members(lib):
    rng = np.random.default_rng(7)
    reads = _reads(60, 8)
    out = [bam.header([("chr1", 10)])]
    for i, (name, seq, qual) in enumerate(reads):
        n = 70000 if i % 7 == 3 else int(rng.integers(0, 200))
        payload = bytes(rng.integers(0, 256, n, dtype=np.uint8))
        out.append(bam.record(name, seq, qual, aux=b"XBBC" + struct.pack("<i", n) + payload))
    raw = b"".join(out)
    want = _expect(reads)
    for tile in (64, 4096, 65536):
        for cuts in ([len(raw)], _members(raw, [65280]), _members(raw, [5000, 333])):
            rc, got, st = _run(lib, raw, cuts, tile=tile)
            assert rc == 0 and got == want, (tile, st)
            assert st[5] >= 0


def test_large_header(lib):
    refs = [("contig_%05d_%s" % (i, "x" * (i % 50)), 1000 + i) for i in range(5000)]
    text = b"@HD\tVN:1.6\n" + b"@CO\t" + b"y" * 300000 + b"\n"
    reads = _reads(200, 9)
    raw = bam.header(refs, text) + b"".join(bam.record(n, s, q, ref_id=i % 5000) for i, (n, s, q) in enumerate(reads))
    hl = bam.parse_header(raw)[0]
    assert hl > 3 * 65280
    want = _expect(reads)
    for cuts in (_members(raw, [65280]), _members(raw, [20000, 7])):
        rc, got, st = _run(lib, raw, cuts, tile=256)
        assert rc == 0 and got == want
        assert st[5] >= hl - 65280                                    # the header was carried over calls
    n, r = C.c_ulonglong(), C.c_int()
    assert lib.vgb_host_bam_header(raw, len(raw), C.byref(n), C.byref(r)) == 0 and n.value == hl and r.value == 5000
    assert lib.vgb_host_bam_header(raw, hl - 1, C.byref(n), C.byref(r)) == 1
    rc, _, _ = _run(lib, raw, _members(raw, [65280]), max_header=hl - 1)
    assert rc == 2


def test_flags_missing_quality_and_empty_records(lib):
    recs = [
        (bam.record(b"a", b"ACGTTGCA", b"ABCDEFGH"), b"@\nACGTTGCA\n+\nABCDEFGH\n"),
        (bam.record(b"b", bam.revcomp(b"AACCGGTN"), b"HGFEDCBA", flag=0x10), b"@\nAACCGGTN\n+\nABCDEFGH\n"),
        (bam.record(b"c", b"ACGT", b"IIII", flag=0x100), b""),
        (bam.record(b"d", b"ACGT", b"IIII", flag=0x800), b""),
        (bam.record(b"e", b"ACGT", b"IIII", flag=0x900 | 0x10), b""),
        (bam.record(b"f", b"ACGTA", None), b'@\nACGTA\n+\n"""""\n'),
        (bam.record(b"g", b"ACGTA", None, flag=0x10), b'@\nTACGT\n+\n"""""\n'),
        (bam.record(b"h", b"", b""), b""),
        (bam.record(b"i", b"", None, flag=0x10), b""),
        (bam.record(b"j", b"MRSVWYHKDB=", b"IIIIIIIIIII"), b"@\nMRSVWYHKDB=\n+\nIIIIIIIIIII\n"),
        (bam.record(b"k", b"MRSVWYHKDB=", b"ABCDEFGHIJK", flag=0x10 | 0x1 | 0x40), b"@\n=VHMDRWBSYK\n+\nKJIHGFEDCBA\n"),
    ]
    raw = bam.header() + b"".join(r for r, _ in recs)
    want = b"".join(w for _, w in recs)
    assert bam.to_fastq(raw) == want
    for tile in (64, 65536):
        rc, got, _ = _run(lib, raw, tile=tile)
        assert rc == 0 and got == want


def test_errors_are_reported(lib):
    reads = _reads(200, 10)
    raw = bam.from_reads(reads)
    starts, _ = bam.record_starts(raw)
    hl = bam.parse_header(raw)[0]
    mid = starts[100]
    # truncated: inside a record, inside the header, inside a length field
    for cut in (mid + 20, hl - 3, mid + 2, 3):
        rc, _, _ = _run(lib, raw[:cut], tile=128)
        assert rc == 5, cut
        with pytest.raises(ValueError):
            bam.to_fastq(raw[:cut])
    bad = b"BAM\x02" + raw[4:]
    assert _run(lib, bad)[0] == 1
    for size, code in ((20, 3), (2 << 20, 4)):
        b = bytearray(raw)
        b[mid:mid + 4] = struct.pack("<i", size)                             # block_size too small / record over the limit
        for tile in (64, 65536):
            rc, _, _ = _run(lib, bytes(b), _members(bytes(b), [3000]), tile=tile)
            assert rc == code, (size, tile)
        with pytest.raises(ValueError):
            bam.to_fastq(bytes(b))
    long_read = [(b"x", b"A" * 1500, b"I" * 1500)]
    raw2 = bam.from_reads(reads[:10] + long_read + reads[10:20])
    rc, got, st = _run(lib, raw2, tile=256)
    assert rc == 6 and st[3] == 1 and got == _expect(reads[:20])
    with pytest.raises(ValueError):
        bam.to_fastq(raw2)
    # a corrupt record in the middle of a tile, reached only by the chain
    b = bytearray(raw)
    b[starts[150] + 4:starts[150] + 8] = struct.pack("<i", 7)                # refID out of range
    assert _run(lib, bytes(b), tile=4096)[0] == 3


def test_repair_share_model_matches_the_pipeline(lib):
    raw, _ = _adversarial(400, 11)
    for tile in (256, 4096):
        nt, rep = bam.repair_share(raw, tile)
        rc, _, st = _run(lib, raw, tile=tile)
        assert rc == 0 and st[0] == nt and st[1] == rep
