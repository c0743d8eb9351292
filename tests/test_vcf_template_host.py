"""The VCF template and splice of the device writer (vargeno_b200/csrc/vgb_vcf.cuh) compiled for the HOST must write, for the same
calls, byte for byte what `vargeno-b200 vcf-rewrite` (calls_to_map + rewrite_vcf, the host reference) writes -- and fail with
its message where it fails.  Golden data sets with their golden calls, and small VCFs for every sample-dependent rule."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from vargeno_b200 import build as vb

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("vcf") / "libvcf_host.so")
    subprocess.check_call(["g++", "-O2", "-Wall", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "native", "vcf_host.cpp")])
    L = C.CDLL(so)
    L.vgb_host_vcf_splice.argtypes = [C.c_char_p, C.c_ulonglong, C.c_char_p, C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_ulonglong, C.POINTER(C.c_void_p), C.POINTER(C.c_ulonglong), C.c_char_p]
    L.vgb_host_free.argtypes = [C.c_void_p]
    vb.build()
    return L


def _splice(L, vcf, names, lens, pos, gt, conf):
    lens = np.ascontiguousarray(lens, dtype=np.uint64)
    pos = np.ascontiguousarray(pos, dtype=np.uint32)
    gt = np.ascontiguousarray(gt, dtype=np.uint8)
    conf = np.ascontiguousarray(conf, dtype=np.float64)
    out, n, err = C.c_void_p(), C.c_ulonglong(), C.create_string_buffer(256)
    rc = L.vgb_host_vcf_splice(vcf, len(vcf), "\n".join(names).encode(), lens.ctypes.data, len(names), pos.ctypes.data, gt.ctypes.data,
                               conf.ctypes.data, pos.size, C.byref(out), C.byref(n), err)
    if rc:
        return rc, err.value.decode()
    data = C.string_at(out.value, n.value)
    L.vgb_host_free(out)
    return 0, data


def _rewrite(tmp_path, vcf, names, lens, pos, gt, conf):
    prefix = str(tmp_path / "ix")
    with open(prefix + ".chrlens", "w") as f:
        for n, l in zip(names, lens):
            f.write("%s %d\n" % (n, l))
    with open(str(tmp_path / "calls.tsv"), "w") as f:
        for p, g, c in zip(pos, gt, conf):
            f.write("%d %d %s\n" % (int(p), int(g), float(c).hex()))
    open(str(tmp_path / "in.vcf"), "wb").write(vcf)
    out = str(tmp_path / "out.vcf")
    p = subprocess.run([vb.HOST_BIN, "vcf-rewrite", prefix, str(tmp_path / "calls.tsv"), str(tmp_path / "in.vcf"), out],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if p.returncode:
        return 1, p.stderr.strip().replace("vargeno-b200: ", "")
    return 0, open(out, "rb").read()


def _check(L, tmp_path, vcf, names, lens, pos, gt, conf):
    want = _rewrite(tmp_path, vcf, names, lens, pos, gt, conf)
    got = _splice(L, vcf, names, lens, pos, gt, conf)
    assert (got[0] != 0) == (want[0] != 0), (got, want)
    assert got[1] == want[1]
    return got


@pytest.mark.parametrize("name", ["s0", "advA", "advB"])
def test_golden_calls(lib, cache, name, tmp_path):
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    ix = cache.index(name)
    pos, gt, conf = [], [], []
    for s in gold["sites"]:
        g, c = (0, 0.0)
        if s["ref"] != s["alt"]:
            g, c = orc.call(int(s["ref_cnt"]), int(s["alt_cnt"]), int(s["ref_freq"]), int(s["alt_freq"]))
        pos.append(int(s["pos"])); gt.append(g); conf.append(c)
    vcf = open(cache.dataset(name).vcf, "rb").read()
    rc, out = _check(lib, tmp_path, vcf, ix.chr_names, ix.chr_lens, pos, gt, conf)
    assert rc == 0 and out == open(os.path.join(GOLD, name + ".out.vcf"), "rb").read()


def _vcf_sites(vcf, names, lens):
    """concatenated positions of the data lines of a VCF (CHROM with or without 'chr')"""
    cum = dict(zip(names, np.concatenate([[0], np.cumsum(lens)[:-1]])))
    out = set()
    for line in vcf.split(b"\n"):
        c = line.split(b"\t")
        if len(c) < 2 or line.startswith(b"#"):
            continue
        ch = c[0].decode()
        ch = ch if ch.startswith("c") else "chr" + ch
        if ch in cum and c[1].isdigit():
            out.add(int(cum[ch]) + int(c[1]))
    return sorted(out)


def _random_calls(n, seed, p_call=0.6):
    rng = np.random.default_rng(seed)
    gt = np.where(rng.random(n) < p_call, rng.integers(1, 4, n), 0)
    conf = rng.uniform(1e-6, 1.0, n)
    return gt, conf


def test_ucsc_set_random_calls(lib, cache, tmp_path):
    ix = cache.index("ucscA")
    vcf = open(cache.dataset("ucscA").vcf, "rb").read()
    pos = _vcf_sites(vcf, ix.chr_names, ix.chr_lens)
    pos = sorted(set(pos) | {p + 1 for p in pos[::7]})            # sites that match no record as well
    for seed in range(3):
        gt, conf = _random_calls(len(pos), seed)
        rc, _ = _check(lib, tmp_path, vcf, ix.chr_names, ix.chr_lens, pos, gt, conf)
        assert rc == 0


NAMES, LENS = ["chr1", "chr2"], [1000, 500]
GT_HDR = b'##fileformat=VCFv4.2\n##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
GQ_HDR = b'##FORMAT=<ID=GQ,Number=1,Type=Integer,Description="Genotype Quality">\n'
COLS10 = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n"
COLS8 = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"


def _rec(chrom, pos, fmt=None, smp=None, extra=b""):
    r = b"%s\t%s\tid\tA\tC\t.\tPASS\tX=1" % (chrom, pos)
    if fmt is not None:
        r += b"\t" + fmt + b"\t" + smp
    return r + extra + b"\n"


def _all_calls(vcf, gt_value=3, names=NAMES, lens=LENS, call_every=1):
    pos = _vcf_sites(vcf, names, lens)
    gt = [gt_value if i % call_every == 0 else 0 for i in range(len(pos))]
    conf = [0.5 / (i + 1) for i in range(len(pos))]
    return pos, gt, conf


CASES = {
    # sample columns, GT declared; GT at different places
    "gt_declared": GT_HDR + COLS10 + _rec(b"chr1", b"10", b"GT:DP", b"0|1:5") + _rec(b"chr1", b"20", b"DP:GT", b"7:1|1") +
    _rec(b"chr2", b"5", b"GT", b"0|0", b"\tS2extra"),
    # the header declares GQ (and GT)
    "gq_declared": GT_HDR + GQ_HDR + COLS10 + _rec(b"chr1", b"10", b"GT:GQ", b"0|1:5"),
    # GQ declared, GT not
    "gq_without_gt": b"##fileformat=VCFv4.2\n" + GQ_HDR + COLS10 + _rec(b"chr1", b"10", b"GT:GQ", b"0|1:5"),
    # ## lines behind the '#' line: GQ index preset, then declared
    "gq_declared_late": COLS10 + GQ_HDR + _rec(b"chr1", b"10", b"GT:GQ:DP", b"0|1:5:3") + _rec(b"chr1", b"11", b"GT", b"0|1"),
    "gt_declared_late": COLS10 + GT_HDR + _rec(b"chr1", b"10", b"DP:GT", b"3:0|1"),
    # FORMAT without GT while the header declares it
    "format_without_gt": GT_HDR + COLS10 + _rec(b"chr1", b"10", b"DP", b"5"),
    # the first called record fixes the GT index for the later ones
    "first_format_differs": GT_HDR + COLS10 + _rec(b"chr1", b"10", b"DP:GT", b"5:0|1") + _rec(b"chr1", b"20", b"GT:DP", b"1|1:9") +
    _rec(b"chr1", b"30", b"GT:DP:AD", b"0|0:2:1,1"),
    "first_format_differs_short": GT_HDR + COLS10 + _rec(b"chr1", b"10", b"DP:GT", b"5:0|1") + _rec(b"chr1", b"20", b"GT", b"1|1"),
    # no sample columns: two columns appended
    "no_sample_columns": COLS8 + _rec(b"chr1", b"10") + _rec(b"chr2", b"7"),
    "no_sample_columns_gt": GT_HDR + COLS8 + _rec(b"chr1", b"10"),
    # GT declared, a '#' line of fewer than 10 columns, data lines with GT in FORMAT: rewrite_vcf searches an empty FORMAT
    "no_sample_columns_gt_in_format": GT_HDR + COLS8 + _rec(b"chr1", b"10", b"GT:DP", b"0|1:5") + _rec(b"chr1", b"20", b"DP:GT", b"3:1|1"),
    # CHROM without 'chr', POS with leading zeros, blank lines, one-column lines, CRLF
    "chrom_without_chr": COLS8 + _rec(b"1", b"10") + _rec(b"2", b"7") + _rec(b"chr1", b"30"),
    "pos_leading_zeros": COLS8 + _rec(b"chr1", b"010") + _rec(b"chr1", b"10") + _rec(b"chr1", b"+20"),
    "blank_and_short_lines": COLS8 + b"\n\n" + b"lonely\n" + _rec(b"chr1", b"10") + b"\n" + b"x\r\n" + _rec(b"chr1", b"11"),
    "crlf": GT_HDR.replace(b"\n", b"\r\n") + COLS10.replace(b"\n", b"\r\n") + _rec(b"chr1", b"10", b"GT:DP", b"0|1:5", b"\r") +
    _rec(b"chr1", b"11", b"DP:GT", b"5:0|1", b"\r") + _rec(b"chr1", b"12", b"GT", b"0|1", b"\r"),
    "crlf_no_samples": COLS8.replace(b"\n", b"\r\n") + _rec(b"chr1", b"10", extra=b"\r"),
    # two records at one site
    "two_records_one_site": COLS8 + _rec(b"chr1", b"10") + _rec(b"chr1", b"10", extra=b";second"),
    # no newline at the end; a header with no '#' line at all
    "no_final_newline": COLS8 + _rec(b"chr1", b"10")[:-1],
    "no_header_line": b"##x\n" + _rec(b"chr1", b"10") + _rec(b"chr1", b"12", b"A", b"B"),
    "no_header_line_gq": GQ_HDR + _rec(b"chr1", b"10"),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_small_vcfs(lib, name, tmp_path):
    vcf = CASES[name]
    for gv in (1, 2, 3):
        for every in (1, 2):
            _check(lib, tmp_path, vcf, NAMES, LENS, *_all_calls(vcf, gv, call_every=every))


def test_sites_sharing_a_key(lib, tmp_path):
    """two sites with one key (two contigs of the same name, and a repeated position): the last CALLED one wins"""
    names, lens = ["chr1", "chr1", "chr2"], [100, 100, 50]
    vcf = COLS8 + _rec(b"chr1", b"10") + _rec(b"chr1", b"40") + _rec(b"chr2", b"5")
    pos = [10, 40, 110, 140, 140, 205]
    for gt in ([1, 2, 3, 0, 1, 2], [1, 0, 0, 2, 3, 0], [0, 2, 1, 3, 0, 1], [3, 3, 0, 0, 2, 2]):
        conf = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6]
        _check(lib, tmp_path, vcf, names, lens, pos, gt, conf)


def test_error_record_called_or_not(lib, tmp_path):
    """a record with fewer than 10 columns under a 10-column header fails the sample only when it is called"""
    vcf = GT_HDR + COLS10 + _rec(b"chr1", b"10", b"GT", b"0|1") + _rec(b"chr1", b"20") + _rec(b"chr1", b"30", b"GT", b"1|1")
    pos = _vcf_sites(vcf, NAMES, LENS)
    rc, _ = _check(lib, tmp_path, vcf, NAMES, LENS, pos, [1, 0, 2], [0.5, 0.5, 0.5])
    assert rc == 0
    rc, msg = _check(lib, tmp_path, vcf, NAMES, LENS, pos, [1, 3, 2], [0.5, 0.5, 0.5])
    assert rc != 0 and "fewer columns" in msg
