"""Python harness over the C ABI (tests, bench.py).  The shipped host program is C++ (csrc/host/, binary
`vargeno-b200`, same command line as the reference); this module drives the very same entry points through
ctypes so that parity tests can look at every intermediate (probe results, per-read votes, pileup counters).

Nothing here computes: every method is a call into libvgb200.so.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import VgbError

GT_TEXT = {1: "0/0", 3: "0/1", 2: "1/1"}     # src/qv.cc:1678-1680


class Genotyper:
    """One context = one GPU (vgb_ctx).  Mirrors the life cycle of the reference's genotype() (src/qv.cc:475):
    load index -> walk FASTQ -> call every SNP site."""

    def __init__(self, device: int = 0, trace: bool = False, max_chunk_bytes: int = 64 << 20, world_size: int = 1,
                 rank: int = 0, nccl_unique_id: Optional[bytes] = None):
        self.L = _lib.load()
        self._uid = C.create_string_buffer(nccl_unique_id, 128) if nccl_unique_id else None
        cfg = _lib.Config(device, world_size, rank, _lib.VGB_CFG_TRACE if trace else 0,
                          C.cast(self._uid, C.c_void_p) if self._uid else None, max_chunk_bytes)
        h = C.c_void_p()
        rc = self.L.vgb_ctx_create(C.byref(h), C.byref(cfg))
        if rc:
            raise VgbError(rc, self.L.vgb_last_error(None).decode())
        self.h = h
        self.max_chunk_bytes = max_chunk_bytes
        self.n_sites = 0
        self._keep = []

    # ---- plumbing ----
    def _ck(self, rc):
        if rc:
            raise VgbError(rc, self.L.vgb_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.vgb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @staticmethod
    def nccl_unique_id() -> bytes:
        L = _lib.load()
        buf = C.create_string_buffer(128)
        rc = L.vgb_nccl_unique_id(buf)
        if rc:
            raise VgbError(rc, L.vgb_last_error(None).decode())
        return buf.raw

    # ---- index ----
    def upload_index(self, ix) -> None:
        """ix: vargeno_b200.tools.index_builder.Index (arrays in the on-disk record layouts)."""
        ref = np.ascontiguousarray(ix.ref).view(np.uint8)
        ref_aux = np.ascontiguousarray(ix.ref_aux, dtype="<u4")
        snp = np.ascontiguousarray(ix.snp).view(np.uint8)
        snp_aux = np.ascontiguousarray(ix.snp_aux).view(np.uint8)
        rbf = np.ascontiguousarray(ix.ref_bf, dtype="<u8")
        sbf = np.ascontiguousarray(ix.snp_bf, dtype="<u8")
        v = _lib.IndexView(_lib.ptr(ref), ix.ref.size, _lib.ptr(ref_aux), ix.ref_aux.shape[0],
                           _lib.ptr(snp), ix.snp.size, _lib.ptr(snp_aux), ix.snp_aux.size,
                           _lib.ptr(rbf), ix.ref_bf_bits, rbf.size, _lib.ptr(sbf), ix.snp_bf_bits, sbf.size)
        self._ck(self.L.vgb_index_upload(self.h, C.byref(v)))
        n = C.c_uint64()
        self._ck(self.L.vgb_site_count(self.h, C.byref(n)))
        self.n_sites = n.value
        self.chr_names, self.chr_lens = list(ix.chr_names), list(ix.chr_lens)

    def sites(self) -> Dict[str, np.ndarray]:
        n = self.n_sites
        pos, code, rf, af = np.zeros(n, "<u4"), np.zeros(n, "u1"), np.zeros(n, "u1"), np.zeros(n, "u1")
        self._ck(self.L.vgb_fetch_sites(self.h, _lib.ptr(pos), _lib.ptr(code), _lib.ptr(rf), _lib.ptr(af), n))
        return {"pos": pos, "ref": code & 3, "alt": code >> 2, "ref_freq": rf, "alt_freq": af}

    # ---- reads ----
    @staticmethod
    def split_records(text: np.ndarray, max_bytes: int) -> List[Tuple[int, int, int]]:
        """[(start, end, n_records)] chunks that begin and end at record boundaries (4 lines per record)."""
        nl = np.flatnonzero(text == 10)
        n_lines = nl.size + (1 if text.size and text[-1] != 10 else 0)
        ends = np.concatenate([nl + 1, [text.size]]) if n_lines > nl.size else nl + 1   # end offset of each line
        rec_end = ends[3::4]
        out, start, first = [], 0, 0
        while start < text.size:
            k = int(np.searchsorted(rec_end, start + max_bytes, side="right"))
            if k == first:
                if first >= rec_end.size:              # trailing partial record: hand it over, the library rejects it
                    out.append((start, text.size, 0))
                    break
                k = first + 1                          # a single record larger than the chunk: let the library say so
            end = int(rec_end[k - 1])
            out.append((start, end, k - first))
            start, first = end, k
            if first >= rec_end.size and start < text.size:
                out.append((start, text.size, 0))
                break
        return out

    def submit(self, text, first_read_id: int = 0) -> None:
        """FASTQ text from host memory (bytes or uint8 array), chunked at record boundaries."""
        buf = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else text
        rid = first_read_id
        for s, e, n in self.split_records(buf, self.max_chunk_bytes):
            piece = np.ascontiguousarray(buf[s:e])
            self._ck(self.L.vgb_submit_fastq(self.h, _lib.ptr(piece), piece.size, rid))
            rid += n

    def submit_chunk(self, chunk: np.ndarray, first_read_id: int = 0) -> None:
        """One vgb_submit_fastq call on a buffer that already starts and ends at record boundaries (no host parsing)."""
        self._ck(self.L.vgb_submit_fastq(self.h, _lib.ptr(chunk), chunk.size, first_read_id))

    def pinned_buffer(self, slot: int) -> np.ndarray:
        p, cap = C.c_void_p(), C.c_uint64()
        self._ck(self.L.vgb_pinned_buffer(self.h, slot, C.byref(p), C.byref(cap)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(cap.value,))

    def submit_pinned(self, slot: int, nbytes: int, first_read_id: int = 0) -> None:
        p, cap = C.c_void_p(), C.c_uint64()
        self._ck(self.L.vgb_pinned_buffer(self.h, slot, C.byref(p), C.byref(cap)))
        self._ck(self.L.vgb_submit_fastq(self.h, p, nbytes, first_read_id))

    def submit_bgzf(self, comp: np.ndarray, members: np.ndarray, overlap_bytes: int, last_chunk: bool) -> None:
        """One vgb_submit_bgzf call: `comp` = gzip members back to back (uint8), `members` = uint32[n][3] rows of
        (DEFLATE payload offset in comp, payload length, ISIZE); see tools/bgzf.chunk_arrays."""
        comp = np.ascontiguousarray(comp, dtype=np.uint8)
        members = np.ascontiguousarray(members, dtype="<u4")
        self._ck(self.L.vgb_submit_bgzf(self.h, _lib.ptr(comp), comp.size, _lib.ptr(members), members.shape[0], overlap_bytes, 1 if last_chunk else 0))

    def submit_bgzf_file(self, buf: bytes, own_out: int) -> int:
        """A whole BGZF file image through vgb_submit_bgzf in chunks of about `own_out` inflated bytes, planned the way the C++ host
        plans them (overlap of >= 8 KiB of text from the previous chunk).  Returns the number of chunks."""
        from .tools import bgzf
        mem, plan = bgzf.plan_chunks(bgzf.scan(buf), own_out)
        for k, (o0, i0, i1, ov) in enumerate(plan):
            comp, tab = bgzf.chunk_arrays(buf, mem, o0, i1)
            self.submit_bgzf(comp, tab, ov, k + 1 == len(plan))
        return len(plan)

    def submit_gzip(self, buf, piece_bytes: int, first: bool = True, last: bool = True) -> int:
        """A single-stream gzip image (bytes or uint8 array: one or more gzip members) through vgb_submit_gzip in pieces of
        `piece_bytes` compressed bytes; `first` / `last` mark the first and the last piece as a new stream and the end of the input.
        Returns the number of calls."""
        a = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, dtype=np.uint8)
        step = max(1, min(int(piece_bytes), self.max_chunk_bytes))
        starts = list(range(0, a.size, step)) or [0]
        for i, s in enumerate(starts):
            piece = np.ascontiguousarray(a[s:s + step])
            self._ck(self.L.vgb_submit_gzip(self.h, _lib.ptr(piece), piece.size, 1 if first and i == 0 else 0,
                                            1 if last and i + 1 == len(starts) else 0))
        return len(starts)

    def bam_calls(self, buf, own_out: int) -> List[Tuple[np.ndarray, np.ndarray]]:
        """(compressed members back to back, their vgb_bgzf_member table) of each vgb_submit_bam call of a BAM file image: runs of
        whole BGZF members with at most `own_out` inflated and max_chunk_bytes compressed bytes (tools/bgzf.scan finds them)"""
        from .tools import bgzf
        a = bytes(buf) if isinstance(buf, np.ndarray) else buf
        mem = [m for m in bgzf.scan(a) if m[3]]
        own = max(1, min(int(own_out), self.max_chunk_bytes))
        calls, i = [], 0
        while i < len(mem):
            i0, out, comp = i, 0, 0
            while i < len(mem) and out + mem[i][3] <= own and comp + mem[i][1] <= self.max_chunk_bytes:
                out += mem[i][3]
                comp += mem[i][1]
                i += 1
            if i == i0:
                raise ValueError("a BGZF member does not fit one call")
            calls.append(bgzf.chunk_arrays(a, mem, i0, i))
        return calls or [(np.zeros(0, np.uint8), np.zeros((0, 3), "<u4"))]

    def submit_bam_call(self, comp: np.ndarray, members: np.ndarray, first: bool, last: bool) -> None:
        """One vgb_submit_bam call (see bam_calls)"""
        self._ck(self.L.vgb_submit_bam(self.h, _lib.ptr(comp), comp.size, _lib.ptr(members), members.shape[0], 1 if first else 0, 1 if last else 0))

    def submit_bam(self, buf, own_out: int, first: bool = True, last: bool = True) -> int:
        """A BAM file image (bytes or uint8 array) through vgb_submit_bam in calls of whole BGZF members (bam_calls); `first` /
        `last` mark the file's first and last call.  Returns the number of calls."""
        calls = self.bam_calls(buf, own_out)
        for k, (comp, tab) in enumerate(calls):
            self.submit_bam_call(np.ascontiguousarray(comp), np.ascontiguousarray(tab, dtype="<u4"), first and k == 0, last and k + 1 == len(calls))
        return len(calls)

    def submit_device(self, dptr: int, nbytes: int, first_read_id: int = 0) -> None:
        self._ck(self.L.vgb_submit_fastq_device(self.h, C.c_void_p(dptr), nbytes, first_read_id))

    def sync(self) -> None:
        self._ck(self.L.vgb_sync(self.h))

    def reset(self) -> None:
        self._ck(self.L.vgb_reset_counts(self.h))

    def reset_sample(self) -> None:
        """vgb_reset_sample: end the current sample (counters, statistics, trace, and any unfinished gzip or BAM input) and keep
        the index, so that the next sample is genotyped as if it were the first"""
        self._ck(self.L.vgb_reset_sample(self.h))

    def read_results(self) -> np.ndarray:
        n = C.c_uint64()
        self._ck(self.L.vgb_fetch_read_results(self.h, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=_lib.READ_RESULT)
        self._ck(self.L.vgb_fetch_read_results(self.h, _lib.ptr(out), out.size, C.byref(n)))
        return out

    def stats(self) -> Dict[str, float]:
        s = np.zeros(1, dtype=_lib.STATS)
        self._ck(self.L.vgb_get_stats(self.h, _lib.ptr(s)))
        return {k: (float(s[k][0]) if k.startswith("gpu_ms") else int(s[k][0])) for k in _lib.STATS.names}

    # ---- probes ----
    def lookup(self, kmers: np.ndarray) -> np.ndarray:
        k = np.ascontiguousarray(kmers, dtype="<u8")
        out = np.zeros(k.size, dtype=_lib.HIT)
        self._ck(self.L.vgb_lookup_kmers(self.h, _lib.ptr(k), k.size, _lib.ptr(out)))
        return out

    def probe_bench(self, n: int, mode: int, seed: int = 1, repeats: int = 5) -> Tuple[float, int]:
        ms, found = C.c_double(), C.c_uint64()
        self._ck(self.L.vgb_probe_bench(self.h, n, mode, seed, repeats, C.byref(ms), C.byref(found)))
        return ms.value, found.value

    def random_sector_bench(self, nbytes: int, n_loads: int, repeats: int = 3) -> float:
        g = C.c_double()
        self._ck(self.L.vgb_random_sector_bench(self.h, nbytes, n_loads, repeats, C.byref(g)))
        return g.value

    # ---- pileup + calls ----
    def allreduce(self) -> None:
        self._ck(self.L.vgb_allreduce_pileup(self.h))

    def pileup(self) -> Tuple[np.ndarray, np.ndarray]:
        r, a = np.zeros(self.n_sites, "<u4"), np.zeros(self.n_sites, "<u4")
        self._ck(self.L.vgb_fetch_pileup(self.h, _lib.ptr(r), _lib.ptr(a), self.n_sites))
        return r, a

    def call(self, out: Optional[Tuple[np.ndarray, np.ndarray]] = None) -> Tuple[np.ndarray, np.ndarray]:
        """GT code + confidence per site.  `out`: caller-owned (e.g. pinned) uint8 / float64 arrays of n_sites elements."""
        g, c = out if out is not None else (np.zeros(self.n_sites, "u1"), np.zeros(self.n_sites, "<f8"))
        assert g.dtype == np.uint8 and c.dtype == np.float64 and g.size == self.n_sites and c.size == self.n_sites
        self._ck(self.L.vgb_call(self.h, _lib.ptr(g), _lib.ptr(c), self.n_sites))
        return g, c

    # ---- output VCF ----
    def vcf_template(self, vcf: bytes) -> None:
        """vgb_vcf_template: the input SNP VCF (its bytes) as the output template of this context; needs the index"""
        names = (C.c_char_p * len(self.chr_names))(*[n.encode() for n in self.chr_names])
        lens = np.ascontiguousarray(self.chr_lens, dtype="<u8")
        buf = np.frombuffer(vcf, dtype=np.uint8) if len(vcf) else np.zeros(1, np.uint8)
        self._ck(self.L.vgb_vcf_template(self.h, _lib.ptr(buf), len(vcf), names, _lib.ptr(lens), len(self.chr_names)))

    def vcf_template_copy(self, src: "Genotyper") -> None:
        self._ck(self.L.vgb_vcf_template_copy(self.h, src.h))

    @staticmethod
    def _collector():
        parts = []

        def fn(user, p, n):
            parts.append(C.string_at(p, n))
            return 0
        return parts, _lib.WRITE_FN(fn)

    def vcf_write(self, gt: np.ndarray, gq: np.ndarray, bgzf: bool = False) -> bytes:
        """vgb_vcf_write: this sample's VCF (BGZF with bgzf) from gtype and GQ per site (gq() of each called site's confidence)"""
        gt = np.ascontiguousarray(gt, dtype=np.uint8)
        gq = np.ascontiguousarray(gq, dtype="<i4")
        assert gt.size == self.n_sites and gq.size == self.n_sites
        parts, fn = self._collector()
        self._ck(self.L.vgb_vcf_write(self.h, _lib.ptr(gt), _lib.ptr(gq), self.n_sites, int(bgzf), fn, None, None))
        return b"".join(parts)

    def deflate_bgzf(self, text, eof: bool = True) -> bytes:
        """vgb_deflate_bgzf: BGZF members of host bytes, or of device memory given as (pointer, bytes)"""
        parts, fn = self._collector()
        if isinstance(text, tuple):
            self._ck(self.L.vgb_deflate_bgzf(self.h, C.c_void_p(text[0]), text[1], 1, int(eof), fn, None))
        else:
            a = np.frombuffer(bytes(text), dtype=np.uint8) if len(text) else np.zeros(1, np.uint8)
            self._ck(self.L.vgb_deflate_bgzf(self.h, _lib.ptr(a), len(text), 0, int(eof), fn, None))
        return b"".join(parts)

    def counter_device_ptr(self) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self.L.vgb_counter_device_ptr(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    # ---- device memory helpers for the bench ----
    def dalloc(self, nbytes: int) -> int:
        p = self.L.vgb_device_alloc(self.h, nbytes)
        if not p:
            raise VgbError(_lib.VGB_E_CUDA, self.L.vgb_last_error(self.h).decode())
        return p

    def dfree(self, p: int) -> None:
        self.L.vgb_device_free(self.h, C.c_void_p(p))

    def h2d(self, dptr: int, a: np.ndarray) -> None:
        a = np.ascontiguousarray(a)
        self._ck(self.L.vgb_memcpy_h2d(self.h, C.c_void_p(dptr), _lib.ptr(a), a.nbytes))

    def d2h(self, dptr: int, nbytes: int) -> np.ndarray:
        out = np.empty(nbytes, dtype=np.uint8)
        self._ck(self.L.vgb_memcpy_d2h(self.h, _lib.ptr(out), C.c_void_p(dptr), nbytes))
        return out

    def synth_reads_device(self, hap0_d: int, hap1_d: int, genome_len: int, contig_starts, contig_lens, n_reads: int,
                           read_len: int, seed: int, first_id: int, id_width: int, sub_rate: float, lowq_prob: float,
                           lowq_chars: int, out_d: int, out_cap: int) -> None:
        cs = np.ascontiguousarray(contig_starts, dtype="<u8")
        cl = np.ascontiguousarray(contig_lens, dtype="<u8")
        self._ck(self.L.vgb_synth_reads_device(self.h, C.c_void_p(hap0_d), C.c_void_p(hap1_d), genome_len, _lib.ptr(cs), _lib.ptr(cl),
                                               cs.size, n_reads, read_len, seed, first_id, id_width, sub_rate, lowq_prob,
                                               lowq_chars, C.c_void_p(out_d), out_cap))


class DeviceIndex:
    """Index records built in HBM by vgb_build_index_device (device pointers in the on-disk layouts)."""

    def __init__(self, g: Genotyper, view: "_lib.IndexView", chr_names, chr_lens):
        self.g, self.view, self.chr_names, self.chr_lens = g, view, list(chr_names), list(chr_lens)

    def free(self):
        if self.view is not None:
            self.g.L.vgb_free_index_device(self.g.h, C.byref(self.view))
            self.view = None

    def to_host(self):
        """Copy the records back: a tools.index_builder.Index, byte-identical to what `vargeno index` writes."""
        from .tools import index_builder as ib
        v, g = self.view, self.g
        ref = g.d2h(v.ref_records, 13 * v.n_ref).view(ib.REF_REC) if v.n_ref else np.zeros(0, ib.REF_REC)
        ref_aux = g.d2h(v.ref_aux, 40 * v.n_ref_aux).view("<u4").reshape(-1, 10) if v.n_ref_aux else np.zeros((0, 10), "<u4")
        snp = g.d2h(v.snp_records, 16 * v.n_snp).view(ib.SNP_REC) if v.n_snp else np.zeros(0, ib.SNP_REC)
        snp_aux = g.d2h(v.snp_aux, 78 * v.n_snp_aux).view(ib.SNP_AUX_REC) if v.n_snp_aux else np.zeros(0, ib.SNP_AUX_REC)
        rbf = g.d2h(v.ref_bf_words, 8 * v.ref_bf_nwords).view("<u8")
        sbf = g.d2h(v.snp_bf_words, 8 * v.snp_bf_nwords).view("<u8")
        return ib.Index(ref, ref_aux, snp, snp_aux, v.ref_bf_bits, rbf, v.snp_bf_bits, sbf, self.chr_names, self.chr_lens)


def build_index_device(g: Genotyper, genome_d: int, contig_names, contig_starts, contig_lens, snp_pos0, snp_ref_code, snp_alt_code,
                       snp_ref_freq, snp_alt_freq, bf_pos0) -> DeviceIndex:
    """vgb_build_index_device.  snp_*: the VCF lines that pass the dictionary-side filters (src/dictgen.c:599-748), file order,
    positions 0-based in the concatenation; bf_pos0: the lines that pass the Bloom-filter-side filters (src/generate_bf.cc:224-241)."""
    cs = np.ascontiguousarray(contig_starts, dtype="<u8")
    cl = np.ascontiguousarray(contig_lens, dtype="<u8")
    p0 = np.ascontiguousarray(snp_pos0, dtype="<u4")
    code = np.ascontiguousarray((np.asarray(snp_ref_code, np.uint8) & 3) | (np.asarray(snp_alt_code, np.uint8) << 2), dtype="u1")
    rf = np.ascontiguousarray(snp_ref_freq, dtype="u1")
    af = np.ascontiguousarray(snp_alt_freq, dtype="u1")
    bp = np.ascontiguousarray(bf_pos0, dtype="<u4")
    view = _lib.IndexView()
    g._ck(g.L.vgb_build_index_device(g.h, C.c_void_p(genome_d), int(cs[-1] + cl[-1]), _lib.ptr(cs), _lib.ptr(cl), cs.size, _lib.ptr(p0),
                                     _lib.ptr(code), _lib.ptr(rf), _lib.ptr(af), p0.size, _lib.ptr(bp), bp.size, C.byref(view)))
    return DeviceIndex(g, view, contig_names, [int(x) for x in cl])


def upload_device_index(g: Genotyper, dix: DeviceIndex) -> None:
    g._ck(g.L.vgb_index_upload_device(g.h, C.byref(dix.view)))
    n = C.c_uint64()
    g._ck(g.L.vgb_site_count(g.h, C.byref(n)))
    g.n_sites = n.value
    g.chr_names, g.chr_lens = list(dix.chr_names), list(dix.chr_lens)


def synth_genome_device(g: Genotyper, out_d: int, contig_starts, contig_lens, seed: int) -> None:
    cs = np.ascontiguousarray(contig_starts, dtype="<u8")
    cl = np.ascontiguousarray(contig_lens, dtype="<u8")
    g._ck(g.L.vgb_synth_genome_device(g.h, C.c_void_p(out_d), _lib.ptr(cs), _lib.ptr(cl), cs.size, seed))


def gq(conf: float) -> int:
    """(int)(-1*10*log(conf)), src/qv.cc:1681 -- CPython's math.log is the C library's log."""
    return int(-10.0 * math.log(conf))


def site_gq(gt: np.ndarray, conf: np.ndarray) -> np.ndarray:
    """GQ per site for vgb_vcf_write: gq() of every called site, 0 for the others"""
    out = np.zeros(gt.size, dtype="<i4")
    for i in np.flatnonzero(gt):
        out[i] = gq(float(conf[i]))
    return out
