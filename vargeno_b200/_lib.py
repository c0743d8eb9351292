"""ctypes binding of libvgb200.so (include/vgb200.h).  Fails loudly when the library is missing: there is no
Python / CPU fallback for any compute entry point."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# VGB200_LIB: A/B measurements of two builds of the same library (tools/perf_sweep.py); never a different implementation
LIB_PATH = os.environ.get("VGB200_LIB") or os.path.join(HERE, "libvgb200.so")

VGB_OK, VGB_E_ARG, VGB_E_CUDA, VGB_E_FORMAT, VGB_E_INDEX, VGB_E_NCCL, VGB_E_OVERFLOW = 0, -1, -2, -3, -4, -5, -6
VGB_CFG_TRACE = 1


class VgbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libvgb200 error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("world_size", C.c_int32), ("rank", C.c_int32), ("flags", C.c_uint32),
                ("nccl_unique_id", C.c_void_p), ("max_chunk_bytes", C.c_uint64)]


class IndexView(C.Structure):
    _fields_ = [("ref_records", C.c_void_p), ("n_ref", C.c_uint64), ("ref_aux", C.c_void_p), ("n_ref_aux", C.c_uint64),
                ("snp_records", C.c_void_p), ("n_snp", C.c_uint64), ("snp_aux", C.c_void_p), ("n_snp_aux", C.c_uint64),
                ("ref_bf_words", C.c_void_p), ("ref_bf_bits", C.c_uint64), ("ref_bf_nwords", C.c_uint64),
                ("snp_bf_words", C.c_void_p), ("snp_bf_bits", C.c_uint64), ("snp_bf_nwords", C.c_uint64)]


HIT = np.dtype([("ref_pos", "<u4"), ("snp_pos", "<u4"), ("ref_block_lo", "<u4"), ("ref_block_n", "<u4"),
                ("snp_block_lo", "<u4"), ("snp_block_n", "<u4"), ("ref_found", "u1"), ("ref_flag", "u1"),
                ("snp_found", "u1"), ("snp_flag", "u1"), ("snp_info", "u1"), ("ref_bf", "u1"), ("snp_bf", "u1"), ("pad", "u1")])
READ_RESULT = np.dtype([("flags", "<u4"), ("target", "<u4"), ("freq", "<u2"), ("n_ref", "<u2"), ("n_snp", "<u2"),
                        ("passes", "<u2"), ("ctx_hash", "<u8")])
STATS = np.dtype([(k, "<u8") for k in ("reads", "skipped_n", "passes", "placed", "exact_lookups", "nbr_query_lookups",
                                       "nbr_scan_reads", "bf_probes", "lowq_kmers", "events", "pileup_incr", "big_kmers",
                                       "bad_records", "chunks", "chunk_bytes")] +
                 [("gpu_ms_parse", "<f8"), ("gpu_ms_geno", "<f8"), ("kernel_launches", "<u8"), ("freq_wrap_reads", "<u8")])
assert HIT.itemsize == 32 and READ_RESULT.itemsize == 24 and STATS.itemsize == 19 * 8

# every symbol include/vgb200.h declares (tests check the library exports all of them)
SYMBOLS = ["vgb_abi_version", "vgb_ctx_create", "vgb_ctx_destroy", "vgb_last_error", "vgb_nccl_unique_id", "vgb_index_upload",
           "vgb_site_count", "vgb_fetch_sites", "vgb_pinned_buffer", "vgb_submit_fastq", "vgb_submit_fastq_device", "vgb_sync",
           "vgb_reset_counts", "vgb_fetch_read_results", "vgb_lookup_kmers", "vgb_allreduce_pileup", "vgb_fetch_pileup",
           "vgb_call", "vgb_counter_device_ptr", "vgb_get_stats", "vgb_probe_bench", "vgb_random_sector_bench",
           "vgb_synth_reads_device", "vgb_device_alloc", "vgb_device_free", "vgb_memcpy_d2h", "vgb_memcpy_h2d",
           "vgb_build_index_device", "vgb_free_index_device", "vgb_index_upload_device", "vgb_synth_genome_device",
           "vgb_memcpy_d2d", "vgb_memset_device", "vgb_comm_init", "vgb_build_ref_lite_bf_device", "vgb_build_snp_bf_ucsc_device", "vgb_submit_bgzf",
           "vgb_submit_gzip", "vgb_submit_bam", "vgb_reset_sample", "vgb_vcf_template", "vgb_vcf_template_copy", "vgb_vcf_write",
           "vgb_deflate_bgzf"]

# int (*vgb_write_fn)(void *user, const void *bytes, uint64_t n)
WRITE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64)

_lib = None


def load():
    """dlopen libvgb200.so; raises if it has not been built (python -m vargeno_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: build it with `python -m vargeno_b200.build` (no CPU fallback exists)" % LIB_PATH)
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, u64, i32, u32 = C.c_void_p, C.c_uint64, C.c_int, C.c_uint32
    sig = {
        "vgb_abi_version": (i32, []),
        "vgb_ctx_create": (i32, [C.POINTER(vp), C.POINTER(Config)]),
        "vgb_ctx_destroy": (None, [vp]),
        "vgb_last_error": (C.c_char_p, [vp]),
        "vgb_nccl_unique_id": (i32, [vp]),
        "vgb_index_upload": (i32, [vp, C.POINTER(IndexView)]),
        "vgb_site_count": (i32, [vp, C.POINTER(u64)]),
        "vgb_fetch_sites": (i32, [vp, vp, vp, vp, vp, u64]),
        "vgb_pinned_buffer": (i32, [vp, i32, C.POINTER(vp), C.POINTER(u64)]),
        "vgb_submit_fastq": (i32, [vp, vp, u64, u64]),
        "vgb_submit_fastq_device": (i32, [vp, vp, u64, u64]),
        "vgb_sync": (i32, [vp]),
        "vgb_reset_counts": (i32, [vp]),
        "vgb_reset_sample": (i32, [vp]),
        "vgb_fetch_read_results": (i32, [vp, vp, u64, C.POINTER(u64)]),
        "vgb_lookup_kmers": (i32, [vp, vp, u64, vp]),
        "vgb_allreduce_pileup": (i32, [vp]),
        "vgb_fetch_pileup": (i32, [vp, vp, vp, u64]),
        "vgb_call": (i32, [vp, vp, vp, u64]),
        "vgb_counter_device_ptr": (i32, [vp, C.POINTER(vp), C.POINTER(u64)]),
        "vgb_get_stats": (i32, [vp, vp]),
        "vgb_probe_bench": (i32, [vp, u64, i32, u64, i32, C.POINTER(C.c_double), C.POINTER(u64)]),
        "vgb_random_sector_bench": (i32, [vp, u64, u64, i32, C.POINTER(C.c_double)]),
        "vgb_synth_reads_device": (i32, [vp, vp, vp, u64, vp, vp, u32, u64, u32, u64, u64, u32, C.c_double, C.c_double, u32, vp, u64]),
        "vgb_device_alloc": (vp, [vp, u64]),
        "vgb_device_free": (None, [vp, vp]),
        "vgb_memcpy_d2h": (i32, [vp, vp, vp, u64]),
        "vgb_memcpy_h2d": (i32, [vp, vp, vp, u64]),
        "vgb_build_index_device": (i32, [vp, vp, u64, vp, vp, u32, vp, vp, vp, vp, u64, vp, u64, C.POINTER(IndexView)]),
        "vgb_free_index_device": (None, [vp, C.POINTER(IndexView)]),
        "vgb_index_upload_device": (i32, [vp, C.POINTER(IndexView)]),
        "vgb_synth_genome_device": (i32, [vp, vp, vp, vp, u32, u64]),
        "vgb_memcpy_d2d": (i32, [vp, vp, vp, u64]),
        "vgb_memset_device": (i32, [vp, vp, i32, u64]),
        "vgb_comm_init": (i32, [vp, i32, i32, vp]),
        "vgb_build_snp_bf_ucsc_device": (i32, [vp, vp, vp, vp, u64, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]),
        "vgb_submit_bgzf": (i32, [vp, vp, u64, vp, u32, u64, i32]),
        "vgb_submit_gzip": (i32, [vp, vp, u64, i32, i32]),
        "vgb_submit_bam": (i32, [vp, vp, u64, vp, u32, i32, i32]),
        "vgb_build_ref_lite_bf_device": (i32, [vp, vp, vp, vp, u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]),
        "vgb_vcf_template": (i32, [vp, vp, u64, C.POINTER(C.c_char_p), vp, u32]),
        "vgb_vcf_template_copy": (i32, [vp, vp]),
        "vgb_vcf_write": (i32, [vp, vp, vp, u64, i32, WRITE_FN, vp, C.POINTER(u64)]),
        "vgb_deflate_bgzf": (i32, [vp, vp, u64, i32, i32, WRITE_FN, vp]),
    }
    for name in SYMBOLS:
        fn = getattr(L, name)           # AttributeError if the library does not export what the header declares
        fn.restype, fn.argtypes = sig[name]
    if L.vgb_abi_version() != 2:
        raise ImportError("libvgb200.so ABI version mismatch")
    _lib = L
    return L


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
