"""ctypes binding of libkmerscuda.so -- exactly the symbols include/kmerscuda.h declares.

This is the same binding a Julia `ccall` stub makes (see INTEGRATION.md); there is no CPU
fallback: if the shared library is missing the import fails, and if no CUDA device is present
every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# the in-tree build; KMERSCUDA_LIB selects another build of the same library (A/B measurements)
LIB_PATH = os.environ.get("KMERSCUDA_LIB") or os.path.join(os.path.dirname(_HERE), "libkmerscuda.so")

KMC_OK = 0
KMC_E_BAD_K = 1
KMC_E_BAD_ARG = 2
KMC_E_AMBIGUOUS = 3
KMC_E_OUT_TOO_SMALL = 4
KMC_E_NO_DEVICE = 5
KMC_E_UNSUPPORTED = 6
KMC_E_NCCL = 7
KMC_COMM_ID_BYTES = 128

KMC_FW, KMC_FWRV, KMC_CANON, KMC_UNAMBIG = 0, 1, 2, 3
KMC_HASH_FX, KMC_AOS, KMC_NO_SYNC, KMC_OUT_DEVICE, KMC_DIGEST, KMC_RNA = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
KMC_KMER4 = 0x40
KMC_MAX_K = 128
KMC_MAX_K4 = 64


class kmc_seqs(C.Structure):
    _fields_ = [
        ("words", C.c_void_p),
        ("n_words", C.c_uint64),
        ("n_seqs", C.c_uint64),
        ("seq_word_offset", C.c_void_p),
        ("seq_len", C.c_void_p),
        ("uniform_len", C.c_uint64),
        ("uniform_stride_words", C.c_uint64),
        ("src_bits", C.c_uint32),
        ("first_symbol_offset", C.c_uint32),
    ]


class kmc_out(C.Structure):
    _fields_ = [
        ("a", C.c_void_p),
        ("b", C.c_void_p),
        ("hash", C.c_void_p),
        ("index", C.c_void_p),
        ("seq_out_offset", C.c_void_p),
        ("capacity", C.c_uint64),
        ("index_base", C.c_int64),
    ]


class kmc_result(C.Structure):
    _fields_ = [
        ("n_written", C.c_uint64),
        ("err_seq", C.c_uint64),
        ("err_pos", C.c_uint64),
        ("err_sym", C.c_uint32),
        ("kernel_ms", C.c_float),
        ("digest", C.c_uint64 * 4),
    ]


# name -> (restype, argtypes); must list every function of include/kmerscuda.h
SIGNATURES = {
    "kmc_version": (C.c_int32, []),
    "kmc_device_count": (C.c_int32, [C.POINTER(C.c_int32)]),
    "kmc_ctx_create": (C.c_int32, [C.c_int32, C.POINTER(C.c_void_p)]),
    "kmc_ctx_destroy": (C.c_int32, [C.c_void_p]),
    "kmc_ctx_set_stream": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "kmc_sync": (C.c_int32, [C.c_void_p]),
    "kmc_trim": (C.c_int32, [C.c_void_p]),
    "kmc_last_error": (C.c_char_p, [C.c_void_p]),
    "kmc_status_string": (C.c_char_p, [C.c_int32]),
    "kmc_device_info": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_uint64), C.c_char_p, C.c_int32]),
    "kmc_malloc": (C.c_int32, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "kmc_free": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "kmc_memset": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64]),
    "kmc_upload": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "kmc_download": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "kmc_host_alloc": (C.c_int32, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "kmc_host_free": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "kmc_host_register": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "kmc_host_unregister": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "kmc_count": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
    "kmc_extract": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint32,
                                C.POINTER(kmc_out), C.POINTER(kmc_result)]),
    "kmc_extract_host": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint32,
                                     C.POINTER(kmc_out), C.POINTER(kmc_result)]),
    "kmc_extract_spaced": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint32, C.POINTER(kmc_out),
                                       C.POINTER(kmc_result)]),
    "kmc_fx_hash": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int32, C.c_uint64, C.c_void_p]),
    "kmc_base_hash": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int32, C.c_int32, C.c_uint64, C.c_void_p]),
    "kmc_bucket_count": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p,
                                     C.POINTER(kmc_result)]),
    "kmc_bucket_count_async": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p, C.c_uint32,
                                           C.POINTER(C.c_void_p), C.POINTER(kmc_result)]),
    "kmc_minimizers": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                   C.POINTER(kmc_out), C.POINTER(kmc_result)]),
    "kmc_minhash_sketch": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint64, C.c_void_p,
                                       C.POINTER(kmc_result)]),
    "kmc_minhash_sketch_each": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint64, C.c_void_p,
                                            C.c_void_p, C.POINTER(kmc_result)]),
    "kmc_minhash_compare": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64,
                                        C.c_uint64, C.c_void_p, C.c_void_p]),
    "kmc_composition": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p,
                                    C.POINTER(kmc_result)]),
    "kmc_kmer_count": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint32,
                                   C.POINTER(kmc_result)]),
    "kmc_kmer_table_merge": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                         C.POINTER(C.c_uint64)]),
    "kmc_kmer_table_export": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                          C.POINTER(C.c_uint64)]),
    "kmc_kmer_count2": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint32,
                                    C.POINTER(kmc_result)]),
    "kmc_kmer_table2_merge": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                          C.POINTER(C.c_uint64)]),
    "kmc_kmer_table2_export": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                           C.POINTER(C.c_uint64)]),
    "kmc_kmer_lookup": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint32,
                                    C.c_void_p, C.c_uint64, C.POINTER(kmc_result)]),
    "kmc_kmer_lookup2": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint32,
                                     C.c_void_p, C.c_uint64, C.POINTER(kmc_result)]),
    "kmc_kmer_table_get": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "kmc_kmer_table2_get": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "kmc_kmer_table_histogram": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]),
    "kmc_kmer_table2_histogram": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]),
    "kmc_kmer_table_export_range": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                                C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "kmc_kmer_table2_export_range": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                                 C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "kmc_nccl_version":(C.c_int32, [C.POINTER(C.c_int32)]),
    "kmc_comm_unique_id": (C.c_int32, [C.c_void_p]),
    "kmc_comm_init_rank": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "kmc_comm_destroy": (C.c_int32, [C.c_void_p]),
    "kmc_comm_info": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "kmc_allreduce_u32": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "kmc_allreduce_u64": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "kmc_bucket_count_merge": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_void_p,
                                           C.POINTER(kmc_result)]),
    "kmc_kmer_owner": (C.c_uint32, [C.c_uint64, C.c_uint32]),
    "kmc_kmer_table_exchange": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                            C.POINTER(C.c_uint64)]),
    "kmc_kmer_owner2": (C.c_uint32, [C.c_uint64, C.c_uint64, C.c_uint32]),
    "kmc_kmer_table2_exchange": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                             C.POINTER(C.c_uint64)]),
    "kmc_group_create": (C.c_int32, [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]),
    "kmc_group_destroy": (C.c_int32, [C.c_void_p]),
    "kmc_group_size": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32)]),
    "kmc_group_ctx": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "kmc_group_sync": (C.c_int32, [C.c_void_p]),
    "kmc_group_allreduce_u32": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint64]),
    "kmc_group_allreduce_u64": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint64]),
    "kmc_group_bucket_count": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.POINTER(C.c_void_p),
                                           C.POINTER(kmc_result)]),
    "kmc_group_extract": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint32, C.POINTER(kmc_out),
                                      C.POINTER(kmc_result)]),
    "kmc_group_extract_host": (C.c_int32, [C.c_void_p, C.POINTER(kmc_seqs), C.c_int32, C.c_int32, C.c_uint32, C.POINTER(kmc_out),
                                           C.POINTER(kmc_result)]),
    "kmc_group_kmer_table_exchange": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32,
                                                  C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(C.c_uint64)]),
    "kmc_group_kmer_table2_exchange": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32,
                                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(C.c_uint64)]),
    "kmc_digest": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "kmc_timer_begin": (C.c_int32, [C.c_void_p]),
    "kmc_timer_end": (C.c_int32, [C.c_void_p, C.POINTER(C.c_float)]),
    "kmc_store_probe": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
}

_lib = None


def load():
    """dlopen the in-tree CUDA library.  Raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C kmers.jl_b200/csrc).  There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
