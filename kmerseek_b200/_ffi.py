"""ctypes binding of include/kmerseek_b200.h -- the same seam a Rust `extern "C"` block would bind.

The library is built in-tree (kmerseek_b200/build.py -> kmerseek_b200/libkmerseek_b200.so).  There is
no fallback: if the shared object is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KS_LIB_PATH") or os.path.join(_HERE, "libkmerseek_b200.so")  # (override: kernel experiments)

u8p, u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_double))

KS_OK = 0
STATUS_NAMES = {
    0: "KS_OK", 1: "KS_ERR_INVALID_MOLTYPE", 2: "KS_ERR_INVALID_AMINO_ACID", 3: "KS_ERR_INVALID_KSIZE",
    4: "KS_ERR_NO_SAVED_STATE", 5: "KS_ERR_IO", 6: "KS_ERR_UTF8", 7: "KS_ERR_PARSE", 8: "KS_ERR_BUILDER",
    9: "KS_ERR_VALIDATION", 10: "KS_ERR_NOT_FINALIZED", 100: "KS_ERR_CUDA", 101: "KS_ERR_NCCL",
    102: "KS_ERR_OUT_OF_MEMORY", 103: "KS_ERR_NO_DEVICE", 104: "KS_ERR_CAPACITY",
}
KS_SEARCH_HITS = 1
KS_SEARCH_DEVICE_ONLY = 2
KS_SEARCH_QUERY_SKETCHES = 4
KS_COMM_ID_BYTES = 128
KS_NORMALIZE_KMERSEEK = 0
KS_NORMALIZE_SOURMASH = 1


class ks_params(C.Structure):
    _fields_ = [("ksize", C.c_uint32), ("scaled", C.c_uint32), ("moltype", C.c_int32),
                ("store_raw_sequences", C.c_int32), ("device", C.c_int32), ("reserved", C.c_uint32)]


class ks_stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_proteins", "n_residues", "n_windows", "n_tuples", "n_unique_hashes", "n_groups", "n_distinct_ids",
        "device_bytes", "sketch_launches", "sort_launches", "csr_launches", "search_launches")] + [
        (n, C.c_float) for n in ("ms_upload", "ms_sketch", "ms_sort", "ms_csr", "ms_search", "ms_sort_partition",
                                 "ms_sort_bucket")] + [
        ("finalized", C.c_uint32), ("build_path", C.c_uint32)]


class ks_sketch(C.Structure):
    _fields_ = [("n_proteins", C.c_uint64), ("n_tuples", C.c_uint64), ("hash", u64p), ("pid", u32p), ("pos", u32p),
                ("sig_ptr", u64p), ("mins", u64p), ("abunds", u64p)]


class ks_csr(C.Structure):
    _fields_ = [("n_keys", C.c_uint64), ("n_postings", C.c_uint64), ("keys", u64p), ("row_ptr", u64p),
                ("pid", u32p), ("pos", u32p)]


SCORE_COLUMNS = ["containment", "containment_target_in_query", "max_containment", "jaccard",
                 "query_containment_ani", "match_containment_ani", "average_containment_ani", "max_containment_ani",
                 "average_abund", "median_abund", "std_abund", "f_weighted_target_in_query"]


class ks_search_result(C.Structure):
    _fields_ = ([("n_queries", C.c_uint64), ("q_sig_ptr", u64p), ("q_mins", u64p), ("q_abunds", u64p),
                 ("n_pairs", C.c_uint64), ("pair_qid", u32p), ("pair_pid", u32p), ("intersect_hashes", u32p),
                 ("q_size", u32p), ("t_size", u32p), ("n_weighted_found", u64p), ("total_weighted_hashes", u64p)] +
                [(n, f64p) for n in SCORE_COLUMNS] +
                [("n_hits", C.c_uint64), ("hit_qid", u32p), ("hit_pid", u32p), ("hit_qpos", u32p), ("hit_tpos", u32p),
                 ("hit_hash", u64p), ("device_block", C.c_void_p), ("ms_device", C.c_float)])


# name -> (restype, argtypes); every symbol include/kmerseek_b200.h declares
SIGNATURES = {
    "ks_last_error_message": (C.c_char_p, []),
    "ks_last_error_detail": (None, [u32p, u64p, u64p]),
    "ks_abi_version": (C.c_int, []),
    "ks_device_count": (C.c_int, []),
    "ks_moltype_from_str": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
    "ks_moltype_name": (C.c_char_p, [C.c_int]),
    "ks_max_hash": (C.c_uint64, [C.c_uint32]),
    "ks_translate_residue": (C.c_uint8, [C.c_uint8, C.c_int]),
    "ks_md5_of_mins": (None, [u64p, C.c_uint64, C.c_uint32, C.c_char_p]),
    "ks_id_of_mins": (None, [u64p, C.c_uint64, C.c_char_p]),
    "ks_proteome_from_fasta": (C.c_int, [C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "ks_proteome_from_sequences": (C.c_int, [C.POINTER(C.c_char_p), u64p, C.POINTER(C.c_char_p), C.c_uint64,
                                             C.c_uint64, C.POINTER(C.c_void_p)]),
    "ks_proteome_from_fasta_mode": (C.c_int, [C.c_char_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    "ks_proteome_from_sequences_mode": (C.c_int, [C.POINTER(C.c_char_p), u64p, C.POINTER(C.c_char_p), C.c_uint64,
                                                  C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    "ks_proteome_from_packed": (C.c_int, [u8p, u64p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "ks_proteome_n_proteins": (C.c_uint64, [C.c_void_p]),
    "ks_proteome_n_residues": (C.c_uint64, [C.c_void_p]),
    "ks_proteome_residues": (u8p, [C.c_void_p]),
    "ks_proteome_offsets": (u64p, [C.c_void_p]),
    "ks_proteome_packed": (u8p, [C.c_void_p, u64p]),
    "ks_proteome_name": (C.c_char_p, [C.c_void_p, C.c_uint64]),
    "ks_proteome_free": (None, [C.c_void_p]),
    "ks_index_create": (C.c_int, [C.POINTER(ks_params), C.POINTER(C.c_void_p)]),
    "ks_index_destroy": (None, [C.c_void_p]),
    "ks_index_params": (C.c_int, [C.c_void_p, C.POINTER(ks_params)]),
    "ks_index_stream": (C.c_void_p, [C.c_void_p]),
    "ks_index_sync": (C.c_int, [C.c_void_p]),
    "ks_index_upload": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ks_index_sketch_resident": (C.c_int, [C.c_void_p]),
    "ks_index_add_proteome": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ks_index_finalize": (C.c_int, [C.c_void_p]),
    "ks_index_clear": (C.c_int, [C.c_void_p]),
    "ks_index_process_fasta": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "ks_index_add_tuples": (C.c_int, [C.c_void_p, u64p, u32p, u32p, C.c_uint64, C.c_uint64]),
    "ks_index_append_proteome": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ks_index_append_tuples": (C.c_int, [C.c_void_p, u64p, u32p, u32p, C.c_uint64, C.c_uint64]),
    "ks_index_stats": (C.c_int, [C.c_void_p, C.POINTER(ks_stats)]),
    "ks_index_signature_count": (C.c_int, [C.c_void_p, u64p]),
    "ks_sketch_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.POINTER(ks_sketch))]),
    "ks_sketch_free": (None, [C.POINTER(ks_sketch)]),
    "ks_index_export": (C.c_int, [C.c_void_p, C.POINTER(C.POINTER(ks_sketch))]),
    "ks_index_csr": (C.c_int, [C.c_void_p, C.POINTER(C.POINTER(ks_csr))]),
    "ks_csr_free": (None, [C.POINTER(ks_csr)]),
    "ks_search_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.POINTER(ks_search_result))]),
    "ks_search_result_free": (None, [C.POINTER(ks_search_result)]),
    "ks_search_result_device_column": (C.c_void_p, [C.POINTER(ks_search_result), C.c_char_p]),
    "ks_query_upload": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ks_search_resident": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.POINTER(ks_search_result))]),
    "ks_comm_unique_id": (C.c_int, [u8p]),
    "ks_comm_create": (C.c_int, [u8p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "ks_comm_destroy": (None, [C.c_void_p]),
    "ks_comm_rank": (C.c_int, [C.c_void_p]),
    "ks_comm_world": (C.c_int, [C.c_void_p]),
    "ks_shard_search_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64,
                                        C.POINTER(C.POINTER(ks_search_result))]),
}

_lib = None


def lib():
    """Load libkmerseek_b200.so.  Raises (loudly) when it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m kmerseek_b200.build` "
                "(nvcc, sm_100a). kmerseek_b200 has no CPU or pure-Python fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
