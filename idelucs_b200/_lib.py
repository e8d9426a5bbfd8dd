"""ctypes binding of libidelucs_b200.so (the C ABI declared in include/idelucs_b200.h).

There is NO fallback: if the library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# (IDELUCS_B200_LIB: load a differently built library instead, e.g. to compare two builds with tools/stats_identity.py)
LIB_PATH = os.environ.get("IDELUCS_B200_LIB") or os.path.join(_HERE, "lib", "libidelucs_b200.so")

IDL_OK = 0
KIND_CLEAN, KIND_TRANSITION, KIND_TRANSVERSION, KIND_BOTH, KIND_RANDOM_N, KIND_EXPLICIT = range(6)
OUT_COUNTS_I32, OUT_FREQ_F32, OUT_STD_F32, OUT_FREQ_F64 = range(4)
OUT_CANON_F32, OUT_CANON_STD_F32, OUT_CANON_F64 = 9, 10, 11   # canonical k-mer rows (= 8 + the frequency kind)

c_void_p, c_int, c_i64, c_u64, c_size_t, c_double, c_float = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_size_t, ctypes.c_double, ctypes.c_float)


class Variant(ctypes.Structure):
    """struct idl_variant"""
    _fields_ = [("kind", ctypes.c_int32), ("rng_id", ctypes.c_int32), ("n_bp", ctypes.c_int32),
                ("explicit_idx", ctypes.c_int32), ("p1", c_double), ("p2", c_double)]


# every symbol include/idelucs_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "idl_abi_version": (c_int, []),
    "idl_last_error": (ctypes.c_char_p, []),
    "idl_launch_count": (ctypes.c_longlong, []),
    "idl_geometric_table": (c_int, [c_double, c_void_p]),
    "idl_pack": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "idl_profiles_workspace_bytes": (c_size_t, []),
    "idl_profiles": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int,
                             ctypes.POINTER(Variant), c_int, c_void_p, c_int, c_u64, c_void_p, c_void_p, c_int,
                             c_void_p, ctypes.POINTER(c_i64), c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_size_t, c_void_p]),
    "idl_profile_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, ctypes.POINTER(Variant),
                                  c_u64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, ctypes.POINTER(c_int), c_void_p, c_void_p,
                                  c_size_t, c_void_p]),
    "idl_profiles_chunked_bytes": (c_size_t, [c_i64, c_i64, ctypes.POINTER(Variant), c_int, c_int]),
    "idl_profiles_chunked": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int,
                                     ctypes.POINTER(Variant), c_int, c_void_p, c_int, c_u64, c_void_p, c_void_p, c_int,
                                     c_void_p, ctypes.POINTER(c_i64), c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_i64,
                                     c_void_p, c_size_t, c_void_p]),
    "idl_prepare_bytes": (c_size_t, [c_i64]),
    "idl_profiles_prepare": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, ctypes.POINTER(Variant),
                                     c_int, c_u64, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_int, ctypes.POINTER(c_int), c_void_p,
                                     c_void_p, c_size_t, c_void_p]),
    "idl_profiles_prepared": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, ctypes.POINTER(Variant),
                                      c_int, c_u64, c_int, c_void_p, ctypes.POINTER(c_i64), c_i64, c_int, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]),
    "idl_cgr_map": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p]),
    "idl_revcomp_canonical": (c_int, [c_int, c_void_p]),
    "idl_revcomp_fold": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "idl_normalize_counts": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_void_p]),
    "idl_kmer_counts": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "idl_colstats_parts": (c_int, [c_i64]),
    "idl_colstats": (c_int, [c_void_p, c_int, c_i64, c_int, c_void_p, c_void_p, c_void_p]),
    "idl_scaler_finalize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "idl_standardize_f32": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_void_p, c_void_p, c_void_p]),
    "idl_standardize_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_int, c_void_p, c_void_p, c_void_p]),
    "idl_nce_normalize": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "idl_nce_softmax_xent": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "idl_nce_softmax_xent_scaled": (c_int, [c_void_p, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "idl_nce_normalize_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "idl_nce_normalize_backward_parts": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "idl_iid_partial_s2": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "idl_iid_global_finish": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_void_p, c_float,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_nce_gather_rows": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "idl_nce_softmax_xent_rows": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p]),
    "idl_nce_normalize_backward_global": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                                  c_void_p]),
    "idl_relu_dropout_forward": (c_int, [c_void_p, c_int, c_void_p, c_i64, c_int, c_float, c_u64, c_void_p, ctypes.c_uint32, c_void_p, c_void_p]),
    "idl_relu_dropout_backward": (c_int, [c_void_p, c_void_p, c_i64, c_float, c_void_p, c_void_p]),
    "idl_sum_parts_bias": (c_int, [c_void_p, c_int, c_void_p, c_i64, c_int, c_void_p, c_void_p]),
    "idl_pair_selection": (c_int, [c_void_p, c_int, c_i64, c_void_p, c_void_p, c_void_p]),
    "idl_rmsprop_step": (c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_float, c_float, c_float, c_float, c_float, c_void_p]),
    "idl_rmsprop_allreduce_step": (c_int, [c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_i64, c_int, c_int, c_float, c_float, c_float, c_float, c_void_p]),
    "idl_sgd_step": (c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_float, c_float, c_float, c_void_p, c_float, c_void_p]),
    "idl_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_float, c_double, c_double, c_float, c_float, c_void_p, c_float,
                              c_void_p]),
    "idl_sgd_allreduce_step": (c_int, [c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_i64, c_int, c_int, c_float, c_float, c_float, c_void_p,
                                       c_void_p]),
    "idl_adam_allreduce_step": (c_int, [c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_i64, c_int, c_int, c_float, c_double, c_double,
                                        c_float, c_float, c_void_p, c_void_p]),
    "idl_fasta_scan": (c_int, [c_void_p, c_i64, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "idl_fasta_extract": (c_int, [c_void_p, c_i64, c_i64, c_void_p, c_i64, c_void_p, c_void_p, c_void_p]),
    "idl_iid_loss_max_clusters": (c_int, []),
    "idl_iid_loss_workspace_bytes": (c_size_t, [c_int]),
    "idl_iid_loss": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_size_t, c_void_p]),
    "idl_iid_joint_algebra": (c_int, [c_void_p, c_int, c_float, c_float, c_float, c_float, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    "idl_iid_loss_scaled": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_void_p, c_float, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_hdbscan_workspace_bytes": (c_size_t, [c_i64, c_int]),
    "idl_core_distances": (c_int, [c_void_p, c_i64, c_int, c_i64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_mreach_mst": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_core_distances_rows": (c_int, [c_void_p, c_i64, c_int, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_mreach_mst_parts": (c_int, [c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(c_i64),
                                     ctypes.POINTER(c_i64), c_i64, c_int, c_void_p, c_void_p, c_void_p, ctypes.POINTER(c_void_p),
                                     ctypes.POINTER(c_size_t), ctypes.POINTER(c_void_p)]),
    "idl_silhouette_workspace_bytes": (c_size_t, [c_i64, c_i64]),
    "idl_silhouette_samples": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_i64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "idl_silhouette_samples_rows": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_size_t, c_void_p]),
}

_lib = None


class IdelucsB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once) and bind every prototype.  Raises if it is missing —
    the product path has no CPU or PyTorch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IdelucsB200Error(
            "libidelucs_b200.so not found at %s — build it with `python __graft_entry__.py` "
            "(nvcc, sm_100a). idelucs_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.idl_abi_version() != 3:
        raise IdelucsB200Error("ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc != IDL_OK:
        msg = load().idl_last_error().decode(errors="replace")
        raise IdelucsB200Error("idelucs_b200 call failed (code %d): %s" % (rc, msg))


def ptr(t):
    """device (or host) pointer of a torch tensor / None"""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
