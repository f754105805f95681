"""ctypes binding of libmgcn.so (the C-ABI declared in include/mgcn.h).

There is no CPU fallback: if the shared object is missing this module raises at import of the
first op, and every entry point raises RuntimeError on a non-zero return code.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MGCN_LIB") or os.path.join(_PKG, "lib", "libmgcn.so")   # MGCN_LIB: tuning variants

c_i64 = ctypes.c_int64
c_i32 = ctypes.c_int32
c_int = ctypes.c_int
c_f32 = ctypes.c_float
c_ptr = ctypes.c_void_p
c_size_p = ctypes.POINTER(ctypes.c_size_t)


class MgcnCsr(ctypes.Structure):
    """mirror of mgcn_csr_t (include/mgcn.h)"""
    _fields_ = [
        ("n_rows", c_i64),
        ("nnz_cap", c_i64),
        ("hub_cap", c_i64),
        ("seg_cap", c_i64),
        ("hub_threshold", c_i32),
        ("reserved", c_i32),
        ("rowptr", c_ptr),
        ("nbr", c_ptr),
        ("perm", c_ptr),
        ("order", c_ptr),
        ("hub_rows", c_ptr),
        ("hub_seg0", c_ptr),
        ("hub_count", c_ptr),
        ("seg_row", c_ptr),
        ("seg_beg", c_ptr),
        ("seg_count", c_ptr),
        ("tasks", c_ptr),
        ("nbr_w", c_ptr),
    ]


CSR_P = ctypes.POINTER(MgcnCsr)

# name -> (restype, argtypes); must list every symbol include/mgcn.h declares
SIGNATURES = {
    "mgcn_version": (c_int, []),
    "mgcn_error_string": (ctypes.c_char_p, [c_int]),
    "mgcn_launch_count": (c_i64, []),
    "mgcn_reset_launch_count": (None, []),
    "mgcn_csr_capacities": (c_int, [c_i64, c_i64, c_int, c_i32, ctypes.POINTER(c_i64),
                                    ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "mgcn_csr_build": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, CSR_P, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_csr_build_i32": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, CSR_P, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_edge_fingerprint_i32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr]),
    "mgcn_edge_layout": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_edge_layout_i32": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_csr_build_presorted": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_ptr, c_ptr, CSR_P, c_ptr, c_ptr,
                                         c_size_p, c_ptr]),
    "mgcn_csr_build_presorted_i32": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_ptr, c_ptr, CSR_P, c_ptr,
                                             c_ptr, c_size_p, c_ptr]),
    "mgcn_preprocess_edges": (c_int, [c_ptr, c_i64, c_i64, c_int, c_int, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                      c_ptr, c_size_p, c_ptr]),
    "mgcn_degree_from_rowptr": (c_int, [c_ptr, c_i64, c_ptr, c_ptr]),
    "mgcn_weighted_degree": (c_int, [CSR_P, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "mgcn_gcn_norm": (c_int, [c_ptr, c_i64, c_int, c_ptr, c_ptr]),
    "mgcn_gcn_first_layer_fwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                         c_int, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_gcn_first_layer_fwd_ex": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                            c_ptr, c_ptr, c_f32, c_int, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_gcn_layer_fwd_tc": (c_int, [CSR_P, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int,
                                      c_i64, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_fwd_tc_ex": (c_int, [CSR_P, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                         c_f32, c_int, c_i64, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_fwd_tm": (c_int, [CSR_P, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int,
                                      c_i64, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_segment_max": (c_int, [CSR_P, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_segment_max_ex": (c_int, [CSR_P, c_ptr, c_i64, c_i64, c_int, c_ptr, c_f32, c_ptr, c_ptr, c_ptr]),
    "mgcn_segment_max_bwd": (c_int, [CSR_P, c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "mgcn_scatter_max_bwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr]),
    "mgcn_edge_dot": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_edge_dot_i32": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "mgcn_edge_fingerprint": (c_int, [c_ptr, c_i64, c_ptr, c_ptr]),
    "mgcn_binary_confusion": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr]),
    "mgcn_permute_edge_values": (c_int, [CSR_P, c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "mgcn_spmm": (c_int, [CSR_P, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr, c_int, c_ptr,
                          c_ptr, c_int, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_aggregate_prescaled": (c_int, [CSR_P, c_ptr, c_i64, c_i64, c_ptr, c_int, c_ptr, c_ptr,
                                         c_int, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_linear": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_int,
                            c_ptr, c_ptr]),
    "mgcn_linear_ex": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr,
                               c_int, c_ptr, c_ptr, c_ptr]),
    "mgcn_linear_wide": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_int, c_ptr,
                                 c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_linear_wgrad_ex": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64,
                                     c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_masked_scale": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "mgcn_linear_wgrad": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr,
                                  c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_fwd": (c_int, [CSR_P, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                   c_ptr, c_int, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_bwd": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr,
                                   c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_bwd_tc": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_gcn_layer_bwd_fused": (c_int, [CSR_P, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64,
                                         c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_mask_bits_scale": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "mgcn_dropout_keep_bits": (c_int, [c_ptr, c_i64, c_i64, c_i64, c_f32, c_ptr, c_ptr]),
    "mgcn_dropout_apply": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_f32, c_ptr]),
    "mgcn_cross_entropy_fwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr, c_size_p,
                                       c_ptr]),
    "mgcn_cross_entropy_bwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_ptr]),
    "mgcn_relu_backward": (c_int, [c_ptr, c_ptr, c_i64, c_ptr, c_ptr]),
    "mgcn_batch_to_offsets": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr]),
    "mgcn_segment_reduce": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_segment_broadcast": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_int, c_ptr, c_ptr]),
    "mgcn_head_cross_entropy_fwd": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_int, c_ptr, c_ptr,
                                            c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_head_cross_entropy_bwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_int, c_ptr, c_ptr,
                                            c_ptr, c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_batchnorm_fwd": (c_int, [c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_f32, c_f32, c_int, c_ptr, c_ptr, c_ptr, c_ptr,
                                   c_ptr, c_ptr, c_size_p, c_ptr]),
    "mgcn_batchnorm_bwd": (c_int, [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr,
                                   c_size_p, c_ptr]),
}

_lib = None


def load():
    """Load libmgcn.so (once) and attach signatures.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m meta_gcn_b200.build` "
            "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().mgcn_error_string(code).decode()
        raise RuntimeError(f"libmgcn call failed ({code}): {msg}")


def launch_count():
    return int(load().mgcn_launch_count())


def reset_launch_count():
    load().mgcn_reset_launch_count()
