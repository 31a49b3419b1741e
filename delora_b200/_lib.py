"""ctypes binding of the C ABI in include/delora_b200.h (the "thin torch extension": torch only
supplies device pointers and the current stream).  There is NO fallback: if the shared library
is missing or a GPU is absent the product path raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdelora_b200.so")

c_int, c_float, c_double, c_void_p = ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_void_p
c_u32, c_i64 = ctypes.c_uint32, ctypes.c_int64

# name -> (restype, argtypes); every symbol declared in include/delora_b200.h
SIGNATURES = {
    "delora_abi_version": (c_int, []),
    "delora_last_error": (ctypes.c_char_p, []),
    "delora_project_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_double,
                                   c_double, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "delora_project_uv": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_double,
                                  c_double, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "delora_sort_scratch_bytes": (c_i64, [c_int, c_int]),
    "delora_sort_by_range": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "delora_normals_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "delora_normals_select_staging": (c_int, [c_int]),
    "delora_scan_blocks": (c_int, [c_int]),
    "delora_lists_from_images": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
    "delora_grid_build": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_double,
                                  c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "delora_grids_from_projection": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                             c_void_p, c_void_p, c_void_p]),
    "delora_pack_lists": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "delora_icp_partial_rows": (c_int, [c_int]),
    "delora_icp_scratch_floats": (c_i64, [c_int, c_int]),
    "delora_icp_stats": (c_int, [c_void_p, c_int]),
    "delora_icp_dense_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                         c_double, c_double, c_double, c_double, c_float, c_u32, c_void_p,
                                         c_void_p, c_void_p, c_void_p]),
    "delora_icp_fwd_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_int, c_int, c_int, c_double, c_double, c_double, c_double, c_float,
                                   c_u32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "delora_icp_point_grads": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p]),
    "delora_conv2d_fprop_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "delora_conv_select_kernel": (c_int, [c_int]),
    "delora_conv2d_dgrad_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "delora_conv2d_dgrad_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "delora_conv2d_wgrad_scratch_floats": (c_i64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "delora_conv2d_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_int, c_void_p]),
    "delora_zero_upsample_nhwc_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                               c_void_p]),
    "delora_images_to_nhwc_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_maxpool_w_nhwc_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_maxpool_w_idx_nhwc_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                               c_void_p]),
    "delora_maxpool_w_bwd_nhwc_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                               c_int, c_void_p]),
    "delora_avgpool_nhwc_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_avgpool_bwd_nhwc_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_conv_weight_prep_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "delora_conv_weight_prep_multi": (c_int, [c_void_p, c_int, c_void_p]),
    "delora_images_to_nhwc16_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_stem_weight_prep_bf16": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "delora_stem_fprop_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "delora_stem_wgrad_scratch_floats": (c_i64, [c_int, c_int, c_int]),
    "delora_stem_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "delora_nhwc_to_nchw_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "delora_quat_to_T": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "delora_quat_to_T_bwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "delora_grad_allreduce_flag_words": (c_int, []),
    "delora_grad_allreduce_f32": (c_int, [c_void_p, c_void_p, ctypes.c_uint64, c_int, c_int, ctypes.c_longlong,
                                          ctypes.c_longlong, c_float, c_u32, c_int, c_int, c_void_p, c_void_p]),
}

ABI_VERSION = 1
_lib = None


def lib():
    """Load libdelora_b200.so (built by `python -m delora_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"delora_b200: {LIB_PATH} is missing. Build it with `python delora_b200/build.py` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    handle = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(handle, name)          # AttributeError if the library does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.delora_abi_version() != ABI_VERSION:
        raise RuntimeError("delora_b200: ABI version mismatch between _lib.py and libdelora_b200.so")
    _lib = handle
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().delora_last_error()
        raise RuntimeError(f"{what} failed ({status}): {msg.decode() if msg else ''}")
