"""ctypes binding of ``libcsvit_sm100.so`` (C ABI declared in ``include/csvit.h``).

The product path has no CPU or PyTorch fallback: if the shared library is missing the import of
``cs_vit.ops`` fails loudly with build instructions, and every op raises on non-CUDA tensors.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CSVIT_LIB", os.path.join(_HERE, "..", "lib", "libcsvit_sm100.so"))

# name -> argtypes; restype is int for everything except csvit_last_error.
SIGNATURES = {
    "csvit_abi_version": [],
    "csvit_window_index_map": [c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "csvit_shift_mask": [c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "csvit_rel_pos_index": [c_int, c_void_p, c_void_p],
    "csvit_merge_index_map": [c_int, c_int, c_void_p, c_void_p],
    "csvit_host_window_index_map": [c_int, c_int, c_int, c_int, c_void_p],
    "csvit_host_shift_mask": [c_int, c_int, c_int, c_int, c_void_p],
    "csvit_host_rel_pos_index": [c_int, c_void_p],
    "csvit_host_merge_index_map": [c_int, c_int, c_void_p],
    "csvit_expand_rel_bias": [c_void_p, c_void_p, c_int, c_int, c_void_p],
    "csvit_layernorm": [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_longlong, c_int, c_int, c_int,
                        c_int, c_int, c_int, c_int, c_void_p],
    "csvit_affine_rows": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_int, c_void_p],
    "csvit_patch_im2col": [c_void_p, c_void_p, c_int, c_int, c_int, ctypes.POINTER(c_float), ctypes.POINTER(c_float),
                           c_void_p],
    "csvit_linear": [c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                     c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "csvit_mlp_fused": [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p,
                        c_longlong, c_int, c_int, c_int, c_void_p],
    "csvit_swin_attn_fused": [c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                              c_int, c_int, c_int, c_int, c_void_p],
    "csvit_swin_attn_core": [c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                             c_int, c_int, c_void_p],
    "csvit_crop_resize": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p],
    "csvit_rot6d_to_axis_angle": [c_void_p, c_void_p, c_longlong, c_void_p],
    "csvit_mano_fk": [c_void_p] * 10 + [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p],
    "csvit_allreduce_f32": [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_float, c_int, c_void_p],
    "csvit_last_gemm_kernel": [],
    "csvit_set_gemm_tuning": [c_int, c_int, c_int, c_int],
    "csvit_window_attention": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "csvit_attention": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_longlong, c_longlong, c_longlong,
                        c_int, c_int, c_int, c_int, c_float, c_void_p],
    "csvit_swinv2_window_attention": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_int, c_int, c_void_p],
    "csvit_swinv2_qkv": [c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_longlong,
                         c_void_p],
    "csvit_swinv2_qkv_train": [c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_longlong, c_void_p, c_void_p],
    "csvit_swinv2_cosnorm_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                 c_void_p],
    "csvit_swinv2_attn_tc": [c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                             c_void_p],
    "csvit_swinv2_attn_tc_train": [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                   c_int, c_void_p],
    "csvit_swinv2_attn_tc_bwd": [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "csvit_swinv2_attn8_tc": [c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                              c_void_p],
    "csvit_swinv2_attn8_tc_train": [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                    c_int, c_void_p],
    "csvit_swinv2_attn8_tc_bwd": [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "csvit_layernorm_post": [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_longlong,
                             c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "csvit_gemm_ex": [c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_int, c_void_p, c_longlong,
                      c_int, c_int, c_int, c_int, c_void_p],
    "csvit_col_reduce": [c_void_p, c_int, c_longlong, c_void_p, c_longlong, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                         c_int, c_int, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p],
    "csvit_transpose_f32": [c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_void_p],
    "csvit_row_scale_add": [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p],
    "csvit_eltwise": [c_int, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p],
    "csvit_affine2_rows": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_void_p],
    "csvit_layernorm_bwd": [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_float, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "csvit_attention_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_longlong,
                            c_longlong, c_longlong, c_longlong, c_longlong, c_longlong, c_int, c_int, c_int, c_int, c_float,
                            c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
}

_lib = None


class CsvitError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = os.path.abspath(LIB_PATH)
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found. cs_vit has no CPU/PyTorch fallback: build the sm_100a kernels first with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` or `make -C cs-vit_b200/csrc`.")
    lib = ctypes.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_int
    lib.csvit_last_error.argtypes = []
    lib.csvit_last_error.restype = c_char_p
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise CsvitError(load().csvit_last_error().decode("utf-8", "replace"))
