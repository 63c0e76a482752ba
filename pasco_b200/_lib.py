"""ctypes binding of libpasco_sm100.so (the C-ABI declared in include/pasco_sm100.h).

There is NO fallback: if the shared library is missing, or a compute entry point is called
without a CUDA device, this raises.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpasco_sm100.so")

_p = C.c_void_p
_i32, _i64 = C.c_int32, C.c_int64

# name → (restype, argtypes); mirrors include/pasco_sm100.h one to one
PROTOTYPES = {
    "pasco_last_error": (C.c_char_p, []),
    "pasco_abi_version": (C.c_int, []),
    "pasco_device_info": (C.c_int, [_p, _p, _p]),
    "pasco_hash_insert": (C.c_int, [_p, _i64, _p, _p, _i64, _p, _p, _p]),
    "pasco_hash_remap": (C.c_int, [_p, _i64, _p, _p]),
    "pasco_hash_lookup": (C.c_int, [_p, _i64, _p, _p, _i64, _p, _p]),
    "pasco_coords_floor": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p]),
    "pasco_coords_generate_k2": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p]),
    "pasco_kernel_map_probe": (C.c_int, [_p, _i64, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p]),
    "pasco_kernel_map_box": (C.c_int, [_p, _i64, _p, _p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p]),
    "pasco_kernel_map_down": (C.c_int, [_p, _i64, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p, _i64, _p]),
    "pasco_mask_block_counts": (C.c_int, [_p, _i64, _p, _p]),
    "pasco_mask_compact": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "pasco_gather_rows": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "pasco_scatter_rows": (C.c_int, [_p, _p, _i64, _i32, _p, _i32, _p]),
    "pasco_gather_coords": (C.c_int, [_p, _p, _i64, _p, _p]),
    "pasco_to_dense": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _i32, _i32, _i32, _i32, _p, _p]),
    "pasco_from_dense": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _i32, _i32, _i32, _i32, _p, _p]),
    "pasco_dense_occupancy": (C.c_int, [_p, _i32, _i32, _i64, _p, _p]),
    "pasco_conv_packed_bytes": (_i64, [_i32, _i32, _i32]),
    "pasco_conv_pack_weights": (C.c_int, [_p, _i32, _i32, _i32, _i32, _p, _p]),
    "pasco_conv_forward_tc": (C.c_int, [_p, _i64, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _p, _p, _i32, _p, _p, _i32, _i64, _i64, _p]),
    "pasco_conv_splitk_workspace_bytes": (_i64, [_i32, _i64, _i32]),
    "pasco_conv_forward_splitk": (C.c_int, [_p, _i64, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _p, _p, _i32, _p, _i32, _i64, _i64, _p, _i64, _p]),
    "pasco_split_planes": (C.c_int, [_p, _i64, _i32, _i64, _p, _p, _i32, _p, _p, _p]),
    "pasco_conv_forward_planes": (C.c_int, [_p, _p, _i64, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _p, _p, _i32, _i64, _i64, _p]),
    "pasco_conv_wgrad_planes": (C.c_int, [_p, _p, _i64, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _i32, _i64, _i64, _p, _i64, _p]),
    "pasco_conv_wgrad_workspace_bytes": (_i64, [_i32, _i64, _i32, _i32]),
    "pasco_conv_wgrad_tc": (C.c_int, [_p, _i64, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _i32, _p, _i32, _i64, _i64, _p, _i64, _p]),
    "pasco_conv_forward_simt": (C.c_int, [_p, _p, _i32, _i64, _i32, _i32, _p, _i32, _p, _p, _p, _p]),
    "pasco_conv_wgrad_simt_workspace_bytes": (_i64, [_i32, _i64, _i32, _i32]),
    "pasco_conv_wgrad_simt": (C.c_int, [_p, _p, _i32, _i64, _i32, _i32, _p, _p, _p, _i64, _p]),
    "pasco_maxpool_forward": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "pasco_scatter_max": (C.c_int, [_p, _p, _i64, _i32, _p, _i64, _p, _p]),
    "pasco_bn_stats": (C.c_int, [_p, _i64, _i32, _p, _p]),
    "pasco_affine_act": (C.c_int, [_p, _i64, _i32, _p, _p, _i32, _p, _p, _p]),
    "pasco_bn_finalize": (C.c_int, [_p, _p, C.c_double, _i32, _p, _p, C.c_float, C.c_float, _p, _p, _p, _p, _p, _p, _p]),
    "pasco_bn_bwd_coefs": (C.c_int, [_p, _p, C.c_double, _i32, _p, _p, _p, C.c_float, _p, _p, _p, _p, _p, _p]),
    "pasco_bn_bwd_reduce": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _i32, _p, _p]),
    "pasco_xattn_workspace_bytes": (_i64, [_i32, _i64, _i32, _i32]),
    "pasco_xattn_forward": (C.c_int, [_p, _p, _p, _p, _i32, _i64, _i32, _i32, C.c_float, _p, _p, _p, _i64, _p]),
    "pasco_xattn_backward": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _i64, _i32, _i32, C.c_float, _p, _p, _p, _p, _i64, _p]),
    "pasco_bn_bwd_apply": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "pasco_eval_ssc_workspace_bytes": (_i64, [_i64, _i32]),
    "pasco_eval_ssc": (C.c_int, [_p, _p, _i64, _i32, _p, _i32, _p, _p, _p, _i64, _p, _p]),
    "pasco_eval_pairs": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _i32, _i32, _p, _p, _p]),
    "pasco_eval_calib_workspace_bytes": (_i64, [_i64, _i32]),
    "pasco_eval_calib": (C.c_int, [_p, _p, _p, _i64, _p, _p, _i64, _p, _i32, _p, _i32, _p, _p, _p, _i64, _p, _p]),
}

_lib: Optional[C.CDLL] = None


class PascoError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the in-tree library and type every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PascoError(
                f"{LIB_PATH} not found — build it with `python -m pasco_b200.build` "
                "(pasco_b200 has no CPU or eager fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)          # AttributeError ⇒ header / library out of sync
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    assert t.is_cuda, "pasco_b200 ops take CUDA tensors only (no CPU path)"
    assert t.is_contiguous(), "pasco_b200 ops take contiguous tensors"
    return t.data_ptr()


def call(name: str, *args):
    """Invoke a C-ABI entry point on torch's current stream; raise RuntimeError on failure
    (MinkowskiEngine's pybind layer raises the same way)."""
    lib = load()
    if not torch.cuda.is_available():
        raise PascoError(f"{name}: no CUDA device — pasco_b200 has no CPU fallback")
    rc = getattr(lib, name)(*args, _stream())
    if rc != 0:
        raise PascoError(f"{name} failed ({rc}): {lib.pasco_last_error().decode()}")


def int_array(vals):
    return (C.c_int32 * len(vals))(*[int(v) for v in vals])
