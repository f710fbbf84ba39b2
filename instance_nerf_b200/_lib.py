"""ctypes binding of libinerf_b200.so (the C-ABI declared in include/inerf_b200.h).

This is the L1<->L0 boundary of the reference (the `_backend` pybind modules,
raymarching/raymarching.py:9-12, gridencoder/grid.py:9-12,
shencoder/sphere_harmonics.py:9-12) re-expressed as a plain C ABI: raw device
pointers, explicit sizes, the CUDA stream passed explicitly, integer return
codes turned into RuntimeError here.

There is NO fallback: if the shared library is missing or a CUDA tensor is not
supplied the call raises.  PyTorch only provides device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_size_t, c_uint8, c_uint32, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# INERF_B200_LIB: development override (A/B builds of the same library, csrc/Makefile VARIANT=); never a fallback
LIB_PATH = os.environ.get("INERF_B200_LIB") or os.path.join(_HERE, "libinerf_b200.so")
CSRC = os.path.join(_HERE, "csrc")

_lib = None


class InerfError(RuntimeError):
    pass


class FieldDesc(ctypes.Structure):
    """struct inerf_field_desc (include/inerf_b200.h)."""

    _fields_ = [
        ("table_packed", c_void_p),
        ("offsets", c_void_p),
        ("weights", c_void_p),
        ("L", c_uint32),
        ("H", c_uint32),
        ("S", c_float),
        ("bound", c_float),
        ("K", c_uint32),
        ("density_scale", c_float),
        ("n_valid", c_void_p),
    ]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libinerf_b200.so in-tree with nvcc for sm_100a (csrc/Makefile)."""
    if force:
        subprocess.run(["make", "-C", CSRC, "clean"], check=True, capture_output=not verbose)
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if r.returncode != 0:
        raise InerfError("building libinerf_b200.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    if verbose:
        print(r.stdout)
    return LIB_PATH


# name -> argtypes (restype is always int unless listed in _SPECIAL)
_P = c_void_p
_U = c_uint32
_F = c_float
_I = c_int
_PROTOS = {
    "inerf_near_far_from_aabb": [_P, _P, _P, _U, _F, _P, _P, _P],
    "inerf_sph_from_ray": [_P, _P, _F, _U, _P, _P],
    "inerf_morton3D": [_P, _U, _P, _P],
    "inerf_morton3D_invert": [_P, _U, _P, _P],
    "inerf_packbits": [_P, _U, _F, _P, _P],
    "inerf_march_rays_train": [_P, _P, _P, _F, _F, _U, _U, _U, _U, _U, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "inerf_march_rays_train_count_t": [_P, _P, _P, _F, _F, _U, _U, _U, _U, _P, _P, _P, _P, _P, _P, _P],
    "inerf_march_rays_train_expand": [_P, _P, _F, _F, _U, _U, _U, _U, _U, _P, _P, _P, _P, _P, _P, _P, _P],
    "inerf_composite_rays_train_forward": [_P, _P, _P, _P, _U, _U, _F, _P, _P, _P, _P],
    "inerf_composite_rays_train_backward": [_P, _P, _P, _P, _P, _P, _P, _P, _U, _U, _F, _P, _P, _P],
    "inerf_composite_rays_with_masks_train_forward": [_P, _P, _P, _P, _P, _U, _U, _U, _F, _P, _P, _P, _P, _P],
    "inerf_composite_rays_with_masks_train_backward": [_P] * 11 + [_U, _U, _U, _F, _P, _P, _P, _P, _P],
    "inerf_composite_rays_with_masks_train_backward_dense": [_P] * 11 + [_U, _U, _U, _F, _P, _P, _P, _P],
    "inerf_march_rays": [_U, _U, _P, _P, _P, _P, _F, _F, _U, _U, _U, _P, _P, _P, _P, _P, _P, _P, _P],
    "inerf_composite_rays": [_U, _U, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "inerf_composite_rays_with_masks": [_U, _U, _U, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "inerf_compact_alive": [_P, _U, _P, _P, _P],
    "inerf_frame_to_u8": [_P, _P, _P, _U, _U, _P, _P, _P, _P],
    "inerf_project_labels": [_P, _P, _U, _P, _U, _U, _U, _P, _P, _P, _P],
    "inerf_get_rays": [_P, _U, _F, _F, _F, _F, _U, _U, _P, _U, _P, _P, _P, _F, _P, _P, _P],
    "inerf_grid_encode_forward": [_P, _P, _P, _P, _U, _U, _U, _U, _F, _U, _P, _U, _I, _U, _I, _I, _P],
    "inerf_grid_encode_backward": [_P, _P, _P, _P, _P, _U, _U, _U, _U, _F, _U, _P, _P, _U, _I, _U, _I, _I, _P],
    "inerf_grad_total_variation": [_P, _P, _P, _P, _F, _U, _U, _U, _U, _F, _U, _U, _I, _I, _P],
    "inerf_sh_encode_forward": [_P, _P, _U, _U, _U, _P, _P],
    "inerf_sh_encode_backward": [_P, _P, _U, _U, _U, _P, _P, _P],
    "inerf_mask_loss": [_P, _P, _P, _U, _U, _U, _F, _P, _P, _P],
    "inerf_mask_loss_backward": [_P, _P, _P, _U, _U, _U, _F, _P, _P, _P, _P],
    "inerf_occupancy_ema": [_P, _P, _U, _F, _P, _P],
    "inerf_occupancy_pack": [_P, _U, _P, _F, _P, _P, _P],
    "inerf_occupancy_sample_cells": [_P, _U, _U, _U, _P, _P, ctypes.c_uint64, _P, _P, _P],
    "inerf_occupancy_points": [_U, _U, _F, _P, _U, _P, ctypes.c_uint64, _P, _P, _P],
    "inerf_occupancy_density": [POINTER(FieldDesc), _U, _U, _P, _U, _P, ctypes.c_uint64, _P, _P],
    "inerf_mark_untrained_grid": [_P, _U, _F, _F, _F, _F, _U, _U, _F, _P, _P, _P],
    "inerf_fill_f32": [_P, _U, _F, _P],
    "inerf_field_pack_weights": [_P] * 8 + [_U, _P],
    "inerf_field_pack_tables": [_P, _P, _I, ctypes.c_uint64, _P, _P],
    "inerf_field_forward": [POINTER(FieldDesc), _P, _P, _U, _P, _P, _P, _P],
    "inerf_field_forward_train": [POINTER(FieldDesc), _P, _P, _U, _P, _P, _P, _P, _P],
    "inerf_field_pack_weights_bwd": [_P, _P, _P, _U, _P],
    "inerf_field_pack_weights_device": [_P] * 8 + [_U, _P, _P, _P],
    "inerf_field_backward_mask": [POINTER(FieldDesc), _P, _P, _P, _P, _U, _P, _P, _P, _P, _P],
    "inerf_field_forward_train_rgb": [POINTER(FieldDesc), _P, _P, _U, _P, _P, _P, _P],
    "inerf_field_pack_weights_rgb_bwd_device": [_P, _P, _P, _P, _P, _P, _P],
    "inerf_field_backward_rgb": [POINTER(FieldDesc), _P, _P, _P, _P, _P, _P, _P, _U, _P, _P, _P, _P, _P, _P, _P],
    "inerf_adam_step": [_P, _P, _P, _P, ctypes.c_uint64, _F, _F, _F, _F, _P, _P, _P, _F, _P],
    "inerf_adam_advance": [_P, _P, _P],
    "inerf_render_fused": [POINTER(FieldDesc), _P, _P, _P, _P, _P, _U, _U, _U, _F, _U, _F, _P, _P, _P, _P, _P, _P],
    "inerf_render_fused_perturb": [POINTER(FieldDesc), _P, _P, _P, _P, _P, _P, _U, _U, _U, _F, _U, _F, _P, _P, _P, _P, _P, _P],
    "inerf_volume_points": [_P, _U, _U, _U, _P, _U, _U, _F, _P, _P, _P],
    "inerf_extract_volume": [POINTER(FieldDesc), _P, _U, _U, _U, _P, _U, _U, _P, _F, _P, _P, _P, _P, _P, _P],
    "inerf_mesh_count": [_P, _U, _U, _U, _F, _P, _P, _P],
    "inerf_mesh_emit": [_P, _U, _U, _U, _P, _F, _P, _P, _P, _P],
}
_SPECIAL = {
    "inerf_version": ([], c_int),
    "inerf_error_string": ([c_int], c_char_p),
    "inerf_field_weights_bytes": ([_U], c_size_t),
    "inerf_field_bwd_weights_bytes": ([], c_size_t),
    "inerf_field_rgb_bwd_weights_bytes": ([], c_size_t),
    "inerf_march_scratch_floats": ([_U, _U], c_size_t),
    "inerf_occupancy_sample_scratch_ints": ([_U, _U], c_size_t),
    "inerf_extract_scratch_ints": ([_U, _U, _U], c_size_t),
    "inerf_mesh_scratch_ints": ([_U, _U, _U], c_size_t),
}

# Every symbol include/inerf_b200.h declares; tests check the .so exports all of them.
EXPORTED_SYMBOLS = sorted(list(_PROTOS) + list(_SPECIAL))


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise InerfError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C instance_nerf_b200/csrc`). There is no CPU or PyTorch fallback."
            )
        L = ctypes.CDLL(LIB_PATH)
        for name, argtypes in _PROTOS.items():
            fn = getattr(L, name, None)
            if fn is None:
                continue  # reported by tests/test_abi.py; calling it raises AttributeError
            fn.argtypes = argtypes
            fn.restype = c_int
        for name, (argtypes, restype) in _SPECIAL.items():
            fn = getattr(L, name, None)
            if fn is None:
                continue
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = L
    return _lib


# Derived device copies (fp16 tables, packed weight blobs) are cached and keyed on each parameter's version counter.
# Fused / foreach optimizers update parameters WITHOUT bumping `_version` (measured: torch.optim.Adam(fused=True)), so a
# global optimizer-step hook advances this epoch, which is part of every cache key.  After writing parameters through
# `.data` by hand, call `invalidate_param_caches()`.
PARAM_EPOCH = [0]


def invalidate_param_caches(*_args, **_kwargs) -> None:
    PARAM_EPOCH[0] += 1


try:
    from torch.optim.optimizer import register_optimizer_step_post_hook as _reg_hook
    _reg_hook(invalidate_param_caches)
except ImportError:  # very old torch: callers must invalidate by hand
    pass


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().inerf_error_string(code).decode()
        raise InerfError(f"{what}: {msg} (code {code})" if what else f"{msg} (code {code})")


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise InerfError("libinerf_b200 takes CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise InerfError("tensor must be contiguous")
    return t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def call(name: str, *args) -> None:
    check(getattr(lib(), name)(*args), name)
