"""ctypes binding of libpresight_b200.so — the only door from Python into the CUDA kernels.

The library is built in-tree by `presight_b200.build` (nvcc, sm_100a).  There is no fallback:
if the shared object is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", f"libpresight_b200{os.environ.get('PS_LIB_SUFFIX', '')}.so")

_p = C.c_void_p
_i64 = C.c_int64
_i = C.c_int
_f = C.c_float
_fp = C.POINTER(C.c_float)
_pp = C.POINTER(C.c_void_p)
_ip = C.POINTER(C.c_int)

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/presight_b200.h
SIGNATURES = {
    "ps_hash_fwd": [_p, _i64, _p, _fp, _i, _i, _i, _p, _p],
    "ps_hash_bwd": [_p, _i64, _p, _fp, _i, _i, _i, _p, _p, _p, _p],
    "ps_hash_fwd_lm": [_p, _i64, _p, _fp, _i, _i, _i, _p, _p],
    "ps_hash_bwd_lm": [_p, _i64, _p, _fp, _i, _i, _i, _p, _p, _p, _p],
    "ps_hash_levels_per_thread": [_i, _i, _i],
    "ps_hash_indices": [_p, _i64, _fp, _i, _i, _p, _p, _p],
    "ps_normalize_positions": [_p, _i64, _fp, _i, _p, _p, _p],
    "ps_sample_positions": [_p, _p, _p, _i64, _i, _p, _p],
    "ps_ray_points": [_p, _p, _p, _i64, _i, _fp, _i, _p, _p, _p],
    "ps_mlp_fwd_ex": [_p, _i, _i64, _pp, _pp, _ip, _i, _i, _i, _p, _p, _p, _p],
    "ps_mlp_bwd_ex": [_p, _i, _p, _i64, _pp, _pp, _ip, _i, _i, _i, _pp, _pp, _p, _p, _p],
    "ps_prior_finalize": [_pp, _i, _p, _i64, _i, _p, _p, _p],
    "ps_sh4": [_p, _i64, _i, _p, _p],
    "ps_nearest_centroid": [_p, _i64, _p, _i, _p, _p],
    "ps_mlp_fwd": [_p, _i64, _pp, _pp, _ip, _i, _i, _i, _p, _p],
    "ps_mlp_bwd": [_p, _p, _p, _i64, _pp, _pp, _ip, _i, _i, _i, _p, _pp, _pp, _p],
    "ps_trunc_exp_fwd": [_p, _p, _i64, _i64, _p, _p],
    "ps_trunc_exp_bwd": [_p, _p, _p, _i64, _i64, _p, _i64, _p],
    "ps_spaced_bins": [_p, _p, _p, _p, _i64, _i, _f, _p, _p, _p],
    "ps_pdf_resample": [_p, _p, _p, _p, _p, _p, _i64, _i, _i, _f, _f, _f, _f, _p, _p, _p, _p, _p, _p],
    "ps_searchsorted_right": [_p, _p, _i64, _i, _i, _p, _p],
    "ps_weights_fwd": [_p, _p, _i64, _i, _p, _p],
    "ps_weights_bwd": [_p, _p, _p, _i64, _i, _p, _p],
    "ps_render_fwd": [_p, _p, _i64, _i, _i, _p, _p],
    "ps_render_bwd": [_p, _p, _p, _i64, _i, _i, _p, _p, _p],
    "ps_depth_threshold": [_p, _p, _i64, _i, _f, _p, _p, _p],
    "ps_composite_fwd": [_p, _p, _p, _p, _i64, _i, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_composite_bwd": [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_interlevel_loss": [_p, _p, _p, _p, _i64, _i, _i, _p, _p, _p],
    "ps_distortion_loss": [_p, _p, _i64, _i, _p, _p, _p],
    "ps_zaa_interlevel_loss": [_p, _p, _i64, _i, _p, _p, _i, C.c_double, _p, _p, _p],
    "ps_sky_blend_fwd": [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p],
    "ps_sky_blend_bwd": [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p, _p],
    "ps_render_losses": [_p, _p, _p, _p, _p, _p, _i64, _i, _f, _p, _p, _p, _p, _p],
    "ps_depth_losses": [_p, _p, _p, _p, _p, _p, _i64, _i, _f, _p, _f, _f, _i, _p, _p, _p, _p],
    "ps_ms_route": [_p, _p, _p, _p, _i64, _i, _p, _i, _p, _p, _p],
    "ps_ms_plan": [_p, _i64, _i, _i, _i, _i64, _p, _p, _p],
    "ps_ms_scatter": [_p, _p, _p, _p, _i64, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p],
    "ps_hash_fwd_ms": [_p, _i64, _p, _p, _fp, _i, _i, _i, _p, _p],
    "ps_hash_bwd_ms": [_p, _i64, _p, _p, _p, _fp, _i, _i, _i, _p, _p],
    "ps_prop_level_fwd_ms": [_p, _i, _p, _p, _p, _p, _i64, _p, _fp, _i, _i, _i, _p, _p, _p],
    "ps_prop_level_bwd_ms": [_p, _i, _p, _p, _p, _p, _i64, _p, _fp, _i, _i, _i, _p, _p, _p],
    "ps_field_level_fwd_ms": [_p, _i, _p, _i, _i, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p],
    "ps_field_level_bwd_ms": [_p, _i, _p, _i, _i, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_voxel_min_bound": [_p, _p, _i64, _p, _p],
    "ps_voxel_accumulate": [_p, _p, _p, _p, _i64, _i, _p, C.c_double, _p, _i64, _p, _p, _p, _p, _p, _p],
    "ps_voxel_finalize": [_p, _i64, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p],
    "ps_hits_quantile": [_p, _i64, C.c_double, _p, _i64, _p, _p, _p],
    "ps_voxel_insert": [_p, _i64, _p, C.c_double, _p, _i64, _p, _p, _p],
    "ps_voxel_rehash": [_p, _i64, _p, _i64, _p, _p],
    "ps_voxel_assign_rows": [_p, _i64, _p, _i64, _p, _p, _p],
    "ps_voxel_accumulate_rows": [_p, _p, _p, _i64, _i, _p, C.c_double, _p, _p, _i64, _p, _p, _p, _p, _p, _p],
    "ps_voxel_finalize_rows": [_p, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p],
    "ps_generate_rays": [_p, _p, _p, _p, _p, _i, _p, _i64, _f, _p, _p, _p, _p, _p],
    "ps_assemble_batch": [_p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_peer_alloc": [C.c_size_t, _p],
    "ps_peer_free": [_p],
    "ps_peer_export": [_p, _p],
    "ps_peer_open": [_p, _p],
    "ps_peer_close": [_p],
    "ps_peer_copy": [_p, _p, C.c_size_t, _p],
    "ps_peer_wait_flags": [_p, _i, _i, C.c_uint32, _p],
    "ps_peer_reduce": [_p, _p, _i, _i64, _f, _p],
    "ps_peer_exchange_range": [_p, _i, _i, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_uint32, _f,
                               _p, _i, _p],
    "ps_adam_step": [_p, _p, _p, _p, _i64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _i64, _p],
    "ps_tc5_probe": [_p, _p, _p, _p, _p, _p, _p, _p],
    "ps_field_level_fwd": [_p, _p, _i, _i, _p, _p, _p, _p, _i64, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_field_level_bwd": [_p, _p, _i, _i, _p, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "ps_prop_level_feat_stride": [_i, _i],
    "ps_prop_level_fwd": [_p, _p, _p, _p, _i64, _i, _fp, _i, _p, _fp, _i, _i, _i, _p, _p, _p],
    "ps_prop_level_bwd": [_p, _p, _p, _p, _i64, _i, _fp, _i, _fp, _i, _i, _i, _p, _p, _p, _p],
    "ps_density_level_fwd": [_p, _p, _p, _p, _i64, _i, _fp, _i, _p, _fp, _i, _i, _i, _p, _p],
    "ps_density_level_fwd_ms": [_p, _i, _p, _p, _p, _p, _i64, _p, _fp, _i, _i, _i, _p, _p],
    "ps_surface_hits": [_p, _p, _p, _i64, _f, _f, _f, _f, _p, _p, _p, _p],
    "ps_hits_append_workspace": [_i64, _p],
    "ps_hits_append": [_p, _p, _p, _p, _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _p],
    "ps_image_metrics_workspace": [_i, _i, _i, _p],
    "ps_image_metrics": [_p, _p, _i, _i, _i, _f, _p, _p, _p, _p, _p],
    "ps_lpips_workspace": [_i, _i, _i, _p],
    "ps_lpips": [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p],
    "ps_colormap_workspace": [_i, _i64, _p],
    "ps_colormap": [_p, _i, _i64, _p, _p, _p, _p, _p],
    "ps_depth_metrics_workspace": [_i, _i64, _p],
    "ps_depth_metrics": [_p, _i, _i64, _p, _f, _p, _f, _f, _p, _p, _p],
    "ps_nn_grid_bounds": [_p, _i64, _p, _p],
    "ps_nn_grid_cells_per_axis": [_fp, C.c_double, _p],
    "ps_nn_grid_keys": [_p, _i64, _fp, C.c_double, _p, _p],
    "ps_nn_grid_count_cells": [_p, _i64, _p, _p],
    "ps_nn_grid_cells": [_p, _p, _p, _i64, _p, _p, _i64, _p, _p, _p],
    "ps_nn_grid_query": [_p, _p, _i64, _i64, C.POINTER(C.c_double), _i, _p, _p, _p, _p],
    "ps_nn_grid_reduce": [_p, _p, _i64, _i, _i64, _p, _p, _p],
}
_RESTYPES = {"ps_last_error": C.c_char_p, "ps_abi_version": C.c_int, "ps_launch_count": C.c_int64}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m presight_b200.build` "
            "(there is no CPU or PyTorch fallback for the presight_b200 kernels)")
    lib = C.CDLL(LIB_PATH)
    for name, restype in _RESTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = C.c_int
        fn.argtypes = argtypes
    _lib = lib
    return lib


def exported_symbols():
    return sorted(list(SIGNATURES) + list(_RESTYPES))


def launch_count() -> int:
    return int(load().ps_launch_count())


def hash_levels_per_thread(L: int, F: int, log2_T: int) -> int:
    return int(load().ps_hash_levels_per_thread(int(L), int(F), int(log2_T)))


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().ps_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"presight_b200.{what} failed (status {status}): {msg}")


def ptr(t: Optional[torch.Tensor]):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("presight_b200 kernels need CUDA tensors (no CPU fallback exists)")
    if not t.is_contiguous():
        raise RuntimeError("presight_b200 kernels need contiguous tensors")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def host_floats(vals: Sequence[float]):
    arr = (C.c_float * len(vals))(*[float(v) for v in vals])
    return arr


def host_ptrs(tensors: Sequence[Optional[torch.Tensor]]):
    arr = (C.c_void_p * len(tensors))(*[None if t is None else ptr(t) for t in tensors])
    return arr


class RowSegment(C.Structure):
    """ps_row_segment of include/presight_b200.h."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("stride", C.c_int64), ("col0", C.c_int),
                ("width", C.c_int), ("group", C.c_int), ("feat_per_level", C.c_int)]


def host_segments(segs):
    """segs: iterable of (src tensor, dst tensor|None, stride, col0, width, group[, feat_per_level])."""
    segs = list(segs)
    arr = (RowSegment * len(segs))()
    for i, seg in enumerate(segs):
        src, dst, stride, col0, width, group = seg[:6]
        arr[i].feat_per_level = int(seg[6]) if len(seg) > 6 else 0
        arr[i].src = src.data_ptr()
        arr[i].dst = None if dst is None else dst.data_ptr()
        arr[i].stride, arr[i].col0, arr[i].width, arr[i].group = int(stride), int(col0), int(width), int(group)
    return arr


class FieldNet(C.Structure):
    """ps_field_net of include/presight_b200.h."""
    _fields_ = [("W", C.c_void_p * 8), ("B", C.c_void_p * 8), ("dW", C.c_void_p * 8), ("dB", C.c_void_p * 8),
                ("app_dim", C.c_int)]


def host_field_net(weights, biases, app_dim, dweights=None, dbiases=None):
    """weights / biases: the 8 layers in the order base0, base1, sem0..2, rgb0..2 (CUDA fp32 tensors)."""
    net = FieldNet()
    for i in range(8):
        net.W[i] = ptr(weights[i])
        net.B[i] = ptr(biases[i])
        net.dW[i] = None if dweights is None else ptr(dweights[i])
        net.dB[i] = None if dbiases is None else ptr(dbiases[i])
    net.app_dim = int(app_dim)
    return net


class PropNet(C.Structure):
    """ps_prop_net of include/presight_b200.h."""
    _fields_ = [("W0", C.c_void_p), ("b0", C.c_void_p), ("W1", C.c_void_p), ("b1", C.c_void_p), ("dW0", C.c_void_p),
                ("db0", C.c_void_p), ("dW1", C.c_void_p), ("db1", C.c_void_p), ("hidden", C.c_int)]


def host_prop_net(ws, bs, dws=None, dbs=None):
    net = PropNet()
    net.W0, net.b0, net.W1, net.b1 = ptr(ws[0]), ptr(bs[0]), ptr(ws[1]), ptr(bs[1])
    if dws is not None:
        net.dW0, net.db0, net.dW1, net.db1 = ptr(dws[0]), ptr(dbs[0]), ptr(dws[1]), ptr(dbs[1])
    net.hidden = int(ws[0].shape[0])
    return net


class PropNetDev(C.Structure):
    """ps_prop_net_dev of include/presight_b200.h (arrays of these live in device memory)."""
    _fields_ = [("W0", C.c_void_p), ("b0", C.c_void_p), ("W1", C.c_void_p), ("b1", C.c_void_p), ("dW0", C.c_void_p),
                ("db0", C.c_void_p), ("dW1", C.c_void_p), ("db1", C.c_void_p)]


class FieldNetDev(C.Structure):
    """ps_field_net_dev of include/presight_b200.h."""
    _fields_ = [("W", C.c_void_p * 8), ("B", C.c_void_p * 8), ("dW", C.c_void_p * 8), ("dB", C.c_void_p * 8),
                ("in_dim", C.c_int), ("app_dim", C.c_int)]


class LpipsNet(C.Structure):
    """ps_lpips_net of include/presight_b200.h."""
    _fields_ = [("conv_w", C.c_void_p * 5), ("conv_b", C.c_void_p * 5), ("lin", C.c_void_p * 5)]


NN_BLOCK_QUERIES = 1024    # PS_NN_BLOCK_QUERIES
NN_MAX_TAUS = 8            # PS_NN_MAX_TAUS


class NNGrid(C.Structure):
    """ps_nn_grid of include/presight_b200.h."""
    _fields_ = [("points", C.c_void_p), ("cell_keys", C.c_void_p), ("cell_ranges", C.c_void_p),
                ("capacity", C.c_int64), ("origin", C.c_float * 3), ("cell", C.c_double)]


_DEV_TABLES = {}


def _device_table(slot, signature, build):
    """Small device-side tables (pointer arrays, network descriptors) are uploaded only when their content changes: the
    upload is a pageable-memory copy, i.e. a stream synchronisation, and in steady state the parameters never move and
    the caching allocator hands the per-step gradient buffers back at the same addresses."""
    hit = _DEV_TABLES.get(slot)
    if hit is None or hit[0] != signature:
        hit = (signature, build())
        _DEV_TABLES[slot] = hit
    return hit[1]


def device_struct_array(structs, device, slot) -> torch.Tensor:
    """ctypes structures -> one uint8 CUDA tensor holding them back to back (cached per `slot`, see _device_table)."""
    raw = b"".join(bytes(st) for st in structs)
    return _device_table((slot, str(device)), raw,
                         lambda: torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(device))


def device_ptr_array(tensors, device, slot) -> torch.Tensor:
    """Device array of the tensors' data pointers (int64), cached per `slot`."""
    sig = tuple(t.data_ptr() for t in tensors)
    return _device_table((slot, str(device)), sig, lambda: torch.tensor(sig, dtype=torch.int64).to(device))


def host_ints(vals: Sequence[int]):
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
