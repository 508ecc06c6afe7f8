"""ctypes binding of ``libfus_b200.so`` (the C ABI of ``include/fus_b200.h``).

There is no CPU fallback: if the library is missing it is built with nvcc, and
if that fails the import of any operator raises.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfus_b200.so")

_lib = None

FUS_TABLES_RESIDENT = 1
FUS_NO_ATOMICS = 2
FUS_HOST_Y_ZERO = 4

P = C.c_void_p
I = C.c_int
L = C.c_int64


def _sigs():
    """name -> argument ctypes, with ``T`` standing for the float type."""
    T = "T"
    s = {
        "fus_set_dphi": [I, P, P],
        "fus_stiffness": [P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness2": [P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness_westervelt": [P, P, P, P, P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness_affine": [P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness_westervelt_affine": [P, P, P, P, P, P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_set_rect_tables": [I, P, P, P],
        "fus_stiffness_rect": [P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness_westervelt_rect": [P, P, P, P, P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness2_affine": [P, P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness2_rect": [P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_trilinear_coeffs": [P, P, P, P, L, P],
        "fus_set_vertex_tables": [I, P, P, P],
        "fus_stiffness_vertex": [P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness2_vertex": [P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_stiffness_westervelt_vertex": [P, P, P, P, P, P, P, P, P, P, P, L, I, I, P],
        "fus_mass_vertex": [P, P, P, P, P, L, I, P],
        "fus_rk_close_westervelt_pw": [P, P, P, P, P, P, P, P, P, P, P, T, T, I, L, P, P, P],
        "fus_compress_geometry": [P, P, P, P, P, P, L, I, T, P],
        "fus_mass": [P, P, P, P, P, L, I, P],
        "fus_axpy": [T, P, P, L, P],
        "fus_copy": [P, P, L, P],
        "fus_fill": [T, P, L, P],
        "fus_pointwise_divide": [P, P, P, L, P],
        "fus_square": [P, P, L, P],
        "fus_pack_fwd": [P, P, P, L, P],
        "fus_unpack_fwd": [P, P, P, L, L, P],
        "fus_pack_rev": [P, P, P, L, L, P],
        "fus_unpack_rev": [P, P, P, L, P],
        "fus_pack_multi": [P, I, P, P, L, L, P],
        "fus_unpack_multi": [P, P, I, P, L, L, I, P],
        "fus_halo_put": [P, P, I, P],
        "fus_halo_wait_forward": [P, P, I, P],
        "fus_halo_get_add": [P, P, I, P],
        "fus_halo_forward": [P, P, I, P],
        "fus_halo_reverse": [P, P, I, P],
        "fus_rk_open": [P, P, P, P, P, P, P, P, T, I, L, P],
        "fus_rk_close": [P, P, P, P, P, P, P, P, P, T, T, I, L, P, P, P],
        "fus_rk_close_shared": [P, I, I, I, P, P, P, P, P, P, P, P, P, P, P, T, T, I, P],
        "fus_leapfrog_close": [P, P, P, P, T, T, L, P, P, P],
        "fus_rk_close_westervelt": [P, P, P, P, P, P, P, P, P, P, T, T, I, L, P, P, P],
        "fus_boundary_terms": [P, P, P, P, P, P, T, T, P, P, I, I, L, P],
        "fus_boundary_terms_signal": [P, P, P, P, P, P, P, T, T, P, P, I, I, L, I, P],
        "fus_boundary_terms_elements": [P, P, P, P, P, P, P, P, P, P, I, I, L, P],
        "fus_boundary_terms_elements_signal": [P, P, P, P, P, P, P, P, P, P, P, I, I, L, I, P],
        "fus_westervelt_mass": [P, P, P, P, P, P, P, P, L, I, P],
        "fus_geometry": [P, P, P, P, P, P, L, I, P],
        "fus_facet_geometry": [P, P, P, P, P, P, L, I, P],
        "fus_eval_points": [P, P, P, P, P, L, I, P],
        "fus_stiffness_host": [P, P, L, P, P, P, P, P, P, L, I, I, P],
    }
    return s


#: every symbol include/fus_b200.h declares (checked by tests/test_abi.py)
UNTYPED = ["fus_abi_version", "fus_last_error", "fus_launch_count", "fus_reset_launch_count",
           "fus_halo_pad_bytes", "fus_halo_create", "fus_halo_destroy", "fus_halo_num_shared",
           "fus_halo_shared_mask", "fus_halo_shared_tail", "fus_halo_status", "fus_halo_signal_reverse", "fus_halo_barrier",
           "fus_halo_wait_reverse", "fus_stiffness_arm_halo_wait"]


class HaloDesc(C.Structure):
    """``fus_halo_desc_t`` of include/fus_b200.h."""

    _fields_ = [("rank", C.c_int32), ("world", C.c_int32),
                ("n_ghost_ranks", C.c_int32), ("ghost_ranks", C.c_void_p),
                ("n_owner_ranks", C.c_int32), ("owner_ranks", C.c_void_p),
                ("n", C.c_int64), ("idx", C.c_void_p), ("remote_pos", C.c_void_p), ("entry_seg", C.c_void_p),
                ("size_local", C.c_int64), ("num_ghosts", C.c_int64),
                ("signal_pad", C.c_void_p), ("peer_pad", C.c_void_p), ("peer_delta", C.c_void_p),
                ("close_group", C.c_int32)]


def exported_symbols():
    names = list(UNTYPED)
    for base in _sigs():
        names += [f"{base}_f64", f"{base}_f32"]
    return names


def lib():
    """Load (building if needed) the shared library and set argtypes."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build

    if _build.needs_build():
        # missing or older than its sources: (re)build, so a stale in-tree .so never ships
        _build.build()
    lb = C.CDLL(LIB_PATH)
    lb.fus_abi_version.restype = I
    lb.fus_last_error.restype = C.c_char_p
    lb.fus_launch_count.restype = L
    lb.fus_reset_launch_count.restype = None
    lb.fus_halo_pad_bytes.restype, lb.fus_halo_pad_bytes.argtypes = L, [I]
    lb.fus_halo_create.restype, lb.fus_halo_create.argtypes = I, [C.POINTER(HaloDesc), C.POINTER(C.c_void_p)]
    lb.fus_halo_destroy.restype, lb.fus_halo_destroy.argtypes = I, [P]
    lb.fus_halo_num_shared.restype, lb.fus_halo_num_shared.argtypes = L, [P]
    lb.fus_halo_shared_mask.restype, lb.fus_halo_shared_mask.argtypes = P, [P]
    lb.fus_halo_shared_tail.restype, lb.fus_halo_shared_tail.argtypes = L, [P]
    lb.fus_halo_status.restype, lb.fus_halo_status.argtypes = I, [P]
    lb.fus_halo_signal_reverse.restype, lb.fus_halo_signal_reverse.argtypes = I, [P, P]
    lb.fus_halo_barrier.restype, lb.fus_halo_barrier.argtypes = I, [P, P]
    lb.fus_halo_wait_reverse.restype, lb.fus_halo_wait_reverse.argtypes = I, [P, P]
    lb.fus_stiffness_arm_halo_wait.restype, lb.fus_stiffness_arm_halo_wait.argtypes = I, [P, L]
    for base, args in _sigs().items():
        for sfx, ft in (("f64", C.c_double), ("f32", C.c_float)):
            fn = getattr(lb, f"{base}_{sfx}", None)
            if fn is None:
                continue
            fn.argtypes = [ft if a == "T" else a for a in args]
            fn.restype = I
    _lib = lb
    return lb


class FusError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().fus_last_error().decode(errors="replace")
        raise FusError(f"{what}: error {rc}: {msg}")


def sfx(dtype) -> str:
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return "f64"
    if dtype == np.float32:
        return "f32"
    raise TypeError(f"unsupported float type {dtype}")


def fn(base: str, dtype):
    return getattr(lib(), f"{base}_{sfx(dtype)}")


# --------------------------------------------------------------------------- #
# device-array plumbing: anything exposing __cuda_array_interface__
# (torch CUDA tensors, Numba DeviceNDArray, CuPy) is accepted, as in the
# reference where call sites pass Numba device arrays.
# --------------------------------------------------------------------------- #

_TORCH_DT = None


def _torch_dtypes():
    global _TORCH_DT
    if _TORCH_DT is None:
        import torch

        _TORCH_DT = {torch.float64: np.dtype(np.float64), torch.float32: np.dtype(np.float32),
                     torch.int32: np.dtype(np.int32), torch.int64: np.dtype(np.int64)}
    return _TORCH_DT


class DevArray:
    """(ptr, dtype, shape) view of a device array."""

    __slots__ = ("ptr", "dtype", "shape", "size")

    def __init__(self, a):
        t = type(a)
        if t.__module__.startswith("torch"):
            if not a.is_cuda:
                raise FusError("expected a CUDA tensor (there is no CPU path)")
            if not a.is_contiguous():
                raise FusError("expected a contiguous tensor")
            self.ptr = a.data_ptr()
            self.dtype = _torch_dtypes()[a.dtype]
            self.shape = tuple(a.shape)
        else:
            cai = getattr(a, "__cuda_array_interface__", None)
            if cai is None:
                raise FusError(f"expected a device array, got {t.__name__} (there is no CPU path)")
            if cai.get("strides") is not None:
                # must be C-contiguous
                st, item, shp = cai["strides"], np.dtype(cai["typestr"]).itemsize, cai["shape"]
                exp = []
                acc = item
                for d in reversed(shp):
                    exp.append(acc)
                    acc *= d
                if tuple(st) != tuple(reversed(exp)) and int(np.prod(shp)) > 1:
                    raise FusError("expected a C-contiguous device array")
            self.ptr = int(cai["data"][0])
            self.dtype = np.dtype(cai["typestr"])
            self.shape = tuple(cai["shape"])
        n = 1
        for d in self.shape:
            n *= int(d)
        self.size = n


def dev(a, dtype=None) -> DevArray:
    d = a if isinstance(a, DevArray) else DevArray(a)
    if dtype is not None and d.dtype != np.dtype(dtype):
        raise FusError(f"expected dtype {np.dtype(dtype)}, got {d.dtype}")
    return d


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
