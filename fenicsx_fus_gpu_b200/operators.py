"""
Operators - the reference's device-kernel surface on hand-written sm_100a CUDA
==============================================================================

Drop-in for ``/root/reference/cuda/operators.py``: same names, same argument
order, same accumulate-into-``y`` semantics, same ``kernel[grid, block](*args)``
launch syntax (the ``[grid, block]`` hint is accepted and ignored - the native
kernels size themselves to the 148 SMs).

    mass_operator[nb, 128](x, entity_constants, y, detJ_entity, entity_dofmap)     # :18-70
    stiffness_operator(P, float_type)[ncells, (n, n, n)](x, c, y, G, dofmap, dphi)  # :73-192
    axpy[nb, 1024](alpha, x, y); copy[..](a, b); fill[..](alpha, x)                 # :195-241
    pointwise_divide[..](a, b, c); square[..](a, b)                                 # :244-274

Array arguments are device arrays: anything exposing
``__cuda_array_interface__`` (torch CUDA tensors, Numba ``DeviceNDArray`` -
what the reference's call sites pass).  Launches are asynchronous on torch's
current stream.  There is no CPU path: host arrays raise.
"""

from __future__ import annotations

import numpy as np

from . import _lib
from ._lib import FUS_NO_ATOMICS, FUS_TABLES_RESIDENT, check, current_stream, dev, fn


class _Kernel:
    """``kernel[grid, block](*args)`` launch syntax of Numba CUDA kernels."""

    def __getitem__(self, _launch_config):
        return self

    def __call__(self, *args):  # pragma: no cover - abstract
        raise NotImplementedError


class _Mass(_Kernel):
    """``y[dm[e,i]] += x[dm[e,i]] * detJ[e,i] * c[e]`` - cuda/operators.py:18-70."""

    def __call__(self, x, entity_constants, y, detJ_entity, entity_dofmap):
        xd = dev(x)
        T = xd.dtype
        yd, cd, jd = dev(y, T), dev(entity_constants, T), dev(detJ_entity, T)
        dm = dev(entity_dofmap, np.int32)
        if len(dm.shape) != 2 or jd.shape != dm.shape:
            raise _lib.FusError(f"mass_operator: dofmap {dm.shape} / detJ {jd.shape} shape mismatch")
        if cd.size != dm.shape[0]:
            raise _lib.FusError("mass_operator: one constant per entity expected")
        if dm.shape[0] == 0:
            # Numba refuses a zero-size grid (the reference guards with `if bfacet_dofmap.any()`)
            raise ValueError("mass_operator: zero entities (empty launch)")
        check(fn("fus_mass", T)(xd.ptr, cd.ptr, yd.ptr, jd.ptr, dm.ptr, dm.shape[0], dm.shape[1],
                                current_stream()), "fus_mass")


mass_operator = _Mass()


class _CellKernel(_Kernel):
    """What every stiffness kernel checks: the degree and float type up front, and per call the
    dofmap shape, the sizes of the per-cell arrays and a non-empty launch, in that order."""

    name = ""

    def __init__(self, P: int, float_type):
        if not 2 <= int(P) <= 7:
            raise ValueError(f"{self.name}: degree {P} not in 2..7")
        self.P, self.n, self.float_type = int(P), int(P) + 1, np.dtype(float_type)
        _lib.sfx(self.float_type)  # validates

    def _dofmap(self, entity_dofmap, sizes):
        """The dofmap on the device.  ``sizes(ncells)`` lists (ok, message) for the other arrays."""
        dm = dev(entity_dofmap, np.int32)
        nd3 = self.n**3
        if len(dm.shape) != 2 or dm.shape[1] != nd3:
            raise _lib.FusError(f"{self.name}: dofmap must be (ncells, {nd3}), got {dm.shape}")
        for ok, msg in sizes(dm.shape[0]):
            if not ok:
                raise _lib.FusError(f"{self.name}: {msg}")
        if dm.shape[0] == 0:
            raise ValueError(f"{self.name}: zero cells (empty launch)")
        return dm


class _Stiffness(_CellKernel):
    """Sum-factorised stiffness action - cuda/operators.py:87-190."""

    name = "stiffness_operator"

    def __init__(self, P: int, float_type, colour_offsets=None):
        super().__init__(P, float_type)
        self.flags = 0
        self.colour_offsets = None
        if colour_offsets is not None:
            off = [int(v) for v in colour_offsets]
            if len(off) < 2 or off[0] != 0 or any(b < a for a, b in zip(off, off[1:])):
                raise ValueError("stiffness_operator: colour_offsets must be 0 = o_0 <= o_1 <= ... <= ncells")
            self.colour_offsets = off

    def __call__(self, x, entity_constants, y, G_entity, entity_dofmap, dphi):
        T = self.float_type
        xd, yd, cd, gd = dev(x, T), dev(y, T), dev(entity_constants, T), dev(G_entity, T)
        nd3 = self.n**3
        dm = self._dofmap(entity_dofmap, lambda nc: [(gd.size == nc * nd3 * 6, "G must be (ncells, n^3, 6)"),
                                                     (cd.size == nc, "one constant per cell expected")])
        if isinstance(dphi, np.ndarray):  # host table is fine: it goes to the constant bank
            tab = np.ascontiguousarray(dphi, dtype=T)
            if tab.size != self.n**2:
                raise _lib.FusError("stiffness_operator: dphi must be (n, n)")
            ptr = tab.ctypes.data
        else:
            td = dev(dphi, T)
            if td.size != self.n**2:
                raise _lib.FusError("stiffness_operator: dphi must be (n, n)")
            ptr = td.ptr
        f, st = fn("fus_stiffness", T), current_stream()
        if self.colour_offsets is None:
            check(f(xd.ptr, cd.ptr, yd.ptr, gd.ptr, dm.ptr, ptr, dm.shape[0], self.P, self.flags, st),
                  "fus_stiffness")
            return
        # deterministic path: the cells are sorted by colour, no two cells of a colour share
        # a dof, so each colour is one launch with plain read-modify-write instead of atomics
        off = self.colour_offsets
        if off[-1] != dm.shape[0]:
            raise _lib.FusError("stiffness_operator: colour_offsets[-1] must equal the number of cells")
        s = T.itemsize
        flags = self.flags | FUS_NO_ATOMICS
        for a, b in zip(off, off[1:]):
            if b > a:
                check(f(xd.ptr, cd.ptr + a * s, yd.ptr, gd.ptr + a * nd3 * 6 * s, dm.ptr + a * nd3 * 4, ptr,
                        b - a, self.P, flags, st), "fus_stiffness")
                flags |= FUS_TABLES_RESIDENT  # the derivative table went up with the first colour


def stiffness_operator(P, float_type, colour_offsets=None):
    """Returns the stiffness kernel for degree ``P`` and ``float_type``
    (cuda/operators.py:73-192).

    ``colour_offsets`` (optional, not in the reference): the cells have been
    permuted so that colour ``c`` occupies rows ``colour_offsets[c] :
    colour_offsets[c+1]`` of every per-cell array (``utils.colour_cells`` /
    ``utils.colour_order``).  The action then runs one atomics-free launch per
    colour and its result is bit-reproducible from run to run; the default
    (atomics) is faster on B200 - see DESIGN.md."""
    return _Stiffness(P, float_type, colour_offsets)


class _StiffnessAffine(_CellKernel):
    """The stiffness action on cells with a constant Jacobian: ``G[c, q, :] = weights[q] *
    Gc[c, :]`` (``precompute.compress_geometry``), so only 6 factors per cell are read."""

    name = "stiffness_operator_affine"

    def __call__(self, x, entity_constants, y, Gc, weights, entity_dofmap, dphi):
        T = self.float_type
        xd, yd, cd, gd, wd = dev(x, T), dev(y, T), dev(entity_constants, T), dev(Gc, T), dev(weights, T)
        nd3 = self.n**3
        dm = self._dofmap(entity_dofmap, lambda nc: [(gd.size == nc * 6 and cd.size == nc and wd.size == nd3,
                                                      "Gc (ncells, 6), constants (ncells,), weights (n^3,)")])
        tab = np.ascontiguousarray(dphi, dtype=T) if isinstance(dphi, np.ndarray) else None
        ptr = tab.ctypes.data if tab is not None else dev(dphi, T).ptr
        check(fn("fus_stiffness_affine", T)(xd.ptr, cd.ptr, yd.ptr, gd.ptr, wd.ptr, dm.ptr, ptr, dm.shape[0],
                                            self.P, 0, current_stream()), "fus_stiffness_affine")


def tensor_tables(dphi_1D, weights, float_type):
    """``(K1, w1)`` for the rectilinear kernels from the 1-D derivative table ``dphi_1D[q, i]``
    and the tensor quadrature weights (n^3,): ``w1`` with ``weights = w1 x w1 x w1`` and
    ``K1 = D^T diag(w1) D``, or None when the weights are not a tensor product."""
    D = np.asarray(dphi_1D, dtype=np.float64)
    n = D.shape[0]
    wq = np.asarray(weights, dtype=np.float64).reshape(n, n, n)
    tot = wq.sum()
    if not tot > 0:
        return None
    w1 = wq.sum(axis=(1, 2)) / tot ** (2.0 / 3.0)
    rtol = 1e-12 if np.dtype(float_type) == np.float64 else 1e-5
    if not np.allclose(w1[:, None, None] * w1[None, :, None] * w1[None, None, :], wq, rtol=rtol, atol=0.0):
        return None
    k1 = (D.T * w1[None, :]) @ D
    return np.ascontiguousarray(k1, dtype=float_type), np.ascontiguousarray(w1, dtype=float_type)


def rect_tables(dphi_1D, weights, float_type):
    """``tensor_tables``; raises when the weights are not a tensor product."""
    tabs = tensor_tables(dphi_1D, weights, float_type)
    if tabs is None:
        raise ValueError("rect_tables: the quadrature weights are not a tensor product")
    return tabs


class _StiffnessRect(_CellKernel):
    """The stiffness action on rectilinear cells (affine with diagonal ``Gc``): three decoupled
    1-D products with ``K1 = D^T diag(w1) D``.  Same call as ``stiffness_operator_affine``."""

    name = "stiffness_operator_rect"

    def __call__(self, x, entity_constants, y, Gc, weights, entity_dofmap, dphi):
        T = self.float_type
        xd, yd, cd, gd = dev(x, T), dev(y, T), dev(entity_constants, T), dev(Gc, T)
        dm = self._dofmap(entity_dofmap, lambda nc: [(gd.size == nc * 6 and cd.size == nc,
                                                      "Gc (ncells, 6), constants (ncells,)")])
        if not isinstance(dphi, np.ndarray) or not isinstance(weights, np.ndarray):
            raise _lib.FusError("stiffness_operator_rect: dphi and weights are host tables (numpy)")
        k1, w1 = rect_tables(dphi, weights, T)
        st = current_stream()
        check(fn("fus_set_rect_tables", T)(self.P, k1.ctypes.data, w1.ctypes.data, st), "fus_set_rect_tables")
        check(fn("fus_stiffness_rect", T)(xd.ptr, cd.ptr, yd.ptr, gd.ptr, dm.ptr, None, dm.shape[0], self.P,
                                          FUS_TABLES_RESIDENT, st), "fus_stiffness_rect")


def stiffness_operator_rect(P, float_type):
    """Stiffness kernel for rectilinear cells (not in the reference):
    ``k[grid, block](x, constants, y, Gc, weights, dofmap, dphi_1D)`` with host tables."""
    return _StiffnessRect(P, float_type)


class _StiffnessVertex(_CellKernel):
    """The stiffness action with the geometric factors recomputed in the kernel from the cells'
    trilinear maps (``csrc/stiffness_vertex.cu``): ``Tc`` from ``precompute.trilinear_coefficients``
    takes the place of the ``G`` table - 36 values per cell instead of 6 n^3."""

    name = "stiffness_operator_vertex"

    def __call__(self, x, entity_constants, y, Tc, points_1d, weights_1d, entity_dofmap, dphi):
        T = self.float_type
        xd, yd, cd, td = dev(x, T), dev(y, T), dev(entity_constants, T), dev(Tc, T)
        dm = self._dofmap(entity_dofmap, lambda nc: [(td.size == nc * 36 and cd.size == nc,
                                                      "Tc (ncells, 36), constants (ncells,)")])
        tabs = []
        for name, a, size in (("dphi", dphi, self.n * self.n), ("points_1d", points_1d, self.n),
                              ("weights_1d", weights_1d, self.n)):
            if not isinstance(a, np.ndarray) or a.size != size:
                raise _lib.FusError(f"stiffness_operator_vertex: {name} is a host table (numpy) of {size} entries")
            tabs.append(np.ascontiguousarray(a, dtype=T))
        D, x1, w1 = tabs
        st = current_stream()
        check(fn("fus_set_dphi", T)(self.P, D.ctypes.data, st), "fus_set_dphi")
        check(fn("fus_set_vertex_tables", T)(self.P, x1.ctypes.data, w1.ctypes.data, st), "fus_set_vertex_tables")
        check(fn("fus_stiffness_vertex", T)(xd.ptr, cd.ptr, yd.ptr, td.ptr, dm.ptr, None, dm.shape[0], self.P,
                                            FUS_TABLES_RESIDENT, st), "fus_stiffness_vertex")


def stiffness_operator_vertex(P, float_type):
    """Stiffness kernel with on-the-fly geometry (not in the reference, which streams ``G``):
    ``k[grid, block](x, constants, y, Tc, points_1d, weights_1d, dofmap, dphi_1D)``; ``Tc`` from
    ``precompute.trilinear_coefficients``, the three tables on the host."""
    return _StiffnessVertex(P, float_type)


def stiffness_operator_affine(P, float_type):
    """Stiffness kernel for affine cells (not in the reference):
    ``k[grid, block](x, constants, y, Gc, weights, dofmap, dphi)``."""
    return _StiffnessAffine(P, float_type)


def _vec3(name):
    class K(_Kernel):
        def __call__(self, a, b, c):
            ad = dev(a)
            T = ad.dtype
            bd, cd_ = dev(b, T), dev(c, T)
            n = min(ad.size, bd.size, cd_.size)
            check(fn(name, T)(ad.ptr, bd.ptr, cd_.ptr, n, current_stream()), name)

    return K()


def _vec2(name):
    class K(_Kernel):
        def __call__(self, a, b):
            ad = dev(a)
            T = ad.dtype
            bd = dev(b, T)
            check(fn(name, T)(ad.ptr, bd.ptr, min(ad.size, bd.size), current_stream()), name)

    return K()


class _Axpy(_Kernel):
    """``y = alpha*x + y`` - cuda/operators.py:195-209."""

    def __call__(self, alpha, x, y):
        xd = dev(x)
        T = xd.dtype
        yd = dev(y, T)
        check(fn("fus_axpy", T)(float(alpha), xd.ptr, yd.ptr, min(xd.size, yd.size),
                                current_stream()), "fus_axpy")


class _Fill(_Kernel):
    """``x[:] = alpha`` - cuda/operators.py:228-241."""

    def __call__(self, alpha, x):
        xd = dev(x)
        check(fn("fus_fill", xd.dtype)(float(alpha), xd.ptr, xd.size, current_stream()), "fus_fill")


axpy = _Axpy()
fill = _Fill()
copy = _vec2("fus_copy")  # b = a            cuda/operators.py:212-225
square = _vec2("fus_square")  # b = a*a      cuda/operators.py:261-274
pointwise_divide = _vec3("fus_pointwise_divide")  # c = a/b   cuda/operators.py:244-258
