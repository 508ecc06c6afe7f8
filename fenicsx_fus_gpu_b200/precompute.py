"""
Precompute - geometry tables, computed on the GPU
=================================================

Drop-in for ``/root/reference/cuda/precompute.py`` (== ``numba-cpu/precompute.py``;
C++ ``cpp/common/precompute.hpp:33-213``): same three functions, same argument
order, each fills a caller-allocated output in place.

The reference evaluates these with serial Numba loops on the host (64 M
quadrature points at the 33 M-dof box, 2e9 at 1 B dofs).  Here one sm_100a
thread handles one (entity, quadrature point) (``csrc/geometry.cu``).  Outputs
and inputs may be device arrays (used in place) or host numpy arrays (staged
through the device: the arithmetic always runs on the GPU, there is no CPU
path).
"""

from __future__ import annotations

import numpy as np

from . import _lib
from ._lib import check, current_stream, fn


def _to_dev(a, dtype):
    """Device tensor for ``a`` (numpy -> upload; device array -> as is)."""
    import torch

    if isinstance(a, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda(), True
    if isinstance(a, torch.Tensor):
        _lib.dev(a, dtype)  # CUDA, contiguous, and of the expected dtype: never reinterpret silently
        return a, False
    d = _lib.dev(a)  # __cuda_array_interface__ object
    if d.dtype != np.dtype(dtype):
        raise _lib.FusError(f"expected dtype {np.dtype(dtype)}, got {d.dtype}")
    return a, False


def _ptr(a):
    return _lib.dev(a).ptr


def _out(a):
    """(device buffer, host array to copy back into or None)"""
    import torch

    if isinstance(a, np.ndarray):
        tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[a.dtype]
        return torch.empty(a.shape, dtype=tdt, device="cuda"), a
    return a, None


def _finish(buf, host):
    if host is not None:
        host[...] = buf.cpu().numpy()


def compute_scaled_jacobian_determinant(detJ, mesh, num_cell, dphi, weights):
    """``detJ[c, q] = w_q |det J_c(x_q)|`` - cuda/precompute.py:76-112."""
    x_dofs, x_g = mesh
    buf, host = _out(detJ)
    T = _lib.dev(buf).dtype
    xd, _ = _to_dev(x_dofs, np.int32)
    xg, _ = _to_dev(x_g, T)
    dp, _ = _to_dev(dphi, T)
    w, _ = _to_dev(weights, T)
    nq = int(_lib.dev(w).size)
    check(fn("fus_geometry", T)(None, _ptr(buf), _ptr(xd), _ptr(xg), _ptr(dp), _ptr(w),
                                int(num_cell), nq, current_stream()), "fus_geometry")
    _finish(buf, host)


def compute_scaled_geometrical_factor(G, mesh, num_cell, dphi, weights):
    """``G[c, q, :] = w_q |det J| (J^-1 J^-T)`` upper triangle
    ``[00, 01, 02, 11, 12, 22]`` - cuda/precompute.py:115-163."""
    x_dofs, x_g = mesh
    buf, host = _out(G)
    T = _lib.dev(buf).dtype
    xd, _ = _to_dev(x_dofs, np.int32)
    xg, _ = _to_dev(x_g, T)
    dp, _ = _to_dev(dphi, T)
    w, _ = _to_dev(weights, T)
    nq = int(_lib.dev(w).size)
    check(fn("fus_geometry", T)(_ptr(buf), None, _ptr(xd), _ptr(xg), _ptr(dp), _ptr(w),
                                int(num_cell), nq, current_stream()), "fus_geometry")
    _finish(buf, host)


def compute_geometry(G, detJ, mesh, num_cell, dphi, weights):
    """Both tables in one pass over the cells (not in the reference, which
    makes two passes: cuda/demo_linear_box.py:245-253)."""
    x_dofs, x_g = mesh
    gbuf, ghost = _out(G)
    jbuf, jhost = _out(detJ)
    T = _lib.dev(gbuf).dtype
    xd, _ = _to_dev(x_dofs, np.int32)
    xg, _ = _to_dev(x_g, T)
    dp, _ = _to_dev(dphi, T)
    w, _ = _to_dev(weights, T)
    nq = int(_lib.dev(w).size)
    check(fn("fus_geometry", T)(_ptr(gbuf), _ptr(jbuf), _ptr(xd), _ptr(xg), _ptr(dp), _ptr(w),
                                int(num_cell), nq, current_stream()), "fus_geometry")
    _finish(gbuf, ghost)
    _finish(jbuf, jhost)


def compute_boundary_facets_scaled_jacobian_determinant(detJ_f, mesh, boundary_data, dphi_f, weights):
    """``detJ_f[i, q] = w_q |J_facet|`` for ``boundary_data[i] = (cell, local
    facet)`` - cuda/precompute.py:17-73."""
    x_dofs, x_g = mesh
    buf, host = _out(detJ_f)
    T = _lib.dev(buf).dtype
    xd, _ = _to_dev(x_dofs, np.int32)
    xg, _ = _to_dev(x_g, T)
    bd, _ = _to_dev(boundary_data, np.int32)
    dp, _ = _to_dev(dphi_f, T)
    w, _ = _to_dev(weights, T)
    nq = int(_lib.dev(w).size)
    nf = int(_lib.dev(bd).shape[0])
    if nf:
        check(fn("fus_facet_geometry", T)(_ptr(buf), _ptr(xd), _ptr(xg), _ptr(bd), _ptr(dp), _ptr(w),
                                          nf, nq, current_stream()), "fus_facet_geometry")
    _finish(buf, host)


def compress_geometry(G, detJ, weights, tol=None):
    """Affine-cell detection and compression (not in the reference).

    On a cell with a constant Jacobian the tables of cuda/precompute.py:76-163
    factor as ``G[c, q, :] = weights[q] * Gc[c, :]`` and ``detJ[c, q] = weights[q]
    * detJc[c]``.  Returns ``(affine, Gc, detJc)`` as device tensors: ``affine``
    (Nc,) int32 is 1 where every weight-normalised record of the cell lies within
    ``tol`` (relative; default 2048 machine epsilons = 4.5e-13 in float64 - the tables of an
    exactly affine cell carry rounding noise of ~N eps from ``dphi @ coords`` on an N^3 box,
    350 eps at N = 250) of the cell mean, ``Gc``
    (Nc, 6) and ``detJc`` (Nc,) are those means.  ``detJ`` may be None.
    ``G`` / ``detJ`` / ``weights`` are device arrays or numpy (uploaded)."""
    import torch

    Gd, _ = _to_dev(G, G.dtype) if isinstance(G, np.ndarray) else (G, False)
    T = _lib.dev(Gd).dtype
    tdt = torch.float64 if T == np.float64 else torch.float32
    w, _ = _to_dev(weights, T)
    nq = int(_lib.dev(w).size)
    nc = int(_lib.dev(Gd).size // (6 * nq))
    Jd = None
    if detJ is not None:
        Jd, _ = _to_dev(detJ, T)
    if tol is None:
        tol = 2048.0 * float(np.finfo(T).eps)
    Gc = torch.empty((nc, 6), dtype=tdt, device="cuda")
    detJc = torch.empty((nc,), dtype=tdt, device="cuda")
    affine = torch.zeros((nc,), dtype=torch.int32, device="cuda")
    check(fn("fus_compress_geometry", T)(_ptr(Gd), None if Jd is None else _ptr(Jd), _ptr(w), _ptr(Gc),
                                         _ptr(detJc) if Jd is not None else None, _ptr(affine), nc, nq,
                                         float(tol), current_stream()), "fus_compress_geometry")
    return affine, Gc, detJc


def compress_trilinear(Tc, tol=None):
    """Affine-cell detection and compression from the trilinear coefficients alone (the
    ``compress_geometry`` of a solver that holds no ``G`` table).

    ``Tc`` (Nc, 36) as ``trilinear_coefficients`` returns it: per cell and reference direction
    ``d`` the tangent ``t_d = Tc[d,0] + u Tc[d,1] + v Tc[d,2] + u v Tc[d,3]``.  A cell is affine
    when every non-constant coefficient vector ``Tc[d, 1..3]`` lies within ``tol`` (relative to
    the largest constant tangent ``Tc[d, 0]`` of the cell; default 2048 machine epsilons, as for
    ``compress_geometry``) of zero.  Returns ``(affine, Gc, detJc)`` as device tensors in the
    type of ``Tc``: ``affine`` (Nc,) int32, ``Gc = |det J| (J^T J)^-1`` (Nc, 6) in the order
    ``[G00 G01 G02 G11 G12 G22]`` and ``detJc = |det J|`` (Nc,), J the constant tangents.  The
    tables of an affine cell factor as ``G = w_q Gc``, ``detJ = w_q detJc`` for any quadrature
    rule, so no weights are needed.  Set-up only: plain torch in float64, on the device of ``Tc``
    (a CUDA tensor, a CPU tensor or numpy)."""
    import torch

    Tc = torch.as_tensor(Tc)
    if tol is None:
        tol = 2048.0 * float(torch.finfo(Tc.dtype).eps)
    t = Tc.to(torch.float64).reshape(-1, 3, 4, 3)
    t0, t1, t2 = t[:, 0, 0], t[:, 1, 0], t[:, 2, 0]
    scale = t[:, :, 0].abs().amax(dim=(1, 2))
    affine = (t[:, :, 1:].abs().amax(dim=(1, 2, 3)) <= tol * scale).to(torch.int32)
    # rows of adj J (as the GEO = 3 kernel forms them): G = (1/|det|) c_a . c_b
    c = torch.stack([torch.linalg.cross(t1, t2), torch.linalg.cross(t2, t0), torch.linalg.cross(t0, t1)], dim=1)
    det = (t0 * c[:, 0]).sum(-1).abs()
    ia, ib = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]
    Gc = (c[:, ia] * c[:, ib]).sum(-1) / det[:, None]
    return affine, Gc.to(Tc.dtype).contiguous(), det.to(Tc.dtype).contiguous()


def trilinear_expansion(dphi, points):
    """``M`` (3, 4, 8) float64 with ``dphi[d, q, :] = sum_m {1, u, v, u v}_m(points[q]) M[d, m, :]``,
    ``(u, v)`` the two reference coordinates other than ``d``: the bilinear expansion of the
    P1-geometry derivative table the reference tabulates from Basix (``cuda/demo_linear_box.py:232-239``).
    Fitted by least squares from the table itself, so no vertex-order or basis convention is assumed;
    raises when the table is not that of a trilinear map."""
    dphi = np.asarray(dphi, dtype=np.float64)
    pts = np.asarray(points, dtype=np.float64)
    if dphi.ndim != 3 or dphi.shape[0] != 3 or dphi.shape[2] != 8 or pts.shape != (dphi.shape[1], 3):
        raise _lib.FusError("trilinear_expansion: dphi (3, nq, 8) and points (nq, 3)")
    M = np.zeros((3, 4, 8))
    for d in range(3):
        a, b = [c for c in range(3) if c != d]
        u, v = pts[:, a], pts[:, b]
        A = np.stack([np.ones_like(u), u, v, u * v], axis=1)
        M[d] = np.linalg.lstsq(A, dphi[d], rcond=None)[0]
        if np.abs(A @ M[d] - dphi[d]).max() > 1e-6 * max(1.0, np.abs(dphi[d]).max()):
            raise _lib.FusError("trilinear_expansion: the derivative table is not that of a trilinear (8-vertex) geometry")
    return M


def trilinear_coefficients(mesh, num_cell, dphi, points, float_type=None):
    """``Tc`` (num_cell, 36) device tensor: per cell the 3 x 4 coefficient vectors of its tangents
    (``fus_trilinear_coeffs_*``; include/fus_b200.h) - what ``stiffness_operator_vertex`` takes in
    place of the ``G`` table of ``compute_scaled_geometrical_factor``.  ``mesh = (x_dofs, x_g)`` as
    for the other geometry functions (device arrays or numpy); ``dphi`` / ``points``: host tables."""
    import torch

    x_dofs, x_g = mesh
    T = np.dtype(x_g.dtype) if isinstance(x_g, np.ndarray) else _lib.dev(x_g).dtype
    if float_type is not None and np.dtype(float_type) != T:
        raise _lib.FusError(f"trilinear_coefficients: x_g is {T}, expected {np.dtype(float_type)}")
    if T not in (np.dtype(np.float64), np.dtype(np.float32)):
        raise _lib.FusError(f"trilinear_coefficients: x_g must be float32 or float64, got {T}")
    xg, _ = _to_dev(x_g, T)
    xd, _ = _to_dev(x_dofs, np.int32)
    tdt = torch.float64 if T == np.float64 else torch.float32
    M = torch.from_numpy(np.ascontiguousarray(trilinear_expansion(dphi, points), dtype=T)).cuda()
    Tc = torch.empty((int(num_cell), 36), dtype=tdt, device="cuda")
    check(fn("fus_trilinear_coeffs", T)(_ptr(Tc), _ptr(xd), _ptr(xg), _ptr(M), int(num_cell), current_stream()),
          "fus_trilinear_coeffs")
    return Tc
