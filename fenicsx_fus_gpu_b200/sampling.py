"""
Sampling - the demos' output path, kept on the device
=====================================================

The reference dumps pressure fields by copying the WHOLE solution vector to the
host every sampled step and calling ``dolfinx.fem.Function.eval`` there
(``/root/reference/cuda/demo_linear_piston.py:120-140, 555-582``,
``demo_nonlinear_bowl.py``), after locating the points with DOLFINx bounding-box
trees (``cuda/utils.py:117-154`` ``compute_eval_params``).  Here

* ``compute_eval_params(mesh, points, float_type)`` keeps that name, argument
  order and return value ``(points_on_proc, cells)`` but works on any mesh of
  trilinear hexahedra given as ``(x_dofs, x_g)`` (a uniform bin grid over the
  cell boxes + a Newton pull-back instead of the DOLFINx tree);
* ``PointEvaluator`` tabulates the 1-D Lagrange values at the points' reference
  coordinates once and then evaluates ``u`` at all points with one kernel launch
  (``csrc/sampling.cu``): only the sampled values cross PCIe;
* ``ElementReceiver`` integrates ``u`` over the facets of each element of a
  transducer array (the signal each element receives), with two launches and a
  deterministic reduction.

DOLFINx is absent from this image, so parity with ``Function.eval`` is pinned
through known answers only (polynomials of degree <= P are reproduced exactly;
tests/test_host_logic.py, tests/test_gpu_sampling.py).
"""

from __future__ import annotations

import numpy as np

from . import _lib
from ._lib import check, current_stream, fn


def _mesh_arrays(mesh):
    if isinstance(mesh, (tuple, list)):
        x_dofs, x_g = mesh
    else:
        x_dofs, x_g = mesh.x_dofs, mesh.x_g
    return np.asarray(x_dofs), np.asarray(x_g, dtype=np.float64)


def _p1_basis(X):
    """Trilinear basis (m, 8) and its gradient (m, 8, 3) at reference points X (m, 3);
    vertex v sits at ((v & 1), (v >> 1) & 1, (v >> 2) & 1) - the P1 order of
    ``substrate.p1_hex_basis``."""
    m = X.shape[0]
    phi = np.ones((m, 8))
    dphi = np.ones((m, 8, 3))
    for v in range(8):
        for d in range(3):
            bit = (v >> d) & 1
            f = X[:, d] if bit else 1.0 - X[:, d]
            df = 1.0 if bit else -1.0
            phi[:, v] *= f
            for e in range(3):
                dphi[:, v, e] *= df if e == d else f
    return phi, dphi


def pull_back(coords, points, tol=1e-14, maxit=30):
    """Reference coordinates X (m, 3) in [0, 1]^3 of physical ``points`` (m, 3) inside
    hexahedra with vertex coordinates ``coords`` (m, 8, 3): Newton on the trilinear map
    (one step is exact on an affine cell).  Returns ``(X, converged)``."""
    coords = np.asarray(coords, dtype=np.float64)
    points = np.asarray(points, dtype=np.float64)
    m = points.shape[0]
    X = np.full((m, 3), 0.5)
    ok = np.zeros(m, bool)
    if m == 0:
        return X, ok
    scale = np.maximum(np.ptp(coords, axis=1).max(axis=1), 1e-300)
    for _ in range(maxit):
        phi, dphi = _p1_basis(X)
        r = np.einsum("mv,mvd->md", phi, coords) - points
        ok = np.abs(r).max(axis=1) <= tol * scale
        if ok.all():
            break
        J = np.einsum("mvd,mve->mde", coords, dphi)  # dx_d / dX_e
        with np.errstate(all="ignore"):
            try:
                dX = np.linalg.solve(J, r[:, :, None])[:, :, 0]
            except np.linalg.LinAlgError:
                dX = np.zeros_like(r)
        dX[~np.isfinite(dX)] = 0.0
        X = np.clip(X - dX, -2.0, 3.0)  # keep runaway iterates (point far outside the cell) bounded
    return X, ok


def compute_eval_params(mesh, points, float_type, padding=1e-12):
    """Evaluation parameters for ``PointEvaluator`` - cuda/utils.py:117-154.

    ``points`` is (3, npts) as in the reference.  Returns ``points_on_proc``
    ((m, 3) ``float_type``: the points that lie in a local cell, in input order)
    and ``cells`` (list of m local cell indices; the lowest-numbered colliding cell
    when a point sits on a shared face).  ``mesh`` is anything with ``x_dofs``
    (Nc, 8) / ``x_g`` (nv, 3) attributes, or that pair."""
    x_dofs, x_g = _mesh_arrays(mesh)
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64).T)
    npts, nc = pts.shape[0], x_dofs.shape[0]
    if npts == 0 or nc == 0:
        return np.zeros((0, 3), dtype=float_type), []
    cc = x_g[x_dofs]  # (Nc, 8, 3)
    lo, hi = cc.min(axis=1), cc.max(axis=1)
    g0, g1 = lo.min(axis=0), hi.max(axis=0)
    span = np.maximum(g1 - g0, 1e-300)
    pad = padding * span.max()
    nb = np.maximum(1, np.floor(np.cbrt(nc) * span / span.max()).astype(np.int64))
    bs = span / nb

    def bins(x):
        return np.clip(np.floor((x - g0) / bs).astype(np.int64), 0, nb - 1)

    # (bin, cell) pairs: every bin a cell's padded box overlaps
    blo, bhi = bins(lo - pad), bins(hi + pad)
    ext = (bhi - blo).max(axis=0) + 1
    pb, pc = [], []
    cells_all = np.arange(nc)
    for a in range(int(ext[0])):
        for b in range(int(ext[1])):
            for c in range(int(ext[2])):
                off = np.array([a, b, c])
                msk = np.all(blo + off <= bhi, axis=1)
                if msk.any():
                    bb = blo[msk] + off
                    pb.append((bb[:, 0] * nb[1] + bb[:, 1]) * nb[2] + bb[:, 2])
                    pc.append(cells_all[msk])
    pb, pc = np.concatenate(pb), np.concatenate(pc)
    order = np.lexsort((pc, pb))  # by bin, cells ascending inside a bin
    pb, pc = pb[order], pc[order]
    nbins = int(np.prod(nb))
    start = np.searchsorted(pb, np.arange(nbins + 1))

    inside = np.all((pts >= g0 - pad) & (pts <= g1 + pad), axis=1)
    pbin = bins(pts)
    pbin = (pbin[:, 0] * nb[1] + pbin[:, 1]) * nb[2] + pbin[:, 2]
    ncand = np.where(inside, start[pbin + 1] - start[pbin], 0)
    found = np.full(npts, -1, dtype=np.int64)
    eps = 1e-9
    for k in range(int(ncand.max(initial=0))):
        todo = np.nonzero((found < 0) & (ncand > k))[0]
        if todo.size == 0:
            break
        cand = pc[start[pbin[todo]] + k]
        p = pts[todo]
        box = np.all((p >= lo[cand] - pad) & (p <= hi[cand] + pad), axis=1)
        todo, cand, p = todo[box], cand[box], p[box]
        if todo.size == 0:
            continue
        X, ok = pull_back(cc[cand], p)
        hit = ok & np.all((X >= -eps) & (X <= 1.0 + eps), axis=1)
        found[todo[hit]] = cand[hit]
    sel = found >= 0
    return np.ascontiguousarray(pts[sel], dtype=float_type), [int(c) for c in found[sel]]


def lagrange_1d(nodes, x):
    """``l_i(x)`` (m, n) of the Lagrange basis on ``nodes`` (n,), first barycentric form;
    exact Kronecker delta at the nodes."""
    nodes = np.asarray(nodes, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    diff = nodes[:, None] - nodes[None, :]
    np.fill_diagonal(diff, 1.0)
    bw = 1.0 / np.prod(diff, axis=1)
    d = x[:, None] - nodes[None, :]
    exact = d == 0.0
    d = np.where(exact, 1.0, d)
    full = np.prod(np.where(exact, 1.0, d), axis=1)  # prod over the non-coincident nodes
    out = bw[None, :] * full[:, None] / d
    hit = exact.any(axis=1)
    out[hit] = exact[hit].astype(np.float64)
    return out


def reference_basis(mesh, points_on_proc, cells, nodes_1d):
    """``(X, phi)``: reference coordinates (m, 3) of the points in their cells and the
    1-D Lagrange values phi (m, 3, n) there (``nodes_1d`` in dof order: ``ElementTables.pts_1d``)."""
    x_dofs, x_g = _mesh_arrays(mesh)
    cells = np.asarray(cells, dtype=np.int64)
    pts = np.asarray(points_on_proc, dtype=np.float64).reshape(-1, 3)
    X, ok = pull_back(x_g[x_dofs[cells]], pts)
    if not ok.all():
        raise ValueError(f"{int((~ok).sum())} point(s) could not be pulled back to their cell")
    phi = np.stack([lagrange_1d(nodes_1d, X[:, d]) for d in range(3)], axis=1)
    return X, phi


class PointEvaluator:
    """``u`` at fixed points, on the device: ``ev = PointEvaluator(P, float_type, dofmap, mesh,
    x_eval, cell_eval, nodes_1d); values = ev(u_d)`` replaces ``u_n_d.copy_to_host(u_n);
    u_n_.eval(x_eval, cell_eval)`` (cuda/demo_linear_piston.py:564-570).  ``dofmap`` is the
    tensor-product dofmap (device tensor or numpy); ghost entries of ``u`` must be current
    (forward halo) where sampled cells touch them, as in the reference (:566)."""

    def __init__(self, P, float_type, dofmap, mesh, points_on_proc, cells, nodes_1d):
        import torch

        if not torch.cuda.is_available():
            raise _lib.FusError("no CUDA device: this package has no CPU path")
        self.P, self.n = int(P), int(P) + 1
        self.dtype = np.dtype(float_type)
        self.T = torch.float64 if self.dtype == np.float64 else torch.float32
        self.npts = len(cells)
        self.X, phi = reference_basis(mesh, points_on_proc, cells, nodes_1d)
        if phi.shape[2] != self.n:
            raise ValueError("nodes_1d must hold P + 1 nodes")
        self.phi = torch.from_numpy(np.ascontiguousarray(phi, dtype=self.dtype)).cuda()
        self.cells = torch.from_numpy(np.asarray(cells, dtype=np.int32)).cuda()
        self.dofmap = dofmap if isinstance(dofmap, torch.Tensor) else torch.from_numpy(
            np.ascontiguousarray(dofmap, dtype=np.int32)).cuda()
        if self.dofmap.dtype != torch.int32 or self.dofmap.shape[1] != self.n**3:
            raise _lib.FusError(f"dofmap must be int32 (ncells, {self.n**3})")
        self.out = torch.empty(self.npts, dtype=self.T, device="cuda")
        self._host = None

    def __call__(self, u, out=None):
        """Device tensor (npts,) of the values; asynchronous on the current stream."""
        out = self.out if out is None else out
        ud = _lib.dev(u, self.dtype)
        check(fn("fus_eval_points", self.dtype)(ud.ptr, self.dofmap.data_ptr(), self.cells.data_ptr(),
                                                self.phi.data_ptr(), out.data_ptr(), self.npts, self.P,
                                                current_stream()), "fus_eval_points")
        return out

    def record(self, u, out, step_dev, step_base, first, rows):
        """``u`` into row ``step_base + step_dev - first`` of ``out`` (rows, npts), indices read on the
        device (``step_dev`` may be None); nothing is written when that row is outside
        ``[0, rows)``.  The sum of ``__call__``: the same bits.  Asynchronous on the current stream."""
        ud = _lib.dev(u, self.dtype)
        check(fn("fus_record_points", self.dtype)(
            ud.ptr, self.dofmap.data_ptr(), self.cells.data_ptr(), self.phi.data_ptr(), out.data_ptr(), self.npts,
            self.P, None if step_dev is None else step_dev.data_ptr(), step_base.data_ptr(), int(first), int(rows),
            current_stream()), "fus_record_points")
        return out

    def to_host(self, u):
        """Values as numpy: one launch + one device->host copy of npts values (pinned)."""
        import torch

        if self._host is None:
            self._host = torch.empty(self.npts, dtype=self.T).pin_memory()
        self._host.copy_(self(u), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._host.numpy().copy()


def reduce_by_key(key, vals):
    """``(ukey, sums)``: the sorted distinct values of ``key`` (int64 device tensor) and, for every
    tensor of ``vals`` (one value per entry of ``key``), the sum of its values per key.  Each sum runs
    in the order of the entries: a stable sort, then one pass per position inside a key (at most one
    add per key and pass), so no sum depends on the order of atomics."""
    import torch

    key, order = torch.sort(key, stable=True)
    vals = [v[order] for v in vals]
    ukey, inv, counts = torch.unique_consecutive(key, return_inverse=True, return_counts=True)
    pos = torch.arange(key.numel(), dtype=torch.int64, device=key.device) - (torch.cumsum(counts, 0) - counts)[inv]
    sums = [torch.zeros(ukey.numel(), dtype=v.dtype, device=v.device) for v in vals]
    for j in range(int(counts.max().item()) if counts.numel() else 0):
        sel = pos == j
        for acc, v in zip(sums, vals):
            acc.index_add_(0, inv[sel], v[sel])
    return ukey, sums


#: entries per chunk of a receiver's rows: the work of one warp in the first launch
CHUNK = 256


class ElementReceiver:
    """The signal each element of a transducer array receives: ``r_e = int_{Gamma_e} u dS`` over the
    facets of element e, on the device.  ``bfacet_dofmap`` (nf, n^2) and ``detJ_f`` (nf, n^2) are a
    facet group as ``problem.facet_group`` returns it, ``elements`` holds one element index in
    ``[0, num_elements)`` per facet row.

    The rows are built once: for every element and dof, ``w`` = the sum of ``detJ_f`` over the
    element's facets that contain the dof (``reduce_by_key``, facet order), element-major and sorted
    by dof, cut into chunks of ``CHUNK`` entries (``fus_record_elements_*``).  With partitioned meshes
    each rank integrates over the facets of its own cells: summing ``receiver(u)`` (or ``areas``) over
    the ranks gives the integral (the area) up to rounding.  A rank without any of the facets gets
    zeros."""

    def __init__(self, float_type, bfacet_dofmap, detJ_f, elements, num_elements):
        import torch

        if not torch.cuda.is_available():
            raise _lib.FusError("no CUDA device: this package has no CPU path")
        self.dtype = np.dtype(float_type)
        self.T = torch.float64 if self.dtype == np.float64 else torch.float32
        self.E = int(num_elements)
        if self.E < 1:
            raise ValueError(f"ElementReceiver: num_elements must be >= 1, got {self.E}")

        def dev(a, dt):
            t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
            return t.to(device="cuda", dtype=dt).contiguous()

        bdm, dJ, ids = dev(bfacet_dofmap, torch.int32), dev(detJ_f, self.T), dev(elements, torch.int64)
        if bdm.dim() != 2 or tuple(dJ.shape) != tuple(bdm.shape):
            raise ValueError(f"ElementReceiver: bfacet_dofmap {tuple(bdm.shape)} and detJ_f {tuple(dJ.shape)} must "
                             "both be (facets, n^2)")
        nf = int(bdm.shape[0])
        if ids.dim() != 1 or ids.numel() != nf:
            raise ValueError(f"ElementReceiver: elements has {ids.numel()} entries, the facet group {nf} rows")
        if nf:
            lo, hi = int(ids.min().item()), int(ids.max().item())
            if lo < 0 or hi >= self.E:
                raise ValueError(f"ElementReceiver: elements must lie in [0, {self.E}), got [{lo}, {hi}]")
            if int(bdm.min().item()) < 0:
                raise ValueError("ElementReceiver: negative dof in bfacet_dofmap")
        # u must hold every dof the facets touch
        self.ndofs = int(bdm.max().item()) + 1 if bdm.numel() else 0
        i64 = dict(dtype=torch.int64, device="cuda")
        if bdm.numel():
            key = ids.repeat_interleave(bdm.shape[1]) * self.ndofs + bdm.reshape(-1).to(torch.int64)
            ukey, (w,) = reduce_by_key(key, [dJ.reshape(-1)])
        else:
            ukey, w = torch.zeros(0, **i64), torch.zeros(0, dtype=self.T, device="cuda")
        nnz = int(ukey.numel())
        if nnz >= 2**31:
            raise ValueError(f"ElementReceiver: {nnz} entries do not fit the int32 chunk table")
        elem = ukey // max(self.ndofs, 1)
        self.dof = (ukey - elem * self.ndofs).to(torch.int32)
        self.w = w.contiguous()
        count = torch.bincount(elem, minlength=self.E)
        nch = (count + CHUNK - 1) // CHUNK
        self.elem_chunk = torch.cat([torch.zeros(1, **i64), torch.cumsum(nch, 0)]).to(torch.int32)
        self.nchunks = int(self.elem_chunk[-1].item())
        ce = torch.repeat_interleave(torch.arange(self.E, **i64), nch)  # element of every chunk
        j = torch.arange(self.nchunks, **i64) - self.elem_chunk[:-1].to(torch.int64)[ce]
        start = torch.cumsum(count, 0) - count
        self.chunk_beg = torch.cat([start[ce] + j * CHUNK, torch.tensor([nnz], **i64)]).to(torch.int32)
        self.partial = torch.empty(max(self.nchunks, 1), dtype=self.T, device="cuda")  # scratch of the first launch
        self.out = torch.zeros(self.E, dtype=self.T, device="cuda")
        self.areas = self(torch.ones(max(self.ndofs, 1), dtype=self.T, device="cuda")).clone()

    @property
    def nbytes(self):
        """Device bytes of the rows, the chunk tables and the scratch."""
        return sum(t.numel() * t.element_size() for t in (self.dof, self.w, self.elem_chunk, self.chunk_beg,
                                                          self.partial, self.out))

    def _args(self, u):
        ud = _lib.dev(u, self.dtype)
        if ud.size < self.ndofs:
            raise ValueError(f"ElementReceiver: u has {ud.size} entries, the facets reach dof {self.ndofs - 1}")
        return (ud.ptr, self.dof.data_ptr(), self.w.data_ptr(), self.chunk_beg.data_ptr(), self.elem_chunk.data_ptr(),
                self.partial.data_ptr())

    def __call__(self, u, out=None):
        """Device tensor (E,) of this rank's ``r_e``; asynchronous on the current stream."""
        out = self.out if out is None else out
        if self.nchunks == 0:
            return out.zero_()  # no facet here: this rank's part of every integral is 0
        check(fn("fus_eval_elements", self.dtype)(*self._args(u), out.data_ptr(), self.nchunks, self.E,
                                                  current_stream()), "fus_eval_elements")
        return out

    def record(self, u, out, step_dev, step_base, first, rows):
        """``r_e`` into row ``step_base + step_dev - first`` of ``out`` (rows, E), indices read on the
        device (``step_dev`` may be None); nothing is written when that row is outside ``[0, rows)``.
        The sums of ``__call__``: the same bits.  Asynchronous on the current stream."""
        check(fn("fus_record_elements", self.dtype)(
            *self._args(u), out.data_ptr(), self.nchunks, self.E, None if step_dev is None else step_dev.data_ptr(),
            step_base.data_ptr(), int(first), int(rows), current_stream()), "fus_record_elements")
        return out
