"""
Solver - the explicit RK4 hot loops, fused
==========================================

``LinearSpectral3D`` replaces the time loop of
``/root/reference/cuda/demo_linear_box.py:487-567`` (and ``demo_linear_piston.py``;
CPU twin ``numba-cpu/demo_linear_box.py:389-459``; C++ ``LinearSpectral3D`` in
``cpp/common/Linear.hpp:43-344`` whose name and ``init`` / ``rk4`` methods it keeps).
``WesterveltSpectral3D`` replaces ``cuda/demo_nonlinear_bowl.py:529-657`` (and
``demo_nonlinear_box.py``).

What the reference does per RK stage with ~17 kernel launches, >= 8 device
synchronisations and 3-5 host-staged MPI rounds becomes

    [halo forward (un, vn) - one grouped NCCL round]
    stiffness (scatter fused)  + boundary-facet diagonals (+ Westervelt cell mass pair)
    [halo reverse (b[, m])]
    close  (b/m, u,v updates, next stage's un/vn, b = 0  - ONE pass over the vectors)

i.e. 3 launches per stage on one GPU, no host synchronisation, and a whole
time step (4 stages) is captured once as a CUDA graph and replayed.  Steps
"ping-pong": the first stage reads the base state directly (a_0 = 0), the last
one leaves the new state in the accumulators, and base / accumulator buffers
swap roles between steps (two graphs, replayed alternately) - 41 vector passes
per step instead of 48, same arithmetic bit for bit.  Source
amplitudes come from a device table indexed by a device step counter, so a
replay needs no host work at all.

Multi-GPU (peer-memory halo, ``scatterer.P2PHaloExchange``): the cells are split at set-up
into *interior* ones and *interface* ones (those touching a ghost dof), and a stage becomes

    main stream                                        exchange stream
    one-warp wait for the neighbours' puts (they were
      issued beside the previous close: no stall)
    stiffness (split_mode "two" / "fused": interior
      cells first, the wait only before the interface cells)
    boundary terms (+ "my ghost sums are ready" signal)
    close on the dofs nobody shares               ||   one-warp wait for the neighbours' signals;
                                                       ONE kernel: gather their ghost sums, close
                                                       the shared dofs, put the next stage input

so neither the forward nor the reverse exchange of cuda/demo_linear_box.py:536-553 is ever
waited for on the critical path, and there is no barrier: the ordering is per-neighbour
epoch flags raised by the kernels themselves (csrc/halo.cu).

Reference quirks (SURVEY.md section 8a): the source is evaluated at the stage
time ``tn`` as the numba-cpu / C++ paths do (Q1; ``source_at_stage_time=False``
gives the CUDA demos' behaviour); the solution is ``u`` (Q2); vector kernels
run over owned + ghost entries and ghost ``m`` keeps its partial sums (Q3).
"""

from __future__ import annotations

from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import FUS_TABLES_RESIDENT, check, current_stream, fn
from .operators import tensor_tables
from .sampling import reduce_by_key

# a contiguous range of (permuted) cells that one kernel launch covers:
# kind 0 rectilinear, 1 affine, 2 streamed G, 3 trilinear (geometry rebuilt from Tc); c0/n cell range;
# g0 first row of the streamed G / detJ arrays (kind 3: of Tc); ninterior: the first ninterior cells
# of the range touch no ghost dof (peer-memory halo: the launch waits for the forward exchange only
# before its remaining, interface, cells)
Seg = namedtuple("Seg", "kind c0 n g0 ninterior")
# a recorder (record_points: a PointEvaluator, record_elements: an ElementReceiver): its rows, the window
# [first, first + rows) of global step indices and the device int64 holding the global index of the call's
# step 0
_Recorder = namedtuple("_Recorder", "ev out first rows base")
_OUTSIDE = -(1 << 62)  # a base step index that puts every step of a run before any window
KIND_SUFFIX = ("_rect", "_affine", "", "_vertex")  # cell-kernel symbol fus_<form><suffix> per Seg.kind

A_RUNGE = (0.0, 0.5, 0.5, 1.0)
B_RUNGE = (1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0)
C_RUNGE = (0.0, 0.5, 0.5, 1.0)


def _torch():
    import torch

    return torch


def _tdt(dtype):
    torch = _torch()
    return {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[np.dtype(dtype)]


def _dev(a, dtype=None):
    """Device tensor of ``a`` (numpy is uploaded, device tensors pass through)."""
    torch = _torch()
    if isinstance(a, torch.Tensor):
        t = a if a.is_cuda else a.cuda()
    elif isinstance(a, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    else:
        t = torch.as_tensor(a, device="cuda")
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def linear_source(t, f0, p0, c0, alpha=4.0):
    """``g(t)`` of cuda/demo_linear_box.py:511-530 (numba-cpu :341-358).  ``t`` may be an array
    (one time per array element); a scalar ``t`` gives the same bits either way."""
    T = 1.0 / f0
    window = np.where(t < T * alpha, 0.5 * (1.0 - np.cos(f0 * np.pi * t / alpha)), 1.0)
    return window * p0 * 2.0 * np.pi * f0 / c0 * np.cos(2.0 * np.pi * f0 * t), 0.0


def westervelt_source(t, f0, p0, c0, alpha=4.0):
    """``g(t), dg/dt`` of cuda/demo_nonlinear_bowl.py:556-594.  ``t`` may be an array, as for
    ``linear_source``."""
    T = 1.0 / f0
    w0 = 2.0 * np.pi * f0
    ramp = t < T * alpha
    window = np.where(ramp, 0.5 * (1.0 - np.cos(f0 * np.pi * t / alpha)), 1.0)
    dwindow = np.where(ramp, 0.5 * np.pi * f0 / alpha * np.sin(f0 * np.pi * t / alpha), 0.0)
    g = window * 2.0 * p0 * w0 / c0 * np.cos(w0 * t)
    dg = dwindow * 2.0 * p0 * w0 / c0 * np.cos(w0 * t) - window * 2.0 * p0 * w0**2 / c0 * np.sin(w0 * t)
    return g, dg


class _RK4:
    """State vectors, boundary diagonals, graph capture, the stage sequence and the step loop
    shared by the linear and Westervelt solvers.

    ``source_elements`` (phased-array sources): one element index in ``[0, E)`` per row of the
    source facet group, ``E = num_elements`` (default: the largest index + 1; give it on every rank
    of a partitioned run, where a rank may see only some elements or none).  ``source(t)`` then
    returns ``(g, dg)`` as arrays of shape ``(E,)``, one waveform per element, and every source
    launch reads the element's amplitudes from a device table of ``8 E`` values per step
    (``fus_boundary_terms_elements_*``).  The table takes ``rows * 8 E * itemsize`` bytes: about
    80 MB for E = 1024 over 1219 float64 steps.

    A solver class states its cell-kernel form (``form``: the kernels ``fus_<form>[_rect|_affine]``,
    and ``_operands``: their leading arguments for a cell range) and its close (``_close_name``:
    the bulk close kernel, ``_close_variant``: its variant of ``fus_rk_close_shared``, ``_masses``:
    the (m, m0, m2, m5) it reads)."""

    westervelt = False
    integrator = "rk4"

    def __init__(self, P, float_type, ndofs, dofmap, G, dphi_1D, halo=None, source=None,
                 source_at_stage_time=True, use_graph=True, geometry="stream", weights=None,
                 split_cells=True, trilinear=None, source_elements=None, num_elements=None):
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.FusError("no CUDA device: this package has no CPU path")
        self.P = int(P)
        self.n = self.P + 1
        self.dtype = np.dtype(float_type)
        self.T = _tdt(self.dtype)
        self.ndofs = int(ndofs)
        self.dofmap = _dev(dofmap, torch.int32)
        self.ncells = int(self.dofmap.shape[0])
        # geometry = "stream": G (and detJ) are read in full every stage, as the reference does;
        # "auto": cells whose Jacobian is constant (precompute.compress_geometry) keep 6 (+1)
        # values instead of 6 (+1) n^3 and go through the affine kernels, the others are streamed;
        # "vertex": the same split from the trilinear coefficients alone (precompute.compress_trilinear),
        # the other cells rebuild their geometry in the kernel from 36 values each
        # (``trilinear = (Tc, points_1d, weights_1d)``): no (Nc, n^3) table is ever held
        if geometry not in ("stream", "auto", "vertex"):
            raise ValueError("geometry must be 'stream', 'auto' or 'vertex'")
        if geometry != "stream" and weights is None:
            raise ValueError(f"geometry='{geometry}' needs the quadrature weights (n^3,)")
        if geometry == "vertex" and trilinear is None:
            raise ValueError("geometry='vertex' needs trilinear=(Tc, points_1d, weights_1d)")
        if geometry != "vertex" and G is None:
            raise ValueError(f"geometry='{geometry}' needs G")
        self.G = _dev(G, self.T) if geometry != "vertex" else None
        self._Tc = self._vertex_tables = None
        if geometry == "vertex":
            Tc, x1, w1 = trilinear
            self._Tc = _dev(Tc, self.T)
            host = lambda a: np.ascontiguousarray(a.cpu().numpy() if isinstance(a, torch.Tensor) else a,  # noqa: E731
                                                  dtype=self.dtype)
            self._vertex_tables = (host(x1), host(w1))
        self.halo = halo
        self.source = source
        self.source_at_stage_time = bool(source_at_stage_time)
        self.use_graph = bool(use_graph)
        self._dphi_host = np.ascontiguousarray(
            dphi_1D.cpu().numpy() if isinstance(dphi_1D, torch.Tensor) else dphi_1D, dtype=self.dtype)
        z = lambda: torch.zeros(self.ndofs, dtype=self.T, device="cuda")  # noqa: E731
        # With the peer-memory halo (scatterer.P2PHaloExchange) the exchanged vectors live in
        # peer-addressable memory and only their owned part is updated locally: the ghost
        # slots are written by the neighbours.
        self._m_accum = False  # Westervelt "cells" form: m is accumulated per stage (and reverse-exchanged)
        self.p2p = bool(getattr(halo, "p2p", False))
        # peer-memory halo: launch interior cells (no ghost dof) while the forward exchange is in
        # flight and interface cells after it (False: one launch after the exchange, for A/B runs)
        self.split_cells = bool(split_cells)
        # How a stage's stiffness launches wait for the forward exchange (measured on 2 and 8 B200s,
        # profiles/r02_multigpu_timeline.md):
        #   "none"  (default) a one-warp wait kernel, then every cell in one launch.  The neighbours'
        #           put of stage i+1 is issued beside the ~0.5 ms close of stage i, so in steady state
        #           the wait returns at once; fastest.
        #   "two"   interior cells in one launch, interface cells (waiting first) in a second one:
        #           a whole stage of slack against a late neighbour, for a second pipeline fill/drain.
        #   "fused" one launch, every CTA waits in-kernel before its first interface batch: the
        #           conditional barrier in the persistent loop stops the compiler from hoisting the
        #           prefetch loads, which costs more (+25 us per launch) than the second launch.
        self.split_mode = "none"
        self.nupd = int(halo.N) if self.p2p else self.ndofs  # entries the vector kernels update
        zx = halo.alloc if self.p2p else z
        # the reference's 14 vectors (cuda/demo_linear_box.py:380-385, 464-471)
        # shrink to 8: two (u, v) pairs that alternate between "base state of this step" and
        # "accumulator" (= the next step's base), ku un b m  (vn lives in ku; g, u_n, v_n,
        # kv fused away).  The base pair is the stage-0 input, so it is halo-exchanged too.
        self._uv = [(zx(), zx()), (zx(), zx())]
        self._parity = 0  # _uv[_parity] is the base state (the solution between steps)
        self.ku, self.un, self.b = zx(), zx(), zx()
        self.m = zx()
        self._zx = zx
        self.step_dev = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.gtab = None
        self.t = 0.0
        self.nstep = 0
        self._graph = None  # [graph of a step with parity 0, with parity 1]
        self._graph_dt = None
        self._graph_tab = None
        self._graph_rec = None
        # "points" / "elements" -> _Recorder (empty: no record launch anywhere).  Replaced, never mutated,
        # when a recorder is attached or detached, so `is` against _graph_rec tells when to recapture
        self._recs = {}
        self.graph_error = None
        self._opened = False
        self._bdofs = None
        self._src = self._src2 = self._absb = None
        # phased-array source (None: one waveform for every source facet)
        self.num_elements = None
        self._elem_ids = self._erow = self._eelem = self._ew = self._ew2 = self._etab1 = None
        if source_elements is not None:
            ids = _dev(source_elements, torch.int64)
            if ids.dim() != 1:
                raise ValueError("source_elements must be one element index per source facet row")
            lo, hi = (int(ids.min().item()), int(ids.max().item())) if ids.numel() else (0, -1)
            if num_elements is None:
                if hi < 0:
                    raise ValueError("source_elements is empty: give num_elements")
                num_elements = hi + 1
            self.num_elements = int(num_elements)
            if self.num_elements < 1 or lo < 0 or hi >= self.num_elements:
                raise ValueError(f"source_elements must lie in [0, {self.num_elements}), got [{lo}, {hi}]")
            self._elem_ids = ids
        elif num_elements is not None:
            raise ValueError("num_elements needs source_elements")
        self.probe = None  # list: (start, stop) CUDA events around every stage-kernel launch (eager mode)
        self.geometry = geometry
        self._weights = None if weights is None else _dev(weights, self.T)
        self.nrect = 0  # number of rectilinear cells (affine, diagonal Gc)
        self.naff = 0  # number of affine cells (rectilinear ones included)
        self.ntri = 0  # number of trilinear cells (geometry="vertex": the cells that are not affine)
        self.detJ = self.Gc = self.detJc = None
        self._rect_tables = None
        self.cell_perm = None
        # cell ranges, one launch each (per geometry kind; interior cells first inside a range)
        self._segs = [Seg(3 if geometry == "vertex" else 2, 0, self.ncells, 0, self.ncells)]
        self.ninterface = 0

    # the solution between steps (device tensors; write initial data into them before rk4)
    @property
    def u(self):
        return self._uv[self._parity][0]

    @property
    def v(self):
        return self._uv[self._parity][1]

    @property
    def _rec(self):
        """The point recorder, or None."""
        return self._recs.get("points")

    # ---- set-up helpers ------------------------------------------------------
    def _set_tables(self):
        check(fn("fus_set_dphi", self.dtype)(self.P, self._dphi_host.ctypes.data, current_stream()),
              "fus_set_dphi")
        if self._rect_tables is not None:
            k1, w1 = self._rect_tables
            check(fn("fus_set_rect_tables", self.dtype)(self.P, k1.ctypes.data, w1.ctypes.data, current_stream()),
                  "fus_set_rect_tables")
        if self._vertex_tables is not None:
            x1, w1 = self._vertex_tables
            check(fn("fus_set_vertex_tables", self.dtype)(self.P, x1.ctypes.data, w1.ctypes.data, current_stream()),
                  "fus_set_vertex_tables")

    def _mass(self, x, coeff, y, detJ, dofmap):
        if dofmap.shape[0]:
            check(fn("fus_mass", self.dtype)(x.data_ptr(), coeff.data_ptr(), y.data_ptr(), detJ.data_ptr(),
                                             dofmap.data_ptr(), dofmap.shape[0], dofmap.shape[1],
                                             current_stream()), "fus_mass")

    def _cell_mass(self, x, coeff, y, detJ):
        """Lumped cell mass y += M(coeff; x): from the detJ table, or in vertex mode from Tc."""
        if self._Tc is None:
            self._mass(x, coeff, y, detJ, self.dofmap)
        elif self.ncells:
            self._set_tables()
            check(fn("fus_mass_vertex", self.dtype)(x.data_ptr(), coeff.data_ptr(), y.data_ptr(), self._Tc.data_ptr(),
                                                    self.dofmap.data_ptr(), self.ncells, self.P, current_stream()),
                  "fus_mass_vertex")

    def _facets(self, bfacet_dofmap, detJ_f, facet_coeff):
        """(bfacet_dofmap, detJ_f, facet_coeff) of a boundary facet group on the device, or None
        when the group is empty."""
        if bfacet_dofmap is None:
            return None
        bd = _dev(bfacet_dofmap, _torch().int32)
        return (bd, _dev(detJ_f, self.T), _dev(facet_coeff, self.T)) if bd.shape[0] else None

    def _boundary_setup(self, **groups):
        """``groups``: slot ("src", "src2", "absb") -> facet group of ``_facets`` or None.  Builds
        the compact unique-dof list and the diagonals = the facet mass operator applied to ones
        (cuda/demo_linear_box.py:546-551); with a phased-array source, the per-element rows of
        the source slots instead (``_element_rows``)."""
        torch = _torch()
        src = {slot: groups.pop(slot, None) for slot in ("src", "src2")} if self.num_elements is not None else {}
        nonempty = {slot: g for slot, g in {**groups, **src}.items() if g is not None}
        groups = {slot: g for slot, g in groups.items() if g is not None}
        if not nonempty:
            self._bdofs = torch.zeros(0, dtype=torch.int32, device="cuda")
        else:
            self._bdofs = torch.unique(torch.cat([g[0].reshape(-1) for g in nonempty.values()])).to(torch.int32).contiguous()
        idx = self._bdofs.to(torch.int64)
        ones = torch.ones(self.ndofs, dtype=self.T, device="cuda")
        for slot, (bdm, dJ, coeff) in groups.items():
            tmp = torch.zeros(self.ndofs, dtype=self.T, device="cuda")
            self._mass(ones, coeff, tmp, dJ, bdm)
            setattr(self, "_" + slot, tmp[idx].contiguous())
        if self.num_elements is not None:
            self._element_rows(src["src"], src["src2"])

    def _facet_diagonal(self, group):
        """Owner-complete diagonal of a facet group (``_facets``): its facet mass operator applied to
        ones, reverse-exchanged once (peer-addressable with the peer-memory halo).  The compact lists
        of ``_boundary_setup`` hold this rank's partial sums instead, which is what an assembly needs;
        a close that applies the diagonal pointwise needs the complete one."""
        torch = _torch()
        d = torch.zeros(self.ndofs, dtype=self.T, device="cuda") if not self.p2p else self._zx()
        if group is not None:
            bd, dJ, fc = group
            self._mass(torch.ones(self.ndofs, dtype=self.T, device="cuda"), fc, d, dJ, bd)
        if self.halo is not None:
            self.halo.reverse(d)
        return d

    def _element_rows(self, src, src2):
        """CSR rows over ``_bdofs`` of the phased-array source: for every boundary dof, one entry
        (element, w[, w2]) per element whose facets contain it, w = the facet coefficient times
        detJ_f summed over those facets (the facet mass diagonal of the element).  Built on the
        device: the facet rows are expanded into (dof, element, weight) entries, sorted by
        (dof, element) and reduced per key in facet order (``sampling.reduce_by_key``)."""
        torch = _torch()
        E = self.num_elements
        nf = 0 if src is None else int(src[0].shape[0])
        if self._elem_ids.numel() != nf:
            raise ValueError(f"source_elements has {self._elem_ids.numel()} entries, the source facet group {nf} rows")
        i64 = dict(dtype=torch.int64, device="cuda")
        if nf:
            bdm, dJ, coeff = src
            key = bdm.reshape(-1).to(torch.int64) * E + self._elem_ids.repeat_interleave(bdm.shape[1])
            ukey, sums = reduce_by_key(key, [(c[:, None] * dJ).reshape(-1)
                                             for c in (coeff, None if src2 is None else src2[2]) if c is not None])
        else:
            ukey, sums = torch.zeros(0, **i64), [torch.zeros(0, dtype=self.T, device="cuda")] * (1 + (src2 is not None))
        row = torch.searchsorted(ukey // E, self._bdofs.to(torch.int64))
        self._erow = torch.cat([row, torch.tensor([ukey.numel()], **i64)]).to(torch.int32).contiguous()
        # the kernel takes non-null element arrays whenever the dof list is not empty
        pad = lambda t: (t if t.numel() else torch.zeros(1, dtype=t.dtype, device="cuda")).contiguous()  # noqa: E731
        self._eelem = pad((ukey % E).to(torch.int32))
        self._ew = pad(sums[0])
        self._ew2 = pad(sums[1]) if len(sums) > 1 else None

    def _setup_geometry(self, detJ, cell_arrays):
        """Order the cells for the launches of a stage and build the launch ranges.

        geometry='auto' classifies the cells (rectilinear / affine / streamed G), geometry='vertex'
        the same way from Tc (rectilinear / affine / trilinear); the peer-memory halo splits them
        into interior and interface cells (those with a ghost dof).  Cells are sorted by
        (interface, kind), every per-cell array follows (``cell_arrays``: attribute names of (Nc,) /
        (Nc, n^3) tensors; the dofmap, G, detJ and Tc are handled here), G / detJ are kept for the
        streamed cells only, Tc for the trilinear ones.  Summation order inside the atomics aside, a
        cell permutation does not change the result."""
        torch = _torch()
        nc = self.ncells
        if nc == 0:
            return
        other = 3 if self.geometry == "vertex" else 2  # the kind of a cell that is not affine
        kind = torch.full((nc,), other, dtype=torch.int32, device="cuda")
        Gc = detJc = None
        if self.geometry != "stream":
            from . import precompute as pre

            if self.geometry == "vertex":
                affine, Gc, detJc = pre.compress_trilinear(self._Tc)
            else:
                affine, Gc, detJc = pre.compress_geometry(self.G, detJ, self._weights)
            # rectilinear = affine with a diagonal Gc (off-diagonal factors at rounding-noise level)
            # no cell takes the rectilinear path unless the rule is a tensor product
            tabs = tensor_tables(self._dphi_host, self._weights.cpu().numpy(), self.dtype)
            tol = 2048.0 * float(np.finfo(self.dtype).eps)
            diag = Gc[:, [0, 3, 5]].abs().amax(dim=1)
            off = Gc[:, [1, 2, 4]].abs().amax(dim=1)
            rect = (affine > 0) & (off <= tol * diag) if tabs is not None else torch.zeros_like(affine, dtype=torch.bool)
            kind = torch.where(rect, 0, torch.where(affine > 0, 1, other)).to(torch.int32)
            self.naff = int((kind < 2).sum().item())
            self.ntri = int((kind == 3).sum().item())
            self.nrect = int((kind == 0).sum().item())
            if self.nrect:
                self._rect_tables = tabs
        split = self.p2p and self.split_cells
        if split:
            iface = (self.dofmap >= self.halo.N).any(dim=1)
            self.ninterface = int(iface.sum().item())
        else:
            iface = torch.zeros(nc, dtype=torch.bool, device="cuda")
        key = kind * 2 + iface.to(torch.int32)  # rect [interior | interface], affine [..], streamed / trilinear [..]
        counts = torch.bincount(key, minlength=8).cpu().tolist()
        perm = None
        if not bool((key[1:] >= key[:-1]).all().item()):
            perm = torch.argsort(key, stable=True)  # original order kept inside every range
            self.cell_perm = perm
            self.dofmap = self.dofmap[perm].contiguous()
            for name in cell_arrays:
                setattr(self, name, getattr(self, name)[perm].contiguous())
            if Gc is not None:
                Gc, detJc = Gc[perm], detJc[perm]
        if perm is not None or self.naff:
            # G / detJ (Tc) rows of the streamed (trilinear) cells only, in launch order (the caller's
            # tensors are not touched)
            rows = torch.arange(nc, device="cuda") if perm is None else perm
            rows = rows[kind[rows] == other]
            if self._Tc is not None:
                self._Tc = self._Tc[rows].contiguous() if rows.numel() else None
            else:
                self.G = self.G[rows].contiguous() if rows.numel() else None
            if detJ is not None:
                self.detJ = detJ[rows].contiguous() if rows.numel() else None
        if self.naff:
            self.Gc = Gc.contiguous()
            self.detJc = detJc.contiguous() if self._m_accum else None
        # launch ranges: one per geometry kind
        self._segs, c0, g0 = [], 0, 0
        for k in (0, 1, 2, 3):
            nint, nif = counts[2 * k], counts[2 * k + 1]
            if nint + nif:
                self._segs.append(Seg(k, c0, nint + nif, g0, nint if split else nint + nif))
            c0 += nint + nif
            if k >= 2:
                g0 += nint + nif

    # ---- stage pieces --------------------------------------------------------
    def _probed(self, launch):
        """Run ``launch()``; with ``self.probe`` a list (eager mode only), bracket it with CUDA
        events on the launching stream so a benchmark can read the kernel's duration in situ."""
        if self.probe is None:
            launch()
            return
        torch = _torch()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        self.probe.append((e0, e1))

    def _ptr(self, t):
        return None if t is None else t.data_ptr()

    def _boundary(self, stage, g, dg, use_table, vn, signal=False, consume=False):
        """b += g*src + dg*src2 + vn*absb on the boundary dofs.  ``signal`` (peer-memory halo): the
        launch also raises the "ghost sums complete" epoch (and happens even without boundary dofs).
        Phased-array source: the element amplitudes come from the step's table row, or without the
        table from the one-row table ``_load_eager_row`` wrote (``g``, ``dg`` are not used)."""
        nb = int(self._bdofs.numel())
        if not nb and not signal:
            return
        if self.num_elements is not None:
            tab, step = (self.gtab, self.step_dev) if use_table else (self._etab1, None)
            args = (self.b.data_ptr(), vn.data_ptr(), self._bdofs.data_ptr() if nb else None, self._erow.data_ptr(),
                    self._eelem.data_ptr(), self._ew.data_ptr(), self._ptr(self._ew2), self._ptr(self._absb),
                    tab.data_ptr(), self._ptr(step), self.num_elements, stage, nb)
            name = "fus_boundary_terms_elements_signal" if signal else "fus_boundary_terms_elements"
            extra = (self.halo.handle,) if signal else ()
            tail = (int(consume),) if signal else ()
            check(fn(name, self.dtype)(*extra, *args, *tail, current_stream()), name)
            return
        args = (self.b.data_ptr(), vn.data_ptr(), self._bdofs.data_ptr() if nb else None, self._ptr(self._src),
                self._ptr(self._src2), self._ptr(self._absb), float(g), float(dg),
                self.gtab.data_ptr() if use_table else None,
                self.step_dev.data_ptr() if use_table else None, 8, 2 * stage, nb, current_stream())
        if signal:
            check(fn("fus_boundary_terms_signal", self.dtype)(self.halo.handle, *args[:-1], int(consume), args[-1]),
                  "fus_boundary_terms_signal")
        else:
            check(fn("fus_boundary_terms", self.dtype)(*args), "fus_boundary_terms")

    def _open_first(self):
        """b = 0 before the first stage (cuda/demo_linear_box.py:541); the stage-0 input is the
        base state itself (:491-508 at a_0 = 0: un = u0, vn = v0), nothing is copied."""
        self.b.zero_()
        if self._m_accum:
            self.m.zero_()
        if self.p2p:
            self.halo.barrier()  # nobody's first put may land before this rank is set up
        self._opened = True

    def _sptr(self, t, row):
        """Device address of row ``row`` of a per-cell tensor (no view objects on the launch path)."""
        return t.data_ptr() + int(row) * t.stride(0) * t.element_size()

    def _launches(self, wait):
        """(range, armed first-interface cell or None) per launch of a stage.  Peer-memory halo: a
        launch waits in-kernel, before its first interface batch, for the neighbours' puts (without
        the cell split: before its first batch); ``split_mode == "two"`` launches the interior cells
        unarmed and the interface cells armed from their first batch."""
        out = []
        for sg in self._segs:
            if not wait:
                out.append((sg, None))
            elif not self.split_cells:
                out.append((sg, 0))
            elif self.split_mode == "two" and 0 < sg.ninterior < sg.n:
                out.append((Seg(sg.kind, sg.c0, sg.ninterior, sg.g0, sg.ninterior), None))
                g1 = sg.g0 + (sg.ninterior if sg.kind >= 2 else 0)
                out.append((Seg(sg.kind, sg.c0 + sg.ninterior, sg.n - sg.ninterior, g1, 0), 0))
            else:
                out.append((sg, sg.ninterior if sg.ninterior < sg.n else None))
        return out

    def _arm(self, first):
        if first is not None:
            self.halo.arm_stiffness_wait(first)

    def _cell_kernels(self, x, vn, wait=False):
        """The cell-kernel launches of a stage: ``fus_<form><KIND_SUFFIX>`` over every cell range, with
        the form's operands, then the range's geometry (G or Gc; detJ or detJc when the form carries
        the cell-mass pair; the quadrature weights for affine cells; Tc alone for trilinear cells),
        then the common tail."""
        st, sp = current_stream(), self._sptr
        for sg, first in self._launches(wait):
            if sg.kind == 3:
                geo = (sp(self._Tc, sg.g0),)
            else:
                G, dJ, row = (self.G, self.detJ, sg.g0) if sg.kind == 2 else (self.Gc, self.detJc, sg.c0)
                geo = (sp(G, row), sp(dJ, row)) if self._m_accum else (sp(G, row),)
            if sg.kind == 1:
                geo += (self._weights.data_ptr(),)
            self._arm(first)
            name = f"fus_{self.form}{KIND_SUFFIX[sg.kind]}"
            check(fn(name, self.dtype)(*self._operands(x, vn, sg.c0), *geo, sp(self.dofmap, sg.c0), None, sg.n,
                                       self.P, FUS_TABLES_RESIDENT, st), name)

    def _assemble(self, x, vn, wait=False):
        """The cell kernels of a stage as one group for ``probe``."""
        self._probed(lambda: self._cell_kernels(x, vn, wait))

    def _assemble_exchanged(self, stage, g, dg, use_table, x, vn, record=False):
        """b (, m) of a stage with the halo as blocking rounds: forward exchange of the input, cell
        kernels, [the record launch,] boundary terms, reverse exchange of the sums."""
        if self.halo is not None:
            self.halo.forward(x, vn)
        self._assemble(x, vn)
        if record:
            self._record(x, use_table)
        self._boundary(stage, g, dg, use_table, vn)
        if self.halo is not None:
            self.halo.reverse(*((self.b, self.m) if self._m_accum else (self.b,)))

    def _source_at(self, stage, dt, t, use_table):
        """(g, dg) of ``stage`` of the step from ``t``, evaluated on the host; zeros when the
        launches read them from the device table."""
        if use_table or self.source is None:
            return 0.0, 0.0
        return self.source(t + C_RUNGE[stage] * dt if self.source_at_stage_time else t)

    def _stage(self, stage, dt, t, use_table, base, acc):
        """The launches of one stage of the step from ``base`` into ``acc``, under any halo.

        Peer-memory halo (module docstring), main stream: a one-warp wait for the neighbours' puts
        (issued beside the previous stage's close, so normally long since landed; ``split_mode``
        selects the variants that launch the interior cells before waiting); the cell kernels; the
        boundary terms, whose last block signals "my ghost sums are complete"; the close on the
        dofs nobody shares.  Exchange stream, beside that close: a one-warp wait for the
        neighbours' signals, then ONE kernel that gathers their ghost sums, closes the shared dofs
        and puts the next stage input into the neighbours' ghost slots.

        Ordering across GPUs: every wait depends only on signals the neighbours raise from kernels
        that are stream-ordered after kernels of EARLIER phases of this rank, so the step can be
        captured and replayed as a graph without deadlock.  A neighbour's put of stage i+1 is
        issued by the kernel that gathered (and cleared) my ghost sums of stage i, so its FWD epoch
        also says the ghost accumulators are clean.

        Recorders (``record_points``, ``record_elements``): stage 0 records the base ``u``, the state
        at the start of the step, with the record launches after the cell kernels and before the
        boundary launch.  There its
        ghost entries are current: the forward exchange (or the wait for the neighbours' puts) came
        first, and in split modes "two" / "fused" the cell kernels that waited in-kernel precede the
        record launch on this stream.  And no neighbour can overwrite them yet: a neighbour puts into
        this rank's ghost slots only from a close that waits for the signal of this rank's stage-0
        boundary launch, which comes after the record launch."""
        g, dg = self._source_at(stage, dt, t, use_table)
        # stage input: the base state itself in stage 0 (a_0 = 0), un / vn (= ku) afterwards; with the
        # peer-memory halo it is on its way to (or already in) the ghost slots: put there by
        # begin_steps() or by the previous stage's close of the shared dofs
        x, vn = base if stage == 0 else (self.un, self.ku)
        record = stage == 0 and bool(self._recs)
        h = self.halo
        if not self.p2p:
            self._assemble_exchanged(stage, g, dg, use_table, x, vn, record)
            self._close(stage, dt, use_table, base, acc)
            return
        # (the leapfrog step always waits before its launches)
        in_kernel = self.integrator == "rk4" and self.split_cells and self.split_mode in ("two", "fused")
        if in_kernel:
            h.sync_point()
        else:
            h.wait_forward()
        self._assemble(x, vn, wait=in_kernel)
        if record:
            self._record(x, use_table)
        self._boundary(stage, g, dg, use_table, vn, signal=True, consume=in_kernel)
        h.fork()
        with h.side():
            h.wait_reverse()
            self._close_shared(stage, dt, base, acc)
        self._close(stage, dt, use_table, base, acc, **h.bulk_close())
        h.join()

    def _enqueue_step(self, dt, t, use_table, parity=None):
        """The launches of one RK4 step whose base state is ``_uv[parity]`` (default: the current
        one); the new state is left in ``_uv[1 - parity]``.  Does not flip ``_parity``."""
        parity = self._parity if parity is None else parity
        for i in range(4):
            self._stage(i, dt, t, use_table, self._uv[parity], self._uv[1 - parity])

    def begin_steps(self):
        """Peer-memory halo: send the current state to the neighbours' ghost slots before a run
        of steps (every step then ends by putting the next one's input).  Collective; a no-op
        otherwise."""
        if self.p2p:
            self.halo.barrier()  # the neighbours are done reading the ghost values about to be replaced
            self.halo.put(self.u, self.v)

    def end_steps(self):
        """Consume the put the last step of a run left pending (keeps puts and waits paired)."""
        if self.p2p:
            self.halo.wait_forward()

    def _close_args(self, stage, dt, base, acc):
        """(u, v, u0, v0 pointers, bdt, adt_next, next_mode) of the close kernel for ``stage``:
        3 = first stage of a ping-pong step, 1 = chained, 4 = last stage."""
        mode = 3 if stage == 0 else (4 if stage == 3 else 1)
        adt = 0.0 if stage == 3 else A_RUNGE[stage + 1] * dt
        return (acc[0].data_ptr(), acc[1].data_ptr(), base[0].data_ptr(), base[1].data_ptr(),
                B_RUNGE[stage] * dt, adt, mode)

    def _close(self, stage, dt, count_step, base, acc, skip=None, n=None):
        """Close of ``stage`` on the dofs this rank updates alone: every owned one, or beside
        ``_close_shared`` the prefix ``n`` / the dofs outside the ``skip`` mask."""
        u, v, u0, v0, bdt, adt, mode = self._close_args(stage, dt, base, acc)
        masses = [t.data_ptr() for t in self._masses() if t is not None]
        check(fn(self._close_name, self.dtype)(
            u, v, u0, v0, self.ku.data_ptr(), None, self.un.data_ptr(), self.b.data_ptr(), *masses, bdt, adt, mode,
            self.nupd if n is None else n, self.step_dev.data_ptr() if count_step else None, skip, current_stream()),
            self._close_name)

    def _close_shared(self, stage, dt, base, acc):
        """Close of ``stage`` on the shared dofs (peer-memory halo): gathers the neighbours' ghost
        sums, closes and puts the next stage input into their ghost slots."""
        u, v, u0, v0, bdt, adt, mode = self._close_args(stage, dt, base, acc)
        ku, un = (self.ku.data_ptr(), self.un.data_ptr()) if self.integrator == "rk4" else (None, None)
        check(fn("fus_rk_close_shared", self.dtype)(
            self.halo.handle, self._close_variant, 1, 1, u, v, u0, v0, ku, un, self.b.data_ptr(),
            *(self._ptr(t) for t in self._masses()), bdt, adt, mode, current_stream()), "fus_rk_close_shared")

    def _record(self, u, use_table, recs=None):
        """The record launches: ``u`` into every recorder's (or every one of ``recs``) row of global step
        ``base + step_dev`` (without the table: ``base``)."""
        for r in self._recs.values() if recs is None else recs:
            r.ev.record(u, r.out, self.step_dev if use_table else None, r.base, r.first, r.rows)

    def _set_bases(self, step):
        for r in self._recs.values():
            r.base.fill_(step)

    def _record_last(self):
        """After a call: one eager record of the state after its last step, by every recorder whose
        window holds that row.  The ghost entries of ``u`` are current: with the peer-memory halo
        ``end_steps`` has waited for the neighbours' puts; the NCCL-shaped halo exchanges ``u`` forward
        here, once (every rank must then record the same windows: the exchange is collective)."""
        due = [r for r in self._recs.values() if 0 <= self.nstep - r.first < r.rows]
        if not due:
            return
        if self.halo is not None and not self.p2p:
            self.halo.forward(self.u)
        for r in due:
            r.base.fill_(self.nstep)
        self._record(self.u, False, due)

    def _attach(self, kind, ev, first, rows, width, fill):
        """Attach (``ev`` not None) or detach the recorder of ``kind``; returns its rows."""
        torch = _torch()
        if ev is None:
            if kind in self._recs:
                self._recs = {k: r for k, r in self._recs.items() if k != kind}
            return None
        out = torch.full((rows, width), fill, dtype=self.T, device="cuda")
        self._recs = {**self._recs, kind: _Recorder(ev, out, first, rows, torch.zeros(1, dtype=torch.int64,
                                                                                      device="cuda"))}
        return out

    # ---- public --------------------------------------------------------------
    def record_points(self, evaluator, first=0, rows=1):
        """Record ``u`` at the points of ``evaluator`` (``sampling.PointEvaluator``) at every step,
        inside the captured step graphs: returns a device tensor ``(rows, evaluator.npts)`` of the
        solver's float type, filled with NaN, whose row ``j`` receives ``u`` after ``first + j`` steps
        counted from ``init()`` (``nstep``).  After any ``rk4`` / ``step_eager`` call every row with
        ``first + j <= nstep`` is filled, bit-identical to ``evaluator(u)`` on the same state.
        ``record_points(None)`` detaches the recorder; ``init()`` keeps it and its rows.  With a halo,
        every rank attaches a recorder with the same window (its own points, possibly none)."""
        if evaluator is None:
            return self._attach("points", None, 0, 1, 0, 0.0)
        first, rows = int(first), int(rows)
        if np.dtype(evaluator.dtype) != self.dtype:
            raise ValueError(f"record_points: the evaluator is {np.dtype(evaluator.dtype)}, the solver {self.dtype}")
        if int(evaluator.P) != self.P:
            raise ValueError(f"record_points: the evaluator has degree {evaluator.P}, the solver {self.P}")
        if first < 0 or rows < 1:
            raise ValueError(f"record_points: need first >= 0 and rows >= 1, got first = {first}, rows = {rows}")
        return self._attach("points", evaluator, first, rows, evaluator.npts, float("nan"))

    def record_elements(self, receiver, first=0, rows=1):
        """Record what the elements of an array receive (``sampling.ElementReceiver``) at every step,
        inside the captured step graphs: returns a device tensor ``(rows, receiver.E)`` of the solver's
        float type, filled with NaN, whose row ``j`` receives this rank's ``r_e`` (the integral of ``u``
        over element e's facets of this rank) after ``first + j`` steps counted from ``init()``; a rank
        without any receiver facet gets zeros.  After any ``rk4`` / ``step_eager`` call every row with
        ``first + j <= nstep`` is filled, bit-identical to ``receiver(u)`` on the same state.
        ``record_elements(None)`` detaches the receiver; a point recorder may be attached beside it.
        With a halo, every rank attaches a receiver with the same window and E; the sum over ranks is
        the caller's (one ``all_reduce`` after the run)."""
        if receiver is None:
            return self._attach("elements", None, 0, 1, 0, 0.0)
        first, rows = int(first), int(rows)
        if np.dtype(receiver.dtype) != self.dtype:
            raise ValueError(f"record_elements: the receiver is {np.dtype(receiver.dtype)}, the solver {self.dtype}")
        if receiver.ndofs > self.ndofs:
            raise ValueError(f"record_elements: the receiver reaches dof {receiver.ndofs - 1}, the solver has "
                             f"{self.ndofs} dofs")
        if first < 0 or rows < 1:
            raise ValueError(f"record_elements: need first >= 0 and rows >= 1, got first = {first}, rows = {rows}")
        return self._attach("elements", receiver, first, rows, receiver.E,
                            float("nan") if receiver.nchunks else 0.0)

    def init(self):
        """Zero initial state (cpp/common/Linear.hpp:146-154)."""
        for t in (*self._uv[0], *self._uv[1], self.ku, self.un, self.b):
            t.zero_()
        self.t = 0.0
        self.nstep = 0
        self._opened = False

    def source_table(self, t0, dt, nsteps):
        """(nsteps, 8) table of (g, dg) per stage, times accumulated as the
        reference does (``t += dt``).  Phased-array source: (nsteps, 8 E), per stage the E values
        of g, then the E values of dg."""
        if self.num_elements is not None:
            return self._element_table(t0, dt, nsteps)
        tab = np.zeros((max(nsteps, 1), 8), dtype=self.dtype)
        t = t0
        for k in range(nsteps):
            for i in range(4):
                tab[k, 2 * i], tab[k, 2 * i + 1] = self._source_at(i, dt, t, False)
            t += dt
        return tab

    def _element_table(self, t0, dt, nsteps):
        E = self.num_elements
        tab = np.zeros((max(nsteps, 1), 4, 2, E), dtype=self.dtype)
        t = t0
        for k in range(nsteps if self.source is not None else 0):
            for i in range(4):
                g, dg = self._source_at(i, dt, t, False)
                if np.shape(g) != (E,) or np.shape(dg) not in ((E,), ()):
                    raise ValueError(f"source(t) must return (g, dg) of shape ({E},), got {np.shape(g)} and "
                                     f"{np.shape(dg)}")
                tab[k, i, 0], tab[k, i, 1] = g, dg
            t += dt
        return tab.reshape(tab.shape[0], 8 * E)

    def _load_eager_row(self, t, dt):
        """Phased-array source without the table: the element amplitudes of the four stages of the
        step from ``t`` into a one-row device table of its own (the step table and its graph are
        not touched)."""
        torch = _torch()
        row = torch.from_numpy(self._element_table(t, dt, 1))
        if self._etab1 is None:
            self._etab1 = torch.zeros(row.shape, dtype=self.T, device="cuda")
        self._etab1.copy_(row)

    def rk4(self, t0, dt, nsteps):
        """``nsteps`` RK4 steps of size ``dt`` from ``t0``; returns the final time.
        The device is NOT synchronised on return (stream ordered)."""
        torch = _torch()
        self._set_tables()
        self.t = float(t0)
        if not self._opened:
            self._open_first()
        if nsteps <= 0:
            return self.t
        self._load_table(self.source_table(self.t, dt, nsteps))
        self.step_dev.zero_()
        if self.use_graph and (self._graph_dt != dt or self._graph_tab != self.gtab.data_ptr()
                               or self._graph_rec is not self._recs):
            self._capture(dt)
        self._set_bases(self.nstep)  # stream-ordered: the graphs' arguments stay as captured
        if self.use_graph:
            self.begin_steps()
            for _ in range(nsteps):
                self._replay_step(dt)
            self.end_steps()
        else:
            self.begin_steps()
            for k in range(nsteps):
                self._enqueue_step(dt, 0.0, True)
                self._parity ^= 1
            self.end_steps()
        for _ in range(nsteps):
            self.t += dt
        self.nstep += nsteps
        self._record_last()
        return self.t

    def _load_table(self, tab):
        """Copy a host source table into the persistent device table (its address
        is baked into the captured graph, so it only moves when it must grow)."""
        torch = _torch()
        rows = tab.shape[0]
        if self.gtab is None or self.gtab.shape[0] < rows:
            cap = max(rows, 256 if self.gtab is None else 2 * self.gtab.shape[0])
            self.gtab = torch.zeros((cap, tab.shape[1]), dtype=self.T, device="cuda")
        self.gtab[:rows].copy_(torch.from_numpy(np.ascontiguousarray(tab)))

    def step_eager(self, dt):
        """One step with host-evaluated source scalars (no table, no graph)."""
        self._set_tables()
        if not self._opened:
            self._open_first()
        if self.num_elements is not None:
            self._load_eager_row(self.t, dt)
        self._set_bases(self.nstep)
        self.begin_steps()
        self._enqueue_step(dt, self.t, False)
        self._parity ^= 1
        self.end_steps()
        self.t += dt
        self.nstep += 1
        self._record_last()
        return self.t

    def _replay_step(self, dt):
        """One RK4 step reading the source table row ``step_dev`` points at: a
        graph replay (or, when capture is unavailable, the same launches eagerly).
        Private: the caller (``rk4``, or a benchmark that rewrites the one-row table itself)
        is responsible for ``step_dev`` staying inside the loaded table; the step size is
        baked into the captured graph."""
        if self._graph is not None:
            if dt != self._graph_dt:
                raise _lib.FusError(f"_replay_step: the graph was captured with dt = {self._graph_dt}, got {dt}")
            self._graph[self._parity].replay()
        else:
            self._enqueue_step(dt, 0.0, True)
        self._parity ^= 1

    def _capture(self, dt):
        torch = _torch()
        # warm up outside capture (lazy NCCL communicators, module loading)
        saved = [t.clone() for t in self._state()]
        step0 = self.step_dev.clone()
        self._set_bases(_OUTSIDE)  # the warm-up steps record no row (rk4 sets the base next)
        self.begin_steps()
        for parity in (self._parity, 1 - self._parity):  # both buffer roles, each step feeding the next
            self._enqueue_step(dt, 0.0, True, parity)
        self.end_steps()
        torch.cuda.synchronize()
        for t, s in zip(self._state(), saved):
            t.copy_(s)
        self.step_dev.copy_(step0)
        if self.p2p:
            self.halo.barrier()  # every rank has restored its ghost slots before anyone's next put
        self._graph_dt, self._graph_tab, self._graph_rec = dt, self.gtab.data_ptr(), self._recs
        try:
            graphs = []
            for parity in (0, 1):  # base / accumulator buffers swap roles every step
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue_step(dt, 0.0, True, parity)
                graphs.append(g)
            self._graph = graphs  # capture does not execute: state is still the saved one
        except Exception as e:  # e.g. a transport that cannot be captured
            self._graph = None
            self.graph_error = repr(e)
            torch.cuda.synchronize()

    def _state(self):
        return [*self._uv[0], *self._uv[1], self.ku, self.un, self.b, self.m]

    # algorithmic HBM bytes (SURVEY.md section 8d)
    def _stiffness_bytes(self):
        """One stiffness action: dofmap, G (or the compressed factors, or the 36 trilinear
        coefficients) and a coefficient per cell, x read and b written per dof."""
        s = self.dtype.itemsize
        Nd = self.n**3
        nstream = self.ncells - self.naff - self.ntri
        return (nstream * (Nd * 4 + 6 * Nd * s + s) + self.naff * (Nd * 4 + 7 * s) + self.ntri * (Nd * 4 + 37 * s)
                + 2 * s * self.ndofs)

    def stage_bytes(self):
        """One RK stage: vector passes of the close kernels per step 9 + 12 + 12 + 8 (ping-pong),
        i.e. 10.25 a stage."""
        return self._stiffness_bytes() + 10.25 * self.dtype.itemsize * self.ndofs

    def stage_bytes_survey(self):
        """SURVEY.md section 8(d)'s model of a fused linear stage: 6s + stiffness + 8s per dof."""
        return self.stage_bytes() + (14 - 10.25) * self.dtype.itemsize * self.ndofs


class LinearSpectral3D(_RK4):
    """Linear second-order wave equation, explicit RK4, lumped mass
    (cpp/common/Linear.hpp:43-344; cuda/demo_linear_box.py).

    ``cell_coeff1 = 1/(rho c^2)`` (mass), ``cell_coeff2 = -1/rho`` (stiffness),
    source facets ``(bfacet_dofmap1, detJ_f1, facet_coeff1 = 1/rho)``, absorbing
    facets ``(bfacet_dofmap2, detJ_f2, facet_coeff2 = -1/(rho c))`` - the arrays of
    cuda/demo_linear_box.py:336-345, on the device or as numpy.
    """

    def __init__(self, P, float_type, ndofs, dofmap, G, detJ, dphi_1D, cell_coeff1, cell_coeff2,
                 bfacet_dofmap1=None, detJ_f1=None, facet_coeff1=None, bfacet_dofmap2=None,
                 detJ_f2=None, facet_coeff2=None, halo=None, source=None,
                 source_at_stage_time=True, use_graph=True, geometry="stream", weights=None,
                 split_cells=True, trilinear=None, source_elements=None, num_elements=None):
        super().__init__(P, float_type, ndofs, dofmap, G, dphi_1D, halo, source,
                         source_at_stage_time, use_graph, geometry, weights, split_cells, trilinear,
                         source_elements, num_elements)
        torch = _torch()
        self.cell_coeff2 = _dev(cell_coeff2, self.T)
        c1 = _dev(cell_coeff1, self.T)
        dJ = _dev(detJ, self.T) if self._Tc is None else None
        # lumped mass: fill(1) -> mass -> scatter_rev  (cuda/demo_linear_box.py:421-428)
        ones = torch.ones(self.ndofs, dtype=self.T, device="cuda")
        self._cell_mass(ones, c1, self.m, dJ)
        if self.halo is not None:
            self.halo.reverse(self.m)
        self._abs_facets = self._facets(bfacet_dofmap2, detJ_f2, facet_coeff2)
        self._boundary_setup(src=self._facets(bfacet_dofmap1, detJ_f1, facet_coeff1), absb=self._abs_facets)
        self._setup_geometry(None, ["cell_coeff2"])

    # b += K(-1/rho; un)                                      (cuda/demo_linear_box.py:543-545)
    form = "stiffness"

    def _operands(self, x, vn, c0):
        return x.data_ptr(), self._sptr(self.cell_coeff2, c0), self.b.data_ptr()

    def _stiffness(self, x=None, wait=False):
        self._cell_kernels(self.un if x is None else x, None, wait)

    # close with the lumped mass: fus_rk_close, variant 0 of fus_rk_close_shared
    _close_name, _close_variant = "fus_rk_close", 0

    def _masses(self):
        return self.m, None, None, None


class LinearLeapfrog3D(LinearSpectral3D):
    """The same linear wave problem advanced with the LEAPFROG (Stoermer-Verlet) scheme instead of
    RK4: ``u`` lives at whole steps, ``v`` at half steps,

        b = K(-1/rho; u^n) + g(t_n) src + absb v^{n-1/2}
        v^{n+1/2} = v^{n-1/2} + dt b / (m - dt/2 absb)        (absorbing term time-centred)
        u^{n+1}   = u^n + dt v^{n+1/2}

    ONE stiffness action and 7 vector passes per step (RK4: four and 41), second order in time,
    stable for ``dt <= 2 / sqrt(lambda_max)`` (RK4: 2.78 / sqrt(lambda_max)).  The north star names
    "RK4/leapfrog"; the reference implements RK4 only (cuda/demo_linear_box.py:437-567), so this
    scheme has no reference twin: it is pinned to the oracle's restatement (bit-for-bit the same
    operations) and to its convergence order against the RK4 solution (tests/test_gpu_leapfrog.py).

    Same constructor as ``LinearSpectral3D``; ``rk4`` is kept as the stepping entry point (alias
    ``steps``) so the demos, ``bench.py`` and the graph machinery drive either integrator.
    After ``n`` steps ``u`` is ``u(t_n)`` and ``v`` is ``v(t_n - dt/2)``."""

    integrator = "leapfrog"

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self._absd = self._facet_diagonal(self._abs_facets)
        self._mlf = None
        self._mlf_dt = None

    @property
    def u(self):
        return self._uv[0][0]

    @property
    def v(self):
        return self._uv[0][1]

    def _lf_close(self, m, dt_v, dt_u, count_step, skip=None, n=None):
        u, v = self._uv[0]
        check(fn("fus_leapfrog_close", self.dtype)(
            u.data_ptr(), v.data_ptr(), self.b.data_ptr(), m.data_ptr(), dt_v, dt_u, self.nupd if n is None else n,
            self.step_dev.data_ptr() if count_step else None, skip, current_stream()), "fus_leapfrog_close")

    def _kick(self, t0, dt):
        """v(t0) -> v(t0 - dt/2): half a step backwards with the acceleration at t0."""
        g, dg = self._source_at(0, dt, t0, False)
        if self.num_elements is not None:
            self._load_eager_row(t0, dt)
        self._assemble_exchanged(0, g, dg, False, self.u, self.v)
        self._lf_close(self.m, -0.5 * dt, 0.0, False)
        if self.p2p and self.ndofs > self.nupd:
            self.b[self.nupd:].zero_()  # the stand-alone reverse keeps the ghost sums; the steps expect them cleared

    def rk4(self, t0, dt, nsteps):
        """``nsteps`` leapfrog steps of size ``dt`` from ``t0`` (the name is the solvers' common
        stepping entry point); returns the final time."""
        if self._mlf_dt != dt:
            self._mlf = (self.m - (0.5 * dt) * self._absd).contiguous()
            self._mlf_dt = dt
        if not self._opened:
            self._set_tables()
            self._open_first()
            self._kick(float(t0), dt)
        return super().rk4(t0, dt, nsteps)

    steps = rk4

    def step_eager(self, dt):
        raise NotImplementedError("LinearLeapfrog3D: use rk4 / steps")

    def _enqueue_step(self, dt, t, use_table, parity=None):
        """One leapfrog step: one stage on ``_uv[0]`` (the ping-pong ``parity`` plays no role)."""
        self._stage(0, dt, t, use_table, self._uv[0], self._uv[0])

    # close with m - dt/2 absb: fus_leapfrog_close, variant 3 of fus_rk_close_shared (u, v are put)
    _close_variant = 3

    def _masses(self):
        return self._mlf, None, None, None

    def _close_args(self, stage, dt, base, acc):
        return base[0].data_ptr(), base[1].data_ptr(), None, None, dt, dt, 4

    def _close(self, stage, dt, count_step, base, acc, skip=None, n=None):
        self._lf_close(self._mlf, dt, dt, count_step, skip, n)

    def stage_bytes(self):
        """Algorithmic HBM bytes of one leapfrog STEP: one stiffness action + 7 vector passes."""
        return self._stiffness_bytes() + 7 * self.dtype.itemsize * self.ndofs


class WesterveltSpectral3D(_RK4):
    """Westervelt equation (nonlinear, diffusive), explicit RK4 with a
    state-dependent lumped mass - cuda/demo_nonlinear_bowl.py:358-374, 459-469,
    529-657.

    Cell coefficients ``c1 = 1/(rho c^2)``, ``c2 = -2 beta/(rho^2 c^4)``,
    ``c3 = -1/rho``, ``c4 = -delta/(rho c^2)``, ``c5 = 2 beta/(rho^2 c^4)``; source
    facets with ``facet_coeff1_1 = 1/rho`` (g) and ``facet_coeff2_1 = delta/(rho c^2)``
    (dg/dt); absorbing facets with ``facet_coeff1_2 = delta/(rho c^3)`` (into m0)
    and ``facet_coeff2_2 = -1/(rho c)``.

    ``mass_form="pointwise"`` (default): the lumped mass is diagonal, so the two cell-mass
    applications of every stage (:609-612 ``m += M(c2; un)``, :626-628 ``b += M(c5; vn^2)``)
    equal ``un * m2`` and ``vn^2 * m5`` with ``m2 = M(c2; 1)``, ``m5 = M(c5; 1)`` assembled
    once: they move into the close kernel, the stage kernel is the dual stiffness action
    alone and only ``b`` is reverse-exchanged.  ``mass_form="cells"`` recomputes them over
    the cells every stage as the reference does (one pass over G, detJ and the dofmap).
    """

    westervelt = True

    def __init__(self, P, float_type, ndofs, dofmap, G, detJ, dphi_1D, cell_coeff1, cell_coeff2,
                 cell_coeff3, cell_coeff4, cell_coeff5, bfacet_dofmap1=None, detJ_f1=None,
                 facet_coeff1_1=None, facet_coeff2_1=None, bfacet_dofmap2=None, detJ_f2=None,
                 facet_coeff1_2=None, facet_coeff2_2=None, halo=None, source=None,
                 source_at_stage_time=True, use_graph=True, geometry="stream", weights=None,
                 mass_form="pointwise", split_cells=True, trilinear=None, source_elements=None,
                 num_elements=None):
        super().__init__(P, float_type, ndofs, dofmap, G, dphi_1D, halo, source,
                         source_at_stage_time, use_graph, geometry, weights, split_cells, trilinear,
                         source_elements, num_elements)
        torch = _torch()
        if mass_form not in ("pointwise", "cells"):
            raise ValueError("mass_form must be 'pointwise' or 'cells'")
        self.mass_form = mass_form
        self._m_accum = mass_form == "cells"
        self.detJ = _dev(detJ, self.T) if self._Tc is None else None
        self.c2, self.c3 = _dev(cell_coeff2, self.T), _dev(cell_coeff3, self.T)
        self.c4, self.c5 = _dev(cell_coeff4, self.T), _dev(cell_coeff5, self.T)
        c1 = _dev(cell_coeff1, self.T)
        # steady LHS m0 (cuda/demo_nonlinear_bowl.py:459-469)
        ones = torch.ones(self.ndofs, dtype=self.T, device="cuda")
        self.m0 = self._zx()  # reverse-exchanged once below: peer-addressable with the P2P halo
        self._cell_mass(ones, c1, self.m0, self.detJ)
        absorbing = self._facets(bfacet_dofmap2, detJ_f2, facet_coeff1_2)
        if absorbing is not None:
            bd2, dJ2, fc = absorbing
            self._mass(ones, fc, self.m0, dJ2, bd2)
        if self.halo is not None:
            self.halo.reverse(self.m0)
        # the -1/(rho c) absorbing facets: a boundary-launch term of every RK stage; the leapfrog step
        # applies them in its close instead (WesterveltLeapfrog3D)
        self._abs_facets = self._facets(bfacet_dofmap2, detJ_f2, facet_coeff2_2)
        self._boundary_setup(src=self._facets(bfacet_dofmap1, detJ_f1, facet_coeff1_1),
                             src2=self._facets(bfacet_dofmap1, detJ_f1, facet_coeff2_1),
                             absb=self._abs_facets if self.integrator == "rk4" else None)
        self.m.zero_()  # "cells" form: state-dependent part, accumulated per stage, zeroed by the close kernel
        self.m2 = self.m5 = None
        if not self._m_accum:
            # lumped M(c2; 1) and M(c5; 1), owner-complete like m0
            self.m2, self.m5 = self._zx(), self._zx()
            self._cell_mass(ones, self.c2, self.m2, self.detJ)
            self._cell_mass(ones, self.c5, self.m5, self.detJ)
            if self.halo is not None:
                self.halo.reverse(self.m2, self.m5)
        self._setup_geometry(self.detJ if self._m_accum else None, ["c2", "c3", "c4", "c5"])
        if not self._m_accum:
            self.detJ = None  # only the set-up needed it
        # b += K(c3; un) + K(c4; vn) [+ M(c5; vn^2) and m += M(c2; un)]: ONE pass over G (, detJ)
        # and the dofmap, un / vn gathered once                    (:609-612, :620-628)
        self.form = "stiffness_westervelt" if self._m_accum else "stiffness2"
        self._close_name, self._close_variant = (("fus_rk_close_westervelt", 1) if self._m_accum else
                                                 ("fus_rk_close_westervelt_pw", 2))

    def _state(self):
        return super()._state() + [self.m0]

    def _operands(self, x, vn, c0):
        sp = self._sptr
        if self._m_accum:
            return (x.data_ptr(), sp(self.c3, c0), vn.data_ptr(), sp(self.c4, c0), sp(self.c2, c0), sp(self.c5, c0),
                    self.m.data_ptr(), self.b.data_ptr())
        return x.data_ptr(), sp(self.c3, c0), vn.data_ptr(), sp(self.c4, c0), self.b.data_ptr()

    def _stage_kernel(self, x=None, vn=None, wait=False):
        self._cell_kernels(self.un if x is None else x, self.ku if vn is None else vn, wait)

    def _masses(self):
        return (self.m, self.m0, None, None) if self._m_accum else (None, self.m0, self.m2, self.m5)

    def stage_bytes(self):
        s = self.dtype.itemsize
        Nd = self.n**3
        if self._m_accum:  # + detJ stream, second gather, m read-modify-write, m0, m zero
            return super().stage_bytes() + (self.ncells - self.naff - self.ntri) * Nd * s + 6 * s * self.ndofs
        # pointwise: + second gather (vn) in the stage kernel; close passes 11 + 15 + 15 + 11 per step
        return super().stage_bytes() + s * self.ndofs + (13 - 10.25) * s * self.ndofs


class WesterveltLeapfrog3D(WesterveltSpectral3D):
    """The Westervelt problem of ``WesterveltSpectral3D`` (pointwise mass form) advanced with an
    explicit second-order LEAPFROG scheme: ``u`` lives at whole steps, ``v`` at half steps and ``w``
    is the velocity extrapolated to the whole step,

        b = K(c3; u^n) + K(c4; w^n) + g(t_n) src + dg(t_n) src2
        a = (b + m5 (w^n)^2 + absd v^{n-1/2}) / (m0 - dt/2 absd + m2 u^n)
        v^{n+1/2} = v^{n-1/2} + dt a
        w^{n+1}   = v^{n+1/2} + dt/2 a                      (= 1.5 v^{n+1/2} - 0.5 v^{n-1/2})
        u^{n+1}   = u^n + dt v^{n+1/2}

    with ``absd`` the owner-complete diagonal of the -1/(rho c) absorbing facets (time-centred by the
    -dt/2 absd in the mass, as in ``LinearLeapfrog3D``).  The mass is diagonal and taken at ``u^n``,
    the velocity terms at ``w^n``, so the step is explicit: ONE dual stiffness action
    (``fus_stiffness2_*``) and 12 vector passes per step (``fus_westervelt_leapfrog_close_*``), against
    RK4's four and 52.  The reference implements RK4 only, so the scheme is pinned to its numpy
    restatement (``tests/westervelt_leapfrog_oracle.py``) and to its convergence order against RK4.

    Same constructor as ``WesterveltSpectral3D``; ``mass_form="cells"`` raises ``ValueError``.  The
    first ``rk4`` / ``steps`` call after ``init()`` kicks off from ``(u0, v0)`` with one eager pass
    (``w = v0``, mass ``m0``: ``v`` goes back half a step).  After ``n`` steps ``u`` is ``u(t_n)`` and
    ``v`` is ``v(t_n - dt/2)``."""

    integrator = "leapfrog"

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        if self.mass_form != "pointwise":
            raise ValueError("WesterveltLeapfrog3D: only mass_form='pointwise' (the mass must be diagonal)")
        self._absd = self._facet_diagonal(self._abs_facets)
        # w is the velocity operand of the cell kernels, the role ku (vn) has in an RK stage: it takes that
        # buffer, which is peer-addressable (the neighbours put w into its ghost slots), zeroed by init()
        # and part of _state(); the 12 vectors then fit the peer-memory arena of problem.box_setup
        self.w = self.ku
        self._mm = None
        self._mm_dt = None

    @property
    def u(self):
        return self._uv[0][0]

    @property
    def v(self):
        return self._uv[0][1]

    def _wl_close(self, m, bdt, cdt, adt, count_step, skip=None, n=None):
        u, v = self._uv[0]
        check(fn("fus_westervelt_leapfrog_close", self.dtype)(
            u.data_ptr(), v.data_ptr(), self.w.data_ptr(), self.b.data_ptr(), m.data_ptr(), self.m2.data_ptr(),
            self.m5.data_ptr(), self._absd.data_ptr(), bdt, cdt, adt, self.nupd if n is None else n,
            self.step_dev.data_ptr() if count_step else None, skip, current_stream()), "fus_westervelt_leapfrog_close")

    def _kick(self, t0, dt):
        """(u0, v0) -> v(t0 - dt/2), w = v0: half a step backwards with the acceleration at t0."""
        self.w.copy_(self.v)
        g, dg = self._source_at(0, dt, t0, False)
        if self.num_elements is not None:
            self._load_eager_row(t0, dt)
        self._assemble_exchanged(0, g, dg, False, self.u, self.w)
        self._wl_close(self.m0, -0.5 * dt, 0.5 * dt, 0.0, False)
        if self.p2p and self.ndofs > self.nupd:
            self.b[self.nupd:].zero_()  # the stand-alone reverse keeps the ghost sums; the steps expect them cleared

    def rk4(self, t0, dt, nsteps):
        """``nsteps`` leapfrog steps of size ``dt`` from ``t0`` (the name is the solvers' common
        stepping entry point); returns the final time."""
        if self._mm_dt != dt:
            self._mm = (self.m0 - (0.5 * dt) * self._absd).contiguous()
            self._mm_dt = dt
        if not self._opened:
            self._set_tables()
            self._open_first()
            self._kick(float(t0), dt)
        return super().rk4(t0, dt, nsteps)

    steps = rk4

    def step_eager(self, dt):
        raise NotImplementedError("WesterveltLeapfrog3D: use rk4 / steps")

    def begin_steps(self):
        """Peer-memory halo: put (u, w), the pair the next step's cell kernels read."""
        if self.p2p:
            self.halo.barrier()
            self.halo.put(self.u, self.w)

    def _enqueue_step(self, dt, t, use_table, parity=None):
        """One leapfrog step: one stage whose cell-kernel input is (u, w) (``parity`` plays no role)."""
        self._stage(0, dt, t, use_table, (self.u, self.w), None)

    def _close(self, stage, dt, count_step, base, acc, skip=None, n=None):
        self._wl_close(self._mm, dt, 0.5 * dt, dt, count_step, skip, n)

    def _close_shared(self, stage, dt, base, acc):
        u, v = self._uv[0]
        check(fn("fus_westervelt_leapfrog_close_shared", self.dtype)(
            self.halo.handle, 1, 1, u.data_ptr(), v.data_ptr(), self.w.data_ptr(), self.b.data_ptr(),
            self._mm.data_ptr(), self.m2.data_ptr(), self.m5.data_ptr(), self._absd.data_ptr(), dt, 0.5 * dt, dt,
            current_stream()), "fus_westervelt_leapfrog_close_shared")

    def stage_bytes(self):
        """Algorithmic HBM bytes of one leapfrog STEP: one dual stiffness action (two gathers) + 12
        vector passes (8 reads + 4 writes per dof)."""
        s = self.dtype.itemsize
        return self._stiffness_bytes() + s * self.ndofs + 12 * s * self.ndofs
