"""
Problem set-up - the demos' preamble, once
==========================================

Everything the reference demos do between ``create_box`` and the time loop
(``cuda/demo_linear_box.py:83-435``, ``cuda/demo_nonlinear_bowl.py:98-470``):
mesh part of this rank, tensor-product dofmap, scatterer data + halo exchange,
geometry tables (on the device), boundary facet groups with their scaled
Jacobians and dofmaps, material coefficient arrays, and the fused RK4 solver.

Meshes are boxes of hexahedra from the synthetic substrate (DOLFINx is not in
this image; the XDMF meshes ``BM1SC2`` and ``H131`` of the piston / bowl demos
are not in the reference tree either): the piston source is the disc of facets
on ``z = 0`` whose centroid lies within ``radius`` of the axis, the bowl demo's
source is the same disc on ``x = 0`` with every exterior facet absorbing, as
``cuda/demo_nonlinear_bowl.py:282-285`` does.
"""

from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import precompute as pre
from . import substrate as S
from . import utils
from .scatterer import HaloExchange, P2PHaloExchange, SymmFabric
from .solver import (LinearLeapfrog3D, LinearSpectral3D, WesterveltLeapfrog3D, WesterveltSpectral3D, linear_source,
                     westervelt_source)


@dataclass
class Setup:
    """One rank's discretisation of a box (host + device arrays)."""

    P: int
    dtype: np.dtype
    rank: int
    world: int
    mesh: S.BoxMesh
    tables: S.ElementTables
    dofmap: np.ndarray  # host (Nc, n^3) int32
    ndofs: int  # owned + ghost
    nlocal: int  # owned
    global_dofs: int
    global_cells: tuple
    halo: object | None
    dev: dict = field(default_factory=dict)  # device tensors: dofmap, G and detJ (or Tc), x_dofs, x_g, tables
    h: float = 0.0
    local_to_serial: np.ndarray | None = None  # (ndofs,) index of every local dof in the unpartitioned box
    # multi-rank set-ups renumber the owned dofs so that the shared ones are contiguous
    # (utils.shared_last_numbering): local_perm[index in the index map's numbering] = index used here
    local_perm: np.ndarray | None = None


def _d(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def box_setup(P, ncells, lengths, dtype=np.float64, rank=0, world=1, comm=None, grid=None,
              perturb=0.0, seed=0, order="basix", max_halo_vecs=3, scatter_data=None,
              halo_kind="nccl", fabric=None, partition="block", renumber_shared=True, geometry="stream") -> Setup:
    """Mesh part, dofmap, halo and device geometry of rank ``rank`` of ``world``.

    ``comm``: torch.distributed group / transport for the halo (None = world
    group when ``world > 1``).  ``partition``: ``"block"`` (``substrate.partition_box``, the
    rank grid) or ``"blob"`` - an unstructured-like partition (``substrate.partition_cells``:
    irregular connected parts, shuffled cell / dof / ghost order, pseudo-random ownership of
    the shared dofs), which exercises the generic index-map -> halo path the way a graph
    partitioner's output would.  ``renumber_shared``: move the owned dofs that neighbours ghost
    to the end of the owned block (``utils.shared_last_numbering``; ``Setup.local_perm``).
    ``geometry``: the solvers' geometry mode this set-up serves; with ``"vertex"`` the (Nc, n^3)
    tables ``G`` and ``detJ`` are not built, ``dev["Tc"]`` holds the 36 trilinear coefficients
    per cell instead."""
    dtype = np.dtype(dtype)
    if np.isscalar(ncells):
        ncells = (int(ncells),) * 3
    if np.isscalar(lengths):
        lengths = (float(lengths),) * 3
    tb = S.element_tables(P, order, dtype)
    halo = None
    l2s = None
    lperm = None
    if world == 1:
        mesh = S.create_box(ncells, lengths, dtype=dtype, perturb=perturb, seed=seed)
        dofmap = S.tensor_dofmap(mesh, P, order)
        ndofs = nlocal = S.num_dofs(ncells, P)
    else:
        if partition == "blob":
            part = S.partition_cells(ncells, P, S.blob_cell_ranks(ncells, world, seed=seed), lengths=lengths,
                                     order=order, dtype=dtype, perturb=perturb, seed=seed, shuffle_seed=seed + 1,
                                     owner_rule="hash")[rank]
        elif partition == "block":
            part = S.partition_box(ncells, P, world, lengths=lengths, order=order, dtype=dtype,
                                   perturb=perturb, seed=seed, ranks=[rank], grid=grid)[0]
        else:
            raise ValueError("partition must be 'block' or 'blob'")
        mesh, dofmap = part.mesh, part.dofmap
        l2s = part.local_to_serial
        nlocal = part.index_map.size_local
        ndofs = nlocal + part.index_map.num_ghosts
        if scatter_data is not None:  # ranks emulated in one process: lists computed for all ranks at once
            od, gd = scatter_data
        else:
            od, gd = utils.compute_scatterer_data(part.index_map, comm)
        if renumber_shared:
            lperm, gd = utils.shared_last_numbering(nlocal, ndofs - nlocal, gd)
            dofmap = np.ascontiguousarray(lperm[dofmap], dtype=np.int32)
            moved = np.empty_like(l2s)
            moved[lperm] = l2s
            l2s = moved
        if halo_kind == "p2p":
            # halo fused into two kernels over NVLink peer memory (scatterer.P2PHaloExchange)
            if fabric is None:
                fabric = SymmFabric(P2PHaloExchange.arena_bytes(ndofs, dtype), comm)
            halo = P2PHaloExchange(fabric, od, gd, nlocal, ndofs - nlocal, dtype)
        else:
            halo = HaloExchange(comm, od, gd, nlocal, dtype, max_vecs=max_halo_vecs)
    nc = mesh.num_cells
    dev = dict(dofmap=_d(dofmap), x_dofs=_d(mesh.x_dofs), x_g=_d(mesh.x_g), dphi=_d(tb.dphi), wts=_d(tb.wts),
               dphi_f=_d(tb.dphi_f), wts_f=_d(tb.wts_f))
    _cell_geometry(dev, nc, tb, geometry)
    h = min(lengths[i] / ncells[i] for i in range(3))
    return Setup(P, dtype, rank, world, mesh, tb, dofmap, ndofs, nlocal, S.num_dofs(ncells, P),
                 tuple(ncells), halo, dev, h, l2s, lperm)


def _cell_geometry(dev, nc, tb, geometry):
    """The per-cell geometry the solvers read: G and detJ tables, or Tc alone for geometry='vertex'."""
    import torch

    if geometry not in ("stream", "auto", "vertex"):
        raise ValueError("geometry must be 'stream', 'auto' or 'vertex'")
    if geometry == "vertex":
        dev["Tc"] = pre.trilinear_coefficients((dev["x_dofs"], dev["x_g"]), nc, tb.dphi, tb.pts)
        return
    tdt = dev["x_g"].dtype
    nd3 = tb.n**3
    dev["G"] = torch.empty((nc, nd3, 6), dtype=tdt, device="cuda")
    dev["detJ"] = torch.empty((nc, nd3), dtype=tdt, device="cuda")
    # one pass for both tables (the reference makes two: cuda/demo_linear_box.py:245-253)
    pre.compute_geometry(dev["G"], dev["detJ"], (dev["x_dofs"], dev["x_g"]), nc, dev["dphi"], dev["wts"])


def _geometry_kw(su: Setup, kw):
    """Solver keywords of the geometry mode: the quadrature weights, and for 'vertex' the trilinear
    coefficients (computed here when the set-up was built for another mode)."""
    geometry = kw.get("geometry", "stream")
    if geometry != "stream":
        kw.setdefault("weights", su.tables.wts)
    if geometry == "vertex":
        if "Tc" not in su.dev:
            su.dev["Tc"] = pre.trilinear_coefficients((su.dev["x_dofs"], su.dev["x_g"]), su.mesh.num_cells,
                                                      su.tables.dphi, su.tables.pts)
        kw.setdefault("trilinear", (su.dev["Tc"], su.tables.pts_1d, su.tables.wts_1d))
    return kw


def facet_group(su: Setup, local_facets, predicate=None):
    """``(bfacet_dofmap (device int32), detJ_f (device), boundary_data (host))`` for the
    exterior facets on the given reference faces (0: z=0, 1: y=0, 2: x=0, 3: x=L, 4: y=L, 5: z=L),
    optionally filtered by ``predicate(centroids)`` - cuda/demo_linear_box.py:256-333.
    ``local_facets`` may instead be the ``boundary_data`` array (nf, 2) of
    ``utils.facet_integration_domain`` (meshes that come from DOLFINx)."""
    import torch

    tdt = torch.float64 if su.dtype == np.float64 else torch.float32
    if isinstance(local_facets, np.ndarray) and local_facets.ndim == 2:
        # rows (cell, local facet) straight from utils.facet_integration_domain (DOLFINx meshes)
        bd = np.ascontiguousarray(local_facets, dtype=np.int32)
    else:
        bds = [S.boundary_facets(su.mesh, f, predicate) for f in local_facets]
        bd = np.concatenate(bds) if bds else np.zeros((0, 2), np.int32)
    n2 = su.tables.n**2
    dJ = torch.empty((bd.shape[0], n2), dtype=tdt, device="cuda")
    if bd.shape[0]:
        pre.compute_boundary_facets_scaled_jacobian_determinant(
            dJ, (su.dev["x_dofs"], su.dev["x_g"]), _d(bd), su.dev["dphi_f"], su.dev["wts_f"])
    fd = S.facet_dofmap(su.dofmap, bd, su.tables.local_facet_dof)
    return _d(fd) if fd.shape[0] else torch.zeros((0, n2), dtype=torch.int32, device="cuda"), dJ, bd


def _full(su, n, v):
    import torch

    return torch.full((int(n),), float(v), dtype=torch.float64 if su.dtype == np.float64 else torch.float32,
                      device="cuda")


def cfl_time_step(P, h, c0, f0, cfl):
    """cuda/demo_linear_box.py:116-120: CFL step rounded to a whole number per period."""
    dt = cfl * h / (c0 * P**2)
    period = 1.0 / f0
    return period / (int(period / dt) + 1)


def facet_centroids(mesh, boundary_data):
    """(nf, 3) centroids of the facets ``boundary_data`` (rows (cell, local facet)) from their four
    vertices."""
    bd = np.asarray(boundary_data).reshape(-1, 2)
    cen = np.zeros((bd.shape[0], 3), dtype=np.asarray(mesh.x_g).dtype)
    for lf in np.unique(bd[:, 1]):
        axis, side = S._FACE_AXIS[int(lf)]
        fv = [v for v in range(8) if ((v >> axis) & 1) == side]
        sel = bd[:, 1] == lf
        cen[sel] = mesh.x_g[mesh.x_dofs[bd[sel, 0]][:, fv]].mean(axis=1)
    return cen


class TileArray:
    """A planar transducer array of ``na x nb`` square elements of side ``pitch`` (no kerf) on a
    source face, centred at the point ``centre`` of that face, its rows along ``axes[0]`` and its
    columns along ``axes[1]``; the third axis is the face normal.  Element ``e = ia * nb + ib``.
    The description is global: every rank holds the same ``centres``."""

    def __init__(self, centre, na, nb, pitch, axes=(0, 1)):
        self.centre = np.asarray(centre, dtype=np.float64).reshape(3)
        self.na, self.nb, self.pitch = int(na), int(nb), float(pitch)
        self.axes = tuple(int(a) for a in axes)
        if self.na < 1 or self.nb < 1 or not self.pitch > 0 or len(set(self.axes)) != 2:
            raise ValueError("TileArray: na, nb >= 1, pitch > 0 and two distinct in-plane axes")
        self.E = self.na * self.nb
        a, b = self.axes
        ia, ib = np.divmod(np.arange(self.E), self.nb)
        self.centres = np.tile(self.centre, (self.E, 1))
        self.centres[:, a] += (ia - 0.5 * (self.na - 1)) * self.pitch
        self.centres[:, b] += (ib - 0.5 * (self.nb - 1)) * self.pitch

    def element_of(self, centroids):
        """Element index of every facet centroid (nf, 3); -1 outside the aperture (such facets
        are not part of the source)."""
        c = np.asarray(centroids, dtype=np.float64).reshape(-1, 3)
        a, b = self.axes
        ia = np.floor((c[:, a] - self.centre[a]) / self.pitch + 0.5 * self.na)
        ib = np.floor((c[:, b] - self.centre[b]) / self.pitch + 0.5 * self.nb)
        inside = (ia >= 0) & (ia < self.na) & (ib >= 0) & (ib < self.nb)
        return np.where(inside, ia * self.nb + ib, -1).astype(np.int64)


def focus_delays(centres, focus, c0):
    """Firing delays that focus an array on ``focus``: ``tau_e = (max_j r_j - r_e) / c0`` with
    ``r_e`` the distance from element centre e, so every wave arrives at the same time and every
    ``tau_e >= 0``."""
    r = np.linalg.norm(np.asarray(centres, dtype=np.float64) - np.asarray(focus, dtype=np.float64), axis=1)
    return (r.max() - r) / c0


def element_source(base, amplitudes, delays):
    """``t -> (A_e g(t - tau_e), A_e dg(t - tau_e))`` for the ``E`` elements of an array, from one
    waveform ``base(t) -> (g, dg)`` that accepts an array ``t`` (``linear_source``,
    ``westervelt_source``).  Element e is silent, both terms exactly 0, for ``t < tau_e``."""
    A = np.asarray(amplitudes, dtype=np.float64)
    tau = np.asarray(delays, dtype=np.float64)
    if A.ndim != 1 or A.shape != tau.shape:
        raise ValueError("element_source: amplitudes and delays must both have shape (E,)")

    def source(t):
        tl = t - tau
        g, dg = base(tl)
        on = tl >= 0.0
        return np.where(on, A * g, 0.0), np.where(on, A * dg, 0.0)

    return source


def _element_facets(su, facets, predicate, elements):
    """``(bfacet_dofmap, detJ_f, boundary_data, ids, E)`` of an array's facets: ``elements`` is a
    ``TileArray`` (the facets outside its aperture are dropped, ``E = tile.E``) or one element index
    per row of the facet group (``E`` None: the caller decides)."""
    tile = elements if isinstance(elements, TileArray) else None
    if tile is not None:
        pred = predicate
        predicate = lambda cen: (tile.element_of(cen) >= 0) & (  # noqa: E731
            True if pred is None else np.asarray(pred(cen), bool))
    fd, dJ, bd = facet_group(su, facets, predicate)
    if tile is None:
        return fd, dJ, bd, np.asarray(elements, dtype=np.int64).reshape(-1), None
    ids = tile.element_of(facet_centroids(su.mesh, bd))
    if (ids < 0).any():  # DOLFINx rows given directly: keep those inside the aperture
        keep = np.flatnonzero(ids >= 0)
        fd, dJ, bd, ids = fd[_d(keep)], dJ[_d(keep)], bd[keep], ids[keep]
    return fd, dJ, bd, ids, tile.E


def _array_source(su, source_facets, source_predicate, base, kw, source_elements, element_amplitudes,
                  element_delays):
    """The source facet group and the solver keywords of a single or a phased-array source.
    ``source_elements``: a ``TileArray`` (the facets outside its aperture are dropped), or one
    element index per row of the source facet group."""
    if source_elements is None:
        if element_amplitudes is not None or element_delays is not None:
            raise ValueError("element_amplitudes / element_delays need source_elements")
        kw["source"] = base
        return facet_group(su, source_facets, source_predicate)
    fd1, dJ1, bd1, ids, E = _element_facets(su, source_facets, source_predicate, source_elements)
    if E is None:
        E = next((len(a) for a in (element_amplitudes, element_delays) if a is not None), None)
    if E is None:
        E = int(ids.max()) + 1 if ids.size else 1
    A = np.ones(E) if element_amplitudes is None else np.asarray(element_amplitudes, dtype=np.float64)
    tau = np.zeros(E) if element_delays is None else np.asarray(element_delays, dtype=np.float64)
    if A.shape != (E,) or tau.shape != (E,):
        raise ValueError(f"element_amplitudes and element_delays must have shape ({E},)")
    kw.update(source=element_source(base, A, tau), source_elements=ids, num_elements=E)
    return fd1, dJ1, bd1


def element_receiver(su: Setup, facets, elements, predicate=None, num_elements=None):
    """``sampling.ElementReceiver`` of an array on the exterior facets ``facets`` (as for
    ``facet_group``), optionally filtered by ``predicate``.  ``elements`` is a ``TileArray`` (the
    facets outside its aperture are dropped; ``E = tile.E`` on every rank) or one element index per
    row of the facet group, with ``E = num_elements`` (default: the largest index + 1; give it on
    every rank of a partitioned run).  The facets and element assignment of the solvers'
    ``source_elements`` with the same arguments: an array receives on the facets it transmits from."""
    from .sampling import ElementReceiver

    fd, dJ, _, ids, E = _element_facets(su, facets, predicate, elements)
    if E is None:
        E = num_elements if num_elements is not None else (int(ids.max()) + 1 if ids.size else None)
        if E is None:
            raise ValueError("element_receiver: no facet here: give num_elements")
    elif num_elements is not None and int(num_elements) != E:
        raise ValueError(f"element_receiver: the TileArray has {E} elements, num_elements = {num_elements}")
    return ElementReceiver(su.dtype, fd, dJ, ids, E)


def linear_solver(su: Setup, source_facets, absorbing_facets, rho=1000.0, c0=1500.0, f0=0.5e6,
                  p0=60000.0, source_predicate=None, absorbing_predicate=None, integrator="rk4",
                  source_elements=None, element_amplitudes=None, element_delays=None,
                  **kw) -> LinearSpectral3D:
    """cuda/demo_linear_box.py:336-345 coefficients + the fused solver (``integrator``: "rk4", the
    reference's scheme, or "leapfrog").  ``source_elements`` (a ``TileArray``, or one element index
    per source facet row) makes the source a phased array: element e emits
    ``A_e g(t - tau_e)`` with ``A = element_amplitudes`` (default 1) and ``tau = element_delays``
    (default 0; ``focus_delays`` focuses)."""
    if integrator not in ("rk4", "leapfrog"):
        raise ValueError("integrator must be 'rk4' or 'leapfrog'")
    cls = LinearLeapfrog3D if integrator == "leapfrog" else LinearSpectral3D
    nc = su.mesh.num_cells
    _geometry_kw(su, kw)
    fd1, dJ1, bd1 = _array_source(su, source_facets, source_predicate, lambda t: linear_source(t, f0, p0, c0), kw,
                                  source_elements, element_amplitudes, element_delays)
    fd2, dJ2, bd2 = facet_group(su, absorbing_facets, absorbing_predicate)
    return cls(
        su.P, su.dtype, su.ndofs, su.dev["dofmap"], su.dev.get("G"), su.dev.get("detJ"), su.tables.dphi_1D,
        _full(su, nc, 1.0 / rho / c0 / c0), _full(su, nc, -1.0 / rho),
        fd1, dJ1, _full(su, bd1.shape[0], 1.0 / rho), fd2, dJ2, _full(su, bd2.shape[0], -1.0 / rho / c0),
        halo=su.halo, **kw)


def westervelt_solver(su: Setup, source_facets, absorbing_facets, rho=1000.0, c0=1480.0, f0=1.1e6,
                      p0=None, beta=3.5, alpha_dB=0.2, source_predicate=None, absorbing_predicate=None,
                      source_elements=None, element_amplitudes=None, element_delays=None, integrator="rk4",
                      **kw) -> WesterveltSpectral3D:
    """cuda/demo_nonlinear_bowl.py:358-374 coefficients + the fused solver (``integrator``: "rk4", the
    reference's scheme, or "leapfrog", pointwise mass form only); phased-array keywords as for
    ``linear_solver``."""
    if integrator not in ("rk4", "leapfrog"):
        raise ValueError("integrator must be 'rk4' or 'leapfrog'")
    cls = WesterveltLeapfrog3D if integrator == "leapfrog" else WesterveltSpectral3D
    if p0 is None:
        p0 = rho * c0 * 0.38557513826589934  # source velocity of the bowl demo (:66-67)
    delta = utils.compute_diffusivity_of_sound(2.0 * np.pi * f0, c0, alpha_dB)
    nc = su.mesh.num_cells
    _geometry_kw(su, kw)
    fd1, dJ1, bd1 = _array_source(su, source_facets, source_predicate, lambda t: westervelt_source(t, f0, p0, c0),
                                  kw, source_elements, element_amplitudes, element_delays)
    fd2, dJ2, bd2 = facet_group(su, absorbing_facets, absorbing_predicate)
    n1, n2 = bd1.shape[0], bd2.shape[0]
    return cls(
        su.P, su.dtype, su.ndofs, su.dev["dofmap"], su.dev.get("G"), su.dev.get("detJ"), su.tables.dphi_1D,
        _full(su, nc, 1.0 / rho / c0 / c0), _full(su, nc, -2.0 * beta / rho / rho / c0**4),
        _full(su, nc, -1.0 / rho), _full(su, nc, -delta / rho / c0 / c0),
        _full(su, nc, 2.0 * beta / rho / rho / c0**4),
        fd1, dJ1, _full(su, n1, 1.0 / rho), _full(su, n1, delta / rho / c0 / c0),
        fd2, dJ2, _full(su, n2, delta / rho / c0**3), _full(su, n2, -1.0 / rho / c0),
        halo=su.halo, **kw)


def disc(axis_a, axis_b, centre, radius):
    """Facet-centroid predicate: inside a disc in the (axis_a, axis_b) plane."""

    def pred(cen):
        return (cen[:, axis_a] - centre[0]) ** 2 + (cen[:, axis_b] - centre[1]) ** 2 < radius**2

    return pred
