"""
DOLFINx bridge - a live DOLFINx mesh / function space -> this package's ``Setup``
================================================================================

The reference demos take mesh, dofmap, index map and facet data from DOLFINx and
Basix on the host (``/root/reference/cuda/demo_linear_box.py:90-113, 155-180,
232-263``; the piston / bowl demos read XDMF meshes with facet tags,
``demo_nonlinear_bowl.py:98-105, 282-285``).  ``setup_from_dolfinx`` performs the
same extraction through duck typing - it touches exactly the attributes the demos
touch - and returns the ``problem.Setup`` the fused solvers are built from, so

    su = setup_from_dolfinx(mesh, V, basis_degree, float_type)
    bd_src = utils.facet_integration_domain(source_facets, mesh)          # (nf, 2)
    bd_abs = utils.facet_integration_domain(absorbing_facets, mesh)
    solver = problem.linear_solver(su, bd_src, bd_abs, rho=..., c0=..., f0=..., p0=...)

replaces everything between ``functionspace(...)`` and the time loop.  A phased-array source takes one
element index per row of ``bd_src`` (``problem.linear_solver(..., source_elements=..., element_delays=...)``).  The mesh may be
unstructured: nothing here assumes a box.  DOLFINx and Basix are not in this image, so
the bridge is exercised with stand-in objects exposing the same attributes
(tests/test_host_logic.py); with Basix importable the element tables come from Basix
itself, otherwise from the synthetic substrate (same tables under the assumptions listed
in SURVEY.md section 8c).
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import substrate as S
from . import utils
from .problem import Setup, _cell_geometry, _d


@dataclass
class HostMesh:
    """What ``problem`` / ``sampling`` need of a mesh: geometry dofmap and vertices."""

    x_dofs: np.ndarray
    x_g: np.ndarray

    @property
    def num_cells(self) -> int:
        return int(self.x_dofs.shape[0])


def basix_tables(P: int, float_type, order: str = "basix"):
    """Element tables from Basix when it is importable (the calls of
    cuda/demo_linear_box.py:167-172, 232-239, 271-299, 348-357), else the substrate's.
    Returns ``(tables, perm)``; ``perm = argsort(tp_element.dof_ordering)`` (:168)."""
    try:
        import basix  # noqa: F401
    except Exception:
        tb = S.element_tables(P, order, float_type)
        return tb, None
    import basix

    ct = basix.CellType.hexahedron
    fam, var = basix.ElementFamily.P, basix.LagrangeVariant.gll_warped
    tp = basix.create_tp_element(fam, ct, P, var, dtype=float_type)
    perm = np.argsort(np.array(tp.dof_ordering, dtype=np.int32))
    qdeg = {2: 3, 3: 4, 4: 6, 5: 8, 6: 10, 7: 12, 8: 14, 9: 16, 10: 18}[P]
    pts, wts = basix.quadrature.make_quadrature(ct, qdeg, basix.QuadratureType.gll)
    gel = basix.create_element(fam, ct, 1, dtype=float_type)
    dphi = gel.tabulate(1, pts)[1:, :, :, 0]
    pts_q, wts_f = basix.quadrature.make_quadrature(basix.CellType.quadrilateral, qdeg, basix.QuadratureType.gll)
    a, b = pts_q[:, 0], pts_q[:, 1]
    z, o = np.zeros_like(a), np.ones_like(a)
    pts_f = np.stack([np.c_[a, b, z], np.c_[a, z, b], np.c_[z, a, b], np.c_[o, a, b], np.c_[a, o, b], np.c_[a, b, o]])
    dphi_f = np.stack([gel.tabulate(1, pts_f[f])[1:, :, :, 0] for f in range(6)])
    e1 = basix.create_element(fam, basix.CellType.interval, P, var, dtype=float_type)
    p1, w1 = basix.quadrature.make_quadrature(basix.CellType.interval, qdeg, basix.QuadratureType.gll)
    dphi_1D = e1.tabulate(1, p1)[1, :, :, 0]  # :346-357
    c = lambda v: np.ascontiguousarray(v, dtype=float_type)  # noqa: E731
    tb = S.ElementTables(P, order, c(p1[:, 0]), c(w1), c(dphi_1D), c(pts), c(wts),
                         c(dphi), c(pts_f), c(wts_f), c(dphi_f),
                         np.array(tp.entity_closure_dofs[2], dtype=np.int32))
    return tb, perm


def setup_from_dolfinx(mesh, V, basis_degree, float_type=np.float64, comm=None, halo_kind="nccl",
                       tables=None, perm=None, max_halo_vecs=3, renumber_shared=True, geometry="stream") -> Setup:
    """``Setup`` of this rank from a DOLFINx ``mesh`` and function space ``V``
    (cuda/demo_linear_box.py:99-113, 175-207, 232-253).

    ``tables`` / ``perm`` override the Basix look-ups (``perm`` reorders ``V.dofmap.list``
    columns into tensor-product order; identity when the space was created on the
    tensor-product element).  ``comm``: torch.distributed group for the halo.  ``geometry``: as for
    ``problem.box_setup`` ("vertex": ``dev["Tc"]`` instead of the ``G`` / ``detJ`` tables)."""
    import torch.distributed as dist

    float_type = np.dtype(float_type)
    if tables is None:
        tables, bperm = basix_tables(basis_degree, float_type)
        perm = bperm if perm is None else perm
    tdim = mesh.topology.dim
    num_cells = int(mesh.topology.index_map(tdim).size_local)
    x_dofs = np.ascontiguousarray(np.asarray(mesh.geometry.dofmap)[:num_cells], dtype=np.int32)
    x_g = np.ascontiguousarray(mesh.geometry.x, dtype=float_type)
    dm = np.asarray(V.dofmap.list)[:num_cells]
    dofmap = np.ascontiguousarray(dm if perm is None else dm[:, perm], dtype=np.int32)
    imap = V.dofmap.index_map
    nlocal, nghost = int(imap.size_local), int(imap.num_ghosts)
    world = dist.get_world_size(comm) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(comm) if world > 1 else 0
    halo = None
    lperm = None
    if world > 1:
        od, gd = utils.compute_scatterer_data(imap, comm)
        if renumber_shared:
            # private renumbering (shared owned dofs last, contiguous): Setup.local_perm maps a DOLFINx
            # local index to the index the solver vectors use - u_dolfinx = sol.u[su.local_perm]
            lperm, gd = utils.shared_last_numbering(nlocal, nghost, gd)
            dofmap = np.ascontiguousarray(lperm[dofmap], dtype=np.int32)
        if halo_kind == "p2p":
            from .scatterer import P2PHaloExchange, SymmFabric

            fabric = SymmFabric(P2PHaloExchange.arena_bytes(nlocal + nghost, float_type), comm)
            halo = P2PHaloExchange(fabric, od, gd, nlocal, nghost, float_type)
        else:
            from .scatterer import HaloExchange

            halo = HaloExchange(comm, od, gd, nlocal, float_type, max_vecs=max_halo_vecs)
    dev = dict(dofmap=_d(dofmap), x_dofs=_d(x_dofs), x_g=_d(x_g), dphi=_d(tables.dphi), wts=_d(tables.wts),
               dphi_f=_d(tables.dphi_f), wts_f=_d(tables.wts_f))
    _cell_geometry(dev, num_cells, tables, geometry)
    # smallest cell diameter of this rank (cpp.mesh.h, cuda/demo_linear_box.py:103-108): longest vertex distance
    cc = x_g[x_dofs].astype(np.float64)
    h = float(np.sqrt(((cc[:, :, None, :] - cc[:, None, :, :]) ** 2).sum(-1)).max(axis=(1, 2)).min()) if num_cells else np.inf
    h = utils.global_min(h, comm)  # mesh_size of the reference: the minimum over all ranks
    return Setup(int(basis_degree), float_type, rank, world, HostMesh(x_dofs, x_g), tables, dofmap, nlocal + nghost,
                 nlocal, int(imap.size_global), (num_cells,), halo, dev, h, None, lperm)
