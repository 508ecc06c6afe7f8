"""
Self-check of the multi-GPU path on the GPUs it runs on
=======================================================

``multi_gpu_parity`` solves ONE small global box twice: block-partitioned over all
ranks of the process group (peer-memory halo, interior / interface overlap, CUDA-graph
replay - the production path of ``bench.py --gpus N``), and unpartitioned on rank 0's
GPU alone.  The owned parts are gathered and compared in rel-L2.  The single-GPU path is
pinned to the oracle / the reference-generated fixtures by the ``-m gpu`` tests, so this
closes the chain: N real GPUs == 1 GPU == reference.

What the reference does for the same purpose: ``/root/reference/cuda/test_scatterer.py:127-151``
compares its scatterers with DOLFINx' own ``scatter_forward/reverse`` under ``mpirun``.
"""

from __future__ import annotations

import numpy as np

from . import problem
from . import substrate as S

TOL = {np.dtype(np.float64): 1e-12, np.dtype(np.float32): 1e-5}


def _solver(su, workload, **kw):
    L = [su.h * n for n in su.global_cells]
    if workload == "linear":
        return problem.linear_solver(su, source_facets=[2], absorbing_facets=[3, 5], **kw)
    if workload == "piston":
        disc = problem.disc(0, 1, (0.5 * L[0], 0.5 * L[1]), 0.3 * L[0])
        return problem.linear_solver(su, source_facets=[0], absorbing_facets=[0, 1, 2, 3, 4, 5],
                                     source_predicate=disc, absorbing_predicate=lambda cen: ~(disc(cen) & (cen[:, 2] < 0.5 * su.h)),
                                     **kw)
    if workload in ("westervelt", "westervelt_cells"):
        disc = problem.disc(1, 2, (0.5 * L[1], 0.5 * L[2]), 0.3 * L[1])
        if workload == "westervelt_cells":
            kw["mass_form"] = "cells"
        return problem.westervelt_solver(su, source_facets=[2], absorbing_facets=[0, 1, 2, 3, 4, 5],
                                         source_predicate=disc, alpha_dB=20.0, p0=1.0e6, **kw)
    raise ValueError(workload)


def multi_gpu_parity(P=4, n_per_rank=6, dtype=np.float64, nsteps=8, workload="linear", halo_kind="p2p",
                     use_graph=True, geometry="stream", perturb=0.1, split_cells=True, split_mode="none", integrator="rk4", group=None,
                     partition="block", renumber_shared=True, grid=None):
    """rel-L2 of the partitioned solve against the single-GPU solve of the same global box.
    ``partition="blob"``: irregular parts with shuffled numbering (``problem.box_setup``) instead
    of the rank grid.

    Collective over ``group`` (default: world).  Returns a dict on every rank
    (``rel_l2_u``, ``rel_l2_v``, ``ok``, ...)."""
    import torch
    import torch.distributed as dist

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    dtype = np.dtype(dtype)
    grid = tuple(grid) if grid is not None else S.block_grid(world)
    ncells = tuple(n_per_rank * g for g in grid)
    h = 0.12 / 80
    lengths = tuple(h * n for n in ncells)
    c0, f0, cfl = (1500.0, 0.5e6, 0.65) if workload in ("linear", "piston") else (1480.0, 1.1e6, 0.4)
    dt = problem.cfl_time_step(P, h * (1.0 - 2.0 * perturb), c0, f0, cfl)
    kw = dict(geometry=geometry, use_graph=use_graph)
    if integrator != "rk4":
        kw["integrator"] = integrator  # "leapfrog": linear, piston and westervelt (pointwise) workloads
        dt = 0.5 * dt

    su = problem.box_setup(P, ncells, lengths, dtype, rank, world, comm=group, grid=grid, perturb=perturb, seed=7,
                           halo_kind=halo_kind, partition=partition, renumber_shared=renumber_shared)
    sol = _solver(su, workload, split_cells=split_cells, **kw)
    sol.split_mode = split_mode
    sol.init()
    sol.rk4(0.0, dt, nsteps)
    torch.cuda.synchronize()
    if getattr(sol.halo, "p2p", False):
        sol.halo.status()
    nl = su.nlocal
    mine = (su.local_to_serial[:nl], sol.u[:nl].cpu().numpy(), sol.v[:nl].cpu().numpy())
    parts = [None] * world
    dist.all_gather_object(parts, mine, group=group)
    out = dict(workload=workload, degree=P, dtype=dtype.name, n_gpus=world, global_cells=list(ncells),
               global_dofs=int(su.global_dofs), steps=nsteps, halo=halo_kind, geometry=geometry, partition=partition, renumber_shared=bool(renumber_shared), rank_grid=list(grid), split_mode=split_mode, integrator=integrator,
               graph=bool(use_graph and sol._graph is not None), interface_cells=int(sol.ninterface),
               shared_dofs=int(getattr(sol.halo, "nshared", 0)), tol=TOL[dtype])
    res = [0.0, 0.0, 0.0]
    if rank == 0:
        s1 = problem.box_setup(P, ncells, lengths, dtype, 0, 1, perturb=perturb, seed=7)
        ref = _solver(s1, workload, **kw)
        ref.init()
        ref.rk4(0.0, dt, nsteps)
        torch.cuda.synchronize()
        u1, v1 = ref.u.cpu().numpy().astype(np.float64), ref.v.cpu().numpy().astype(np.float64)
        u, v = np.full_like(u1, np.nan), np.full_like(v1, np.nan)
        for idx, pu, pv in parts:
            u[idx], v[idx] = pu, pv
        res = [float(np.linalg.norm(u - u1) / np.linalg.norm(u1)), float(np.linalg.norm(v - v1) / np.linalg.norm(v1)),
               float(np.linalg.norm(u1))]
    t = torch.tensor(res, dtype=torch.float64, device="cuda")
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    eu, ev, nrm = (float(x) for x in t.tolist())
    out.update(rel_l2_u=eu, rel_l2_v=ev, norm_u=nrm, ok=bool(nrm > 0 and eu <= TOL[dtype] and ev <= TOL[dtype]))
    return out
