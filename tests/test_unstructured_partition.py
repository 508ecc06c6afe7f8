"""Unstructured-like partitions: what a graph partitioner hands DOLFINx, without DOLFINx.

The piston / bowl demos of the reference run on unstructured hexahedral meshes partitioned by
DOLFINx (cuda/demo_linear_piston.py:83-90, 250-251); their index maps have irregular parts,
neighbour sets of any size, ghosts in no particular order, and no run of consecutive dof indices
along a mesh line.  ``substrate.partition_cells`` produces exactly that from a box (arbitrary
cell -> rank map, shuffled cell / dof / ghost order, lowest-rank or pseudo-random ownership) and
the tests below push it through the generic path: ``compute_scatterer_data`` -> ``HaloExchange``
/ ``P2PHaloExchange`` -> the fused solvers, against the single-rank oracle.

The index maps of two such partitions also went through the reference's own
``cuda/utils.py:compute_scatterer_data`` and ``numba-cpu/scatterer.py`` (tests/golden/scatter_u4.npz,
scatter_u5.npz; ``make_golden.py --only-irregular``): the fixture tests in test_host_logic.py,
test_gpu_solver.py and test_gpu_parity_r2.py are parametrised over them.
"""

import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from fenicsx_fus_gpu_b200 import substrate as S  # noqa: E402
from fenicsx_fus_gpu_b200 import utils  # noqa: E402


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


CASES = [((5, 4, 3), 2, 5, "hash"), ((4, 4, 3), 3, 4, "lowest"), ((3, 3, 3), 4, 3, "hash")]


# --------------------------------------------------------------------------- #
# host side (no GPU)
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("N,P,R,rule", CASES)
def test_partition_cells_properties(N, P, R, rule):
    cr = S.blob_cell_ranks(N, R, seed=4)
    assert np.unique(cr).size == R
    parts = S.partition_cells(N, P, cr, shuffle_seed=7, owner_rule=rule)
    full = S.create_box(N)
    gdm = S.tensor_dofmap(full, P)
    ntot = S.num_dofs(N, P)
    seen = np.zeros(ntot, np.int32)
    offs = 0
    owner_of = np.full(ntot, -1)
    touching = [set(np.unique(gdm[cr == r]).tolist()) for r in range(R)]
    for p in parts:
        im = p.index_map
        nl = im.size_local
        assert im.local_range == (offs, offs + nl)
        offs += nl
        seen[p.local_to_serial[:nl]] += 1
        owner_of[p.local_to_serial[:nl]] = p.rank
        # the local dofmap addresses the same serial dofs as the global one, cell by cell
        assert np.array_equal(p.local_to_serial[p.dofmap], gdm[p.mesh.cell_ids])
        # ghosts: rank-contiguous global indices of dofs this rank touches but does not own
        assert np.array_equal(p.local_to_global[:nl], np.arange(im.local_range[0], im.local_range[1]))
        assert np.array_equal(p.local_to_global[nl:], im.ghosts)
        assert np.all(im.owners != p.rank)
        assert set(p.local_to_serial.tolist()) == touching[p.rank]
    assert offs == ntot and np.all(seen == 1)
    for p in parts:
        im = p.index_map
        nl = im.size_local
        # every ghost's owner is what the owner itself says, and the owner lists me as a destination
        assert np.array_equal(owner_of[p.local_to_serial[nl:]], im.owners)
        for g_serial, o in zip(p.local_to_serial[nl:], im.owners):
            q = parts[o]
            li = int(np.nonzero(q.local_to_serial[:q.index_map.size_local] == g_serial)[0][0])
            assert p.rank in q.index_map.index_to_dest_ranks().links(li)
        # and no destination without a ghost there
        dest = im.index_to_dest_ranks()
        for li in range(nl):
            for q in dest.links(li):
                assert p.local_to_serial[li] in touching[q] and q != p.rank
    if rule == "hash":  # ownership is not monotone in the rank: someone ghosts a dof of a higher rank
        assert any(np.any(p.index_map.owners > p.rank) for p in parts)
    # the shuffle left no structure behind: owned dofs are not in serial order
    assert any(np.any(np.diff(p.local_to_serial[:p.index_map.size_local]) < 0) for p in parts)


@pytest.mark.parametrize("name,N,P,R,rule", [("u5", (5, 4, 3), 2, 5, "hash"), ("u4", (4, 4, 3), 3, 4, "lowest")])
def test_partition_cells_reproduces_fixture_index_maps(golden_dir, name, N, P, R, rule):
    """Deterministic: the index maps the reference's compute_scatterer_data saw when the fixtures
    were made (tests/golden/make_golden.py irregular_scatter_cases)."""
    g = np.load(os.path.join(golden_dir, f"scatter_{name}.npz"))
    parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=4), shuffle_seed=7, owner_rule=rule)
    for r, p in enumerate(parts):
        assert p.index_map.size_local == int(g[f"r{r}_size_local"])
        assert np.array_equal(p.index_map.ghosts, g[f"r{r}_ghosts"])
        assert np.array_equal(p.index_map.owners, g[f"r{r}_owners"])
        assert np.array_equal(p.index_map.index_to_dest_ranks().array, g[f"r{r}_dest_array"])


@pytest.mark.parametrize("N,P,R,rule", CASES[:2])
def test_partitioned_assembly_equals_serial_on_cpu(N, P, R, rule):
    """Oracle only: forward halo of x, per-part stiffness + mass action, reverse halo of y ==
    the serial action (cuda/demo_linear_box.py:536-553 for one stage), on irregular parts."""
    import problems
    from oracle import oracle as orc

    L = (0.011, 0.01, 0.009)
    dtt = np.float64
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=5)
    rng = np.random.default_rng(2)
    x = rng.standard_normal(serial.ndofs)
    y_ref = np.zeros(serial.ndofs)
    orc.stiffness_operator(P, x, serial.cell_coeff2, y_ref, serial.G, serial.dofmap, serial.tb.dphi_1D)
    orc.mass_operator(x, serial.cell_coeff1, y_ref, serial.detJ, serial.dofmap)

    parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=4), lengths=L, perturb=0.1, seed=5,
                              shuffle_seed=9, owner_rule=rule)
    sdata = orc.compute_scatterer_data_all([p.index_map for p in parts])
    mine = utils.compute_scatterer_data_all([p.index_map for p in parts])
    for (od, gd), (od2, gd2) in zip(sdata, mine):  # product == oracle restatement of cuda/utils.py:8-78
        for a_, b_ in ((od, od2), (gd, gd2)):
            assert np.array_equal(np.asarray(a_[2]), np.asarray(b_[2]))
            assert all(np.array_equal(np.asarray(u), np.asarray(v)) for u, v in zip(a_[0], b_[0]))
    nl = [p.index_map.size_local for p in parts]
    xs = []
    for p in parts:  # owned values only; ghosts arrive through the forward halo
        xl = np.zeros(p.local_to_serial.size)
        xl[:p.index_map.size_local] = x[p.local_to_serial[:p.index_map.size_local]]
        xs.append(xl)
    orc.scatter_forward_all(sdata, nl, xs)
    ys = []
    for p, xl in zip(parts, xs):
        assert np.array_equal(xl, x[p.local_to_serial])
        d = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=p.dofmap, ndofs=xl.size)
        yl = np.zeros(xl.size)
        orc.stiffness_operator(P, xl, d.cell_coeff2, yl, d.G, d.dofmap, d.tb.dphi_1D)
        orc.mass_operator(xl, d.cell_coeff1, yl, d.detJ, d.dofmap)
        ys.append(yl)
    orc.scatter_reverse_all(sdata, nl, ys)
    y = np.zeros_like(y_ref)
    for p, yl in zip(parts, ys):
        y[p.local_to_serial[:p.index_map.size_local]] = yl[:p.index_map.size_local]
    assert rel_l2(y, y_ref) < 1e-13
    # boundary facets of the irregular parts: together, exactly the serial ones
    for lf in range(6):
        n = sum(S.boundary_facets(p.mesh, lf).shape[0] for p in parts)
        assert n == S.boundary_facets(serial.mesh, lf).shape[0]


# --------------------------------------------------------------------------- #
# CUDA path, ranks emulated by threads on one GPU
# --------------------------------------------------------------------------- #
def _halo(kind, transport, r, parts, sdata, dtt):
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, P2PHaloExchange, local_fabric

    p = parts[r]
    if kind == "p2p":
        ndmax = max(q.index_map.size_local + q.index_map.num_ghosts for q in parts)
        fab = local_fabric(transport.cluster, r, P2PHaloExchange.arena_bytes(ndmax, dtt))
        return P2PHaloExchange(fab, sdata[r][0], sdata[r][1], p.index_map.size_local, p.index_map.num_ghosts, dtt)
    return HaloExchange(transport, sdata[r][0], sdata[r][1], p.index_map.size_local, dtt)


def _gather(parts, out, ref):
    u = np.full(ref[0].shape, np.nan)
    v = np.full(ref[1].shape, np.nan)
    for r, p in enumerate(parts):
        nl = p.index_map.size_local
        u[p.local_to_serial[:nl]] = out[r][0][:nl]
        v[p.local_to_serial[:nl]] = out[r][1][:nl]
    return u, v


@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["rk4", "leapfrog"])
@pytest.mark.parametrize("kind", ["nccl-shaped", "p2p"])
@pytest.mark.parametrize("N,P,R,rule", CASES)
def test_linear_irregular_partition_vs_serial_oracle(N, P, R, rule, kind, integrator):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import problems
    from fenicsx_fus_gpu_b200.scatterer import LocalCluster
    from fenicsx_fus_gpu_b200.solver import LinearLeapfrog3D, LinearSpectral3D, linear_source
    from oracle import oracle as orc

    dtt, L, nsteps = np.float64, (0.012, 0.01, 0.011), 8
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11, abs_facets=(3, 4))
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0, cfl=0.3)
    m = np.zeros(serial.ndofs, dtt)
    orc.mass_operator(np.ones(serial.ndofs, dtt), serial.cell_coeff1, m, serial.detJ, serial.dofmap)
    prob = orc.LinearProblem(serial.P, serial.dofmap, serial.G, serial.tb.dphi_1D, serial.cell_coeff2, m,
                             serial.bfacet_dofmap1, serial.detJ_f1, serial.facet_coeff1, serial.bfacet_dofmap2,
                             serial.detJ_f2, serial.facet_coeff2, serial.f0, serial.p0, serial.c0)
    u_ref, v_ref = np.zeros(serial.ndofs, dtt), np.zeros(serial.ndofs, dtt)
    if integrator == "rk4":
        orc.linear_rk4(prob, u_ref, v_ref, 0.0, dt, nsteps)
    else:
        orc.linear_leapfrog(prob, u_ref, v_ref, 0.0, dt, nsteps)
    assert np.linalg.norm(u_ref) > 0

    parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=4), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                              shuffle_seed=3, owner_rule=rule)
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    cls = LinearSpectral3D if integrator == "rk4" else LinearLeapfrog3D

    def body(r, transport):
        p = parts[r]
        nd = p.index_map.size_local + p.index_map.num_ghosts
        d = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=p.dofmap, ndofs=nd, abs_facets=(3, 4))
        s = cls(d.P, dtt, d.ndofs, d.dofmap, d.G, d.detJ, d.tb.dphi_1D, d.cell_coeff1, d.cell_coeff2,
                d.bfacet_dofmap1, d.detJ_f1, d.facet_coeff1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff2,
                halo=_halo(kind, transport, r, parts, sdata, dtt),
                source=lambda t: linear_source(t, d.f0, d.p0, d.c0), use_graph=False)
        s.init()
        s.rk4(0.0, dt, nsteps)
        torch.cuda.synchronize()
        return s.u.cpu().numpy(), s.v.cpu().numpy()

    u, v = _gather(parts, LocalCluster(R).run(body), (u_ref, v_ref))
    assert rel_l2(u, u_ref) < 1e-12
    assert rel_l2(v, v_ref) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("mass_form", ["pointwise", "cells"])
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_westervelt_irregular_partition_vs_serial_oracle(tag, mass_form):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import problems
    from fenicsx_fus_gpu_b200.scatterer import LocalCluster
    from fenicsx_fus_gpu_b200.solver import WesterveltSpectral3D, westervelt_source
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32
    N, P, R, L, nsteps = (4, 4, 3), 3, 4, (0.006, 0.006, 0.0045), 6
    d0 = problems.westervelt_problem(P, N, L, np.float64, perturb=0.1, seed=7)  # reference in f64
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), d0.c0, d0.f0, cfl=0.4)
    ones = np.ones(d0.ndofs)
    m0 = np.zeros(d0.ndofs)
    orc.mass_operator(ones, d0.cell_coeff1, m0, d0.detJ, d0.dofmap)
    orc.mass_operator(ones, d0.facet_coeff1_2, m0, d0.detJ_f2, d0.bfacet_dofmap2)
    prob = orc.WesterveltProblem(d0.P, d0.dofmap, d0.G, d0.detJ, d0.tb.dphi_1D, d0.cell_coeff2, d0.cell_coeff3,
                                 d0.cell_coeff4, d0.cell_coeff5, m0, d0.bfacet_dofmap1, d0.detJ_f1,
                                 d0.facet_coeff1_1, d0.facet_coeff2_1, d0.bfacet_dofmap2, d0.detJ_f2,
                                 d0.facet_coeff2_2, d0.f0, d0.p0, d0.c0)
    u_ref, v_ref = np.zeros(d0.ndofs), np.zeros(d0.ndofs)
    orc.westervelt_rk4(prob, u_ref, v_ref, 0.0, dt, nsteps)
    assert np.linalg.norm(u_ref) > 0

    parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=6), lengths=L, dtype=dtt, perturb=0.1, seed=7,
                              shuffle_seed=5, owner_rule="hash")
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])

    def body(r, transport):
        p = parts[r]
        nd = p.index_map.size_local + p.index_map.num_ghosts
        d = problems.westervelt_problem(P, None, None, dtt, mesh=p.mesh, dofmap=p.dofmap, ndofs=nd)
        s = WesterveltSpectral3D(
            d.P, dtt, d.ndofs, d.dofmap, d.G, d.detJ, d.tb.dphi_1D, d.cell_coeff1, d.cell_coeff2,
            d.cell_coeff3, d.cell_coeff4, d.cell_coeff5, d.bfacet_dofmap1, d.detJ_f1, d.facet_coeff1_1,
            d.facet_coeff2_1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff1_2, d.facet_coeff2_2,
            halo=_halo("p2p", transport, r, parts, sdata, dtt),
            source=lambda t: westervelt_source(t, d.f0, d.p0, d.c0), mass_form=mass_form, use_graph=False)
        s.init()
        s.rk4(0.0, dt, nsteps)
        torch.cuda.synchronize()
        return s.u.cpu().numpy(), s.v.cpu().numpy()

    u, v = _gather(parts, LocalCluster(R).run(body), (u_ref, v_ref))
    tol = 1e-12 if tag == "f64" else 1e-5
    assert rel_l2(u, u_ref) < tol
    assert rel_l2(v, v_ref) < tol


@pytest.mark.gpu
def test_operators_on_shuffled_numbering_vs_oracle():
    """Stiffness and mass action on one irregular part (no run of consecutive dofs, cells in random
    order, ghost block included) against the oracle on the same arrays: the kernels assume nothing
    about the numbering."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import problems
    from fenicsx_fus_gpu_b200 import operators as ops
    from oracle import oracle as orc

    for P, N, dtt, tol in ((4, (6, 5, 5), np.float64, 1e-13), (5, (4, 4, 4), np.float32, 2e-6), (2, (9, 8, 7), np.float64, 1e-13)):
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, 3, seed=1), dtype=dtt, perturb=0.12, seed=2,
                                  shuffle_seed=8, owner_rule="hash")
        p = max(parts, key=lambda q: q.mesh.num_cells)
        nd = p.local_to_serial.size
        d = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=p.dofmap, ndofs=nd)
        rng = np.random.default_rng(4)
        x = rng.standard_normal(nd).astype(dtt)
        c = rng.uniform(0.5, 2.0, p.mesh.num_cells).astype(dtt)
        yk, ym = np.zeros(nd, dtt), np.zeros(nd, dtt)
        orc.stiffness_operator(P, x, c, yk, d.G, d.dofmap, d.tb.dphi_1D)
        orc.mass_operator(x, c, ym, d.detJ, d.dofmap)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
        xd, cd, dm = dev(x), dev(c), dev(d.dofmap)
        n = P + 1
        y1 = torch.zeros(nd, dtype=xd.dtype, device="cuda")
        ops.stiffness_operator(P, dtt)[p.mesh.num_cells, (n, n, n)](xd, cd, y1, dev(d.G), dm, dev(d.tb.dphi_1D))
        y2 = torch.zeros(nd, dtype=xd.dtype, device="cuda")
        ops.mass_operator[1, 128](xd, cd, y2, dev(d.detJ), dm)
        assert rel_l2(y1.cpu().numpy(), yk) < tol
        assert rel_l2(y2.cpu().numpy(), ym) < tol


# --------------------------------------------------------------------------- #
# shared-last renumbering (utils.shared_last_numbering)
# --------------------------------------------------------------------------- #
def _renumbered(parts, sdata):
    """What problem.box_setup does per rank: (dofmap, local_to_serial, owners_data, ghosts_data)
    in the numbering with the shared owned dofs moved to a contiguous tail."""
    out = []
    for p, (od, gd) in zip(parts, sdata):
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        perm, gd2 = utils.shared_last_numbering(nl, ng, gd)
        l2s = np.empty_like(p.local_to_serial)
        l2s[perm] = p.local_to_serial
        out.append((np.ascontiguousarray(perm[p.dofmap], dtype=np.int32), l2s, od, gd2, perm))
    return out


@pytest.mark.parametrize("kind", ["box", "blob"])
def test_shared_last_numbering_properties(kind):
    N, P, R = (4, 4, 4), 2, 8
    parts = (S.partition_box(N, P, R) if kind == "box" else
             S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=2), shuffle_seed=1, owner_rule="hash"))
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    for p, (od, gd), (dm, l2s, _, gd2, perm) in zip(parts, sdata, _renumbered(parts, sdata)):
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        assert np.array_equal(np.sort(perm), np.arange(nl + ng))  # a permutation
        assert np.array_equal(perm[nl:], np.arange(nl, nl + ng))  # ghosts stay
        old = [np.asarray(a, np.int64) for a in gd[0]]
        shared_old = np.unique(np.concatenate(old)) if old and sum(a.size for a in old) else np.zeros(0, np.int64)
        ns = shared_old.size
        # shared dofs: the tail of the owned block, old relative order kept; the rest: the head, order kept
        assert np.array_equal(perm[shared_old], nl - ns + np.arange(ns))
        rest = np.setdiff1d(np.arange(nl), shared_old)
        assert np.array_equal(perm[rest], np.arange(nl - ns))
        for a, b in zip(old, gd2[0]):
            assert np.array_equal(perm[a], np.asarray(b))
        # same serial dofs behind every dofmap entry
        assert np.array_equal(l2s[dm], p.local_to_serial[p.dofmap])
    # no neighbours: identity, lists untouched
    perm, gd2 = utils.shared_last_numbering(10, 0, [[], np.zeros(0, np.int64), np.zeros(0, np.int32)])
    assert np.array_equal(perm, np.arange(10)) and gd2[0] == []


@pytest.mark.gpu
@pytest.mark.parametrize("kind,halo,tag", [("box", "p2p", "f64"), ("box", "nccl-shaped", "f64"), ("blob", "p2p", "f64"),
                                           ("box", "p2p", "f32"), ("blob", "p2p", "f32"),
                                           ("blob-empty-bulk", "p2p", "f32")])
def test_linear_rk4_with_shared_last_numbering_vs_serial_oracle(kind, halo, tag):
    """The partitioned solve in the renumbered local ordering (what problem.box_setup hands the
    solvers on > 1 rank) against the single-rank oracle, ranks emulated on one GPU.

    ``blob-empty-bulk``: one rank owns fewer unshared dofs than one close pack, so its bulk close
    has n = 0, and it owns source facets.  Its step counter, which selects the source amplitude
    row, must still advance once per step."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import problems
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, LocalCluster, P2PHaloExchange, local_fabric
    from fenicsx_fus_gpu_b200.solver import LinearSpectral3D, linear_source
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32  # f32: packs of 4, the tail starts on a multiple of 4
    P, N, L, R, nsteps = 3, (4, 4, 4), (0.012, 0.01, 0.011), 8, 8
    src = (2,)
    if kind == "blob-empty-bulk":
        P, N, src = 2, (4, 4, 3), (0,)
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11, src_facets=src)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0)
    m = np.zeros(serial.ndofs, dtt)
    orc.mass_operator(np.ones(serial.ndofs, dtt), serial.cell_coeff1, m, serial.detJ, serial.dofmap)
    prob = orc.LinearProblem(serial.P, serial.dofmap, serial.G, serial.tb.dphi_1D, serial.cell_coeff2, m,
                             serial.bfacet_dofmap1, serial.detJ_f1, serial.facet_coeff1, serial.bfacet_dofmap2,
                             serial.detJ_f2, serial.facet_coeff2, serial.f0, serial.p0, serial.c0)
    u_ref, v_ref = np.zeros(serial.ndofs, dtt), np.zeros(serial.ndofs, dtt)
    orc.linear_rk4(prob, u_ref, v_ref, 0.0, dt, nsteps)

    if kind == "box":
        parts = S.partition_box(N, P, R, lengths=L, dtype=dtt, perturb=0.1, seed=11)
    else:
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                                  shuffle_seed=2, owner_rule="hash")
    ren = _renumbered(parts, utils.compute_scatterer_data_all([p.index_map for p in parts]))
    ndmax = max(q.index_map.size_local + q.index_map.num_ghosts for q in parts)
    if kind == "blob-empty-bulk":
        pack = 16 // np.dtype(dtt).itemsize
        empty = []
        for p, (_, _, _, gd, _) in zip(parts, ren):
            ns = np.unique(np.concatenate([np.asarray(a) for a in gd[0]])).size if sum(len(a) for a in gd[0]) else 0
            if ns and (p.index_map.size_local - ns) // pack == 0 and S.boundary_facets(p.mesh, src[0]).shape[0]:
                empty.append(p.rank)
        assert empty, "no rank with an empty bulk close that owns source facets"

    def body(r, transport):
        p = parts[r]
        dm, _, od, gd, _ = ren[r]
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        d = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=dm, ndofs=nl + ng, src_facets=src)
        if halo == "p2p":
            fab = local_fabric(transport.cluster, r, P2PHaloExchange.arena_bytes(ndmax, dtt))
            h = P2PHaloExchange(fab, od, gd, nl, ng, dtt)
            # the handle sees one contiguous block of shared dofs at the end of the owned range:
            # the bulk close is the prefix in front of it, no mask
            if sum(len(a) for a in gd[0]):
                ns = np.unique(np.concatenate([np.asarray(a) for a in gd[0]])).size
                pack = 16 // np.dtype(dtt).itemsize
                assert h.shared_tail == ((nl - ns) // pack) * pack and h.nshared == nl - h.shared_tail
                assert h.bulk_close() == dict(n=h.shared_tail)
            else:
                assert h.shared_tail == -1 and h.nshared == 0
        else:
            h = HaloExchange(transport, od, gd, nl, dtt)
        s = LinearSpectral3D(d.P, dtt, d.ndofs, d.dofmap, d.G, d.detJ, d.tb.dphi_1D, d.cell_coeff1, d.cell_coeff2,
                             d.bfacet_dofmap1, d.detJ_f1, d.facet_coeff1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff2,
                             halo=h, source=lambda t: linear_source(t, d.f0, d.p0, d.c0), use_graph=False)
        s.init()
        s.rk4(0.0, dt, nsteps)
        torch.cuda.synchronize()
        return s.u.cpu().numpy(), s.v.cpu().numpy()

    out = LocalCluster(R).run(body)
    u, v = np.full_like(u_ref, np.nan), np.full_like(v_ref, np.nan)
    for r, p in enumerate(parts):
        nl = p.index_map.size_local
        u[ren[r][1][:nl]] = out[r][0][:nl]
        v[ren[r][1][:nl]] = out[r][1][:nl]
    tol = 1e-12 if tag == "f64" else 1e-5
    assert rel_l2(u, u_ref) < tol
    assert rel_l2(v, v_ref) < tol
