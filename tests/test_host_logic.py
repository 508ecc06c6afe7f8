"""CPU tests of the host logic: index maps (bit-exact against the fixtures the
reference's cuda/utils.py produced), the torch.distributed plumbing of the halo
exchange over gloo with world_size 2, the synthetic substrate's known answers,
facet integration domains."""

import os
import sys

import numpy as np
import pytest

from fenicsx_fus_gpu_b200 import substrate as S
from fenicsx_fus_gpu_b200 import utils

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _index_maps(g):
    R = int(g["nranks"])
    maps = []
    for r in range(R):
        maps.append(S.IndexMap(
            int(g[f"r{r}_size_local"]), 0, tuple(int(v) for v in g[f"r{r}_local_range"]),
            g[f"r{r}_ghosts"], g[f"r{r}_owners"],
            S.AdjacencyList(g[f"r{r}_dest_array"], g[f"r{r}_dest_offsets"])))
    return maps


@pytest.mark.parametrize("name", ["r2", "r3", "r8", "u4", "u5"])
def test_scatterer_data_bit_exact_vs_reference(golden_dir, name):
    """utils.compute_scatterer_data (vectorised) == cuda/utils.py:8-78 output."""
    g = np.load(os.path.join(golden_dir, f"scatter_{name}.npz"))
    maps = _index_maps(g)
    out = utils.compute_scatterer_data_all(maps)
    for r, (od, gd) in enumerate(out):
        for which, data in (("owners", od), ("ghosts", gd)):
            ranks = g[f"r{r}_{which}_ranks"]
            assert np.array_equal(np.asarray(data[2]), ranks)
            assert np.array_equal(np.asarray(data[1]), g[f"r{r}_{which}_size"])
            assert len(data[0]) == ranks.size
            for i in range(ranks.size):
                a = np.asarray(data[0][i])
                assert a.dtype == np.int64
                assert np.array_equal(a, g[f"r{r}_{which}_idx{i}"])


def test_partition_reproduces_fixture_index_maps(golden_dir):
    """The block partitioner is deterministic: same IndexMap arrays as when the
    fixtures were generated."""
    g = np.load(os.path.join(golden_dir, "scatter_r8.npz"))
    parts = S.partition_box(tuple(int(v) for v in g["ncells"]), int(g["P"]), 8)
    for r, p in enumerate(parts):
        assert p.index_map.size_local == int(g[f"r{r}_size_local"])
        assert np.array_equal(p.index_map.ghosts, g[f"r{r}_ghosts"])
        assert np.array_equal(p.index_map.owners, g[f"r{r}_owners"])


def test_single_rank_has_no_neighbours():
    od, gd = utils.compute_scatterer_data(S.serial_index_map(100))
    assert od[0] == [] and gd[0] == [] and len(od[2]) == 0 and len(gd[2]) == 0


def test_partition_covers_every_dof_once():
    P, N, R = 3, (4, 3, 2), 4
    parts = S.partition_box(N, P, R)
    total = S.num_dofs(N, P)
    seen = np.zeros(total, np.int32)
    for p in parts:
        nl = p.index_map.size_local
        seen[p.local_to_serial[:nl]] += 1
        # ghosts are owned by someone else and sorted by global index
        assert np.all(np.diff(p.index_map.ghosts) > 0)
        assert np.all(p.index_map.owners != p.rank)
    assert np.all(seen == 1)


def _gloo_worker(rank, world, port, golden_dir, q, name="r2"):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, ROOT)
        from fenicsx_fus_gpu_b200.scatterer import TorchDistTransport
        from oracle import oracle as orc

        g = np.load(os.path.join(golden_dir, f"scatter_{name}.npz"))
        im = _index_maps(g)[rank]
        od, gd = utils.compute_scatterer_data(im)  # ghost-index exchange over gloo
        ok = True
        for which, data in (("owners", od), ("ghosts", gd)):
            for i in range(len(data[0])):
                ok &= bool(np.array_equal(np.asarray(data[0][i]), g[f"r{rank}_{which}_idx{i}"]))
        # forward + reverse halo with the product transport; pack/unpack by the oracle
        # (the CUDA pack kernels cannot run here)
        N = im.size_local
        tr = TorchDistTransport()
        v = g[f"r{rank}_vec"].copy()
        send = [np.zeros(len(ix)) for ix in gd[0]]
        for sb, ix in zip(send, gd[0]):
            orc.pack_fwd(v, sb, np.ascontiguousarray(ix, np.int64))
        recv = [torch.zeros(len(ix), dtype=torch.float64) for ix in od[0]]
        tr.exchange([torch.from_numpy(s) for s in send], gd[2], recv, od[2])
        f = v.copy()
        for rb, ix in zip(recv, od[0]):
            orc.unpack_fwd(rb.numpy(), f, np.ascontiguousarray(ix, np.int64), N)
        ok &= bool(np.array_equal(f, g[f"r{rank}_fwd"]))
        send = [np.zeros(len(ix)) for ix in od[0]]
        for sb, ix in zip(send, od[0]):
            orc.pack_rev(v, sb, np.ascontiguousarray(ix, np.int64), N)
        recv = [torch.zeros(len(ix), dtype=torch.float64) for ix in gd[0]]
        tr.exchange([torch.from_numpy(s) for s in send], od[2], recv, gd[2])
        rv = v.copy()
        for rb, ix in zip(recv, gd[0]):
            orc.unpack_rev(rb.numpy(), rv, np.ascontiguousarray(ix, np.int64))
        # (several ranks may add into one dof: the order of the adds is the order of the lists here
        #  and of the message arrival in the reference)
        rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))  # noqa: E731
        ok &= rel(rv, g[f"r{rank}_rev"]) < 1e-15
        # the same reverse round in the shared-last numbering (what box_setup hands the solvers):
        # ghosts_data lists renumbered, owned block permuted, ghost block in place
        perm, gd_p = utils.shared_last_numbering(N, v.size - N, gd)
        vp = np.empty_like(v)
        vp[perm] = v
        recv = [torch.zeros(len(ix), dtype=torch.float64) for ix in gd_p[0]]
        tr.exchange([torch.from_numpy(s) for s in send], od[2], recv, gd_p[2])
        for rb, ix in zip(recv, gd_p[0]):
            orc.unpack_rev(rb.numpy(), vp, np.ascontiguousarray(ix, np.int64))
        ok &= rel(vp[perm], g[f"r{rank}_rev"]) < 1e-15
        # mesh_size = min over ranks of the local hmin (cuda/demo_linear_box.py:103-108)
        ok &= utils.global_min(0.5 + rank) == 0.5 and utils.global_min(2.0 - rank) == 3.0 - world
        q.put((rank, ok))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name,world", [("r2", 2), ("u4", 4)])
def test_index_exchange_and_halo_rounds_over_gloo(golden_dir, name, world):
    """N>1 path on CPU: one process per rank, gloo backend, 127.0.0.1 rendezvous; the block
    partition on 2 ranks and the unstructured-like one on 4 (each rank a different neighbour set)."""
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, golden_dir, q, name)) for r in range(world)]
    [p.start() for p in procs]
    res = [q.get(timeout=240) for _ in procs]
    [p.join(timeout=60) for p in procs]
    assert sorted(res) == [(r, True) for r in range(world)]


# ---- substrate known answers -------------------------------------------------


@pytest.mark.parametrize("n", range(3, 9))
def test_gll_rule(n):
    x, w = S.gll_points_weights(n)
    assert abs(w.sum() - 1.0) < 1e-14 and x[0] == 0.0 and x[-1] == 1.0
    # exact for polynomials up to degree 2n-3
    for k in range(2 * n - 2):
        assert abs(np.dot(w, x**k) - 1.0 / (k + 1)) < 1e-13


@pytest.mark.parametrize("P", range(2, 8))
def test_derivative_table(P):
    tb = S.element_tables(P)
    D, x = tb.dphi_1D, tb.pts_1d
    assert np.abs(D.sum(axis=1)).max() < 1e-12  # constants
    for k in range(1, P + 1):
        assert np.abs(D @ x**k - k * x ** (k - 1)).max() < 1e-10


def test_facet_integration_domain_matches_box_facets():
    """utils.facet_integration_domain on a duck-typed DOLFINx topology gives the
    rows substrate.boundary_facets produces directly."""
    mesh = S.create_box((3, 2, 2))
    Nx, Ny, Nz = mesh.ncells
    ncell = Nx * Ny * Nz
    # number facets: per cell 6 local facets, shared facets de-duplicated via a dict
    key_of = {}
    c2f = np.zeros((ncell, 6), np.int32)
    f2c = {}

    def key(cx, cy, cz, lf):
        axis, side = S._FACE_AXIS[lf]
        pos = [cx, cy, cz]
        pos[axis] += side
        return (axis, tuple(pos))

    for cx in range(Nx):
        for cy in range(Ny):
            for cz in range(Nz):
                c = (cx * Ny + cy) * Nz + cz
                for lf in range(6):
                    k = key(cx, cy, cz, lf)
                    fid = key_of.setdefault(k, len(key_of))
                    c2f[c, lf] = fid
                    f2c.setdefault(fid, []).append(c)

    class Topo:
        dim = 3

        def connectivity(self, a, b):
            if (a, b) == (3, 2):
                return S.AdjacencyList(c2f.ravel(), np.arange(0, 6 * ncell + 1, 6))
            offs = np.cumsum([0] + [len(f2c[f]) for f in range(len(f2c))])
            return S.AdjacencyList(np.concatenate([f2c[f] for f in range(len(f2c))]), offs)

    class M:
        topology = Topo()

    for lf in range(6):
        want = S.boundary_facets(mesh, lf)
        fids = np.array([c2f[c, l] for c, l in want], np.int32)
        got = utils.facet_integration_domain(fids, M())
        assert np.array_equal(got, want)


def test_global_min_without_process_group():
    assert utils.global_min(0.25) == 0.25


def test_diffusivity_of_sound():
    w0, c0, a = 2 * np.pi * 1.1e6, 1480.0, 0.2
    assert utils.compute_diffusivity_of_sound(w0, c0, a) == pytest.approx(
        2 * (a / 20 * np.log(10)) * c0**3 / w0**2, rel=1e-15)


@pytest.mark.parametrize("ncells,perturb", [((5, 4, 6), 0.0), ((3, 3, 3), 0.2), ((1, 1, 1), 0.0), ((2, 1, 7), 0.1)])
def test_cell_colouring_is_a_valid_partition(ncells, perturb):
    """No two cells of a colour share a dof (checked on the FULL degree-3 dofmap although the
    colouring only looks at the 8 vertices per cell); the box colouring uses at most 8 colours."""
    from fenicsx_fus_gpu_b200 import substrate as S, utils

    mesh = S.create_box(ncells, perturb=perturb)
    dofmap = S.tensor_dofmap(mesh, 3)
    for colours in (utils.colour_cells(mesh.x_dofs), utils.colour_cells(mesh.x_dofs, seed=7),
                    S.box_cell_colours(mesh), utils.colour_cells(dofmap)):
        assert colours.shape == (mesh.num_cells,) and colours.min() >= 0
        for c in range(int(colours.max()) + 1):
            touched = dofmap[colours == c].ravel()
            assert np.unique(touched).size == touched.size
        perm, off = utils.colour_order(colours)
        assert off[0] == 0 and off[-1] == mesh.num_cells and np.all(np.diff(colours[perm]) >= 0)
        assert np.array_equal(np.sort(perm), np.arange(mesh.num_cells))
    assert S.box_cell_colours(mesh).max() < 8
    # colours of a part agree with the colours of the same cells in the whole box
    parts = S.partition_box((4, 4, 4), 2, 8)
    whole = S.box_cell_colours(S.create_box((4, 4, 4))).reshape(4, 4, 4)
    for p in parts:
        o, n = p.mesh.cell_origin, p.mesh.ncells
        assert np.array_equal(S.box_cell_colours(p.mesh).reshape(n),
                              whole[o[0]:o[0] + n[0], o[1]:o[1] + n[1], o[2]:o[2] + n[2]])
    assert utils.colour_cells(np.zeros((0, 8), np.int32)).size == 0


def test_compute_eval_params_and_interpolation_known_answers():
    """Point location (the reference's compute_eval_params, cuda/utils.py:117-154) against a
    brute-force search, and the interpolant against polynomials it must reproduce exactly."""
    from fenicsx_fus_gpu_b200 import sampling as sp, substrate as S
    from oracle import oracle as orc

    mesh = S.create_box((5, 4, 3), (1.0, 0.8, 0.6), perturb=0.2, seed=2)
    rng = np.random.default_rng(0)
    pts = rng.uniform([-0.1, -0.1, -0.1], [1.1, 0.9, 0.7], (400, 3))
    xp, cells = sp.compute_eval_params(mesh, pts.T, np.float64)
    assert xp.shape == (len(cells), 3) and 0 < len(cells) < 400
    cc = mesh.x_g[mesh.x_dofs]
    # brute force: pull every point back into every cell
    nc = mesh.num_cells
    found = np.full(400, -1)
    for c in range(nc):
        X, ok = sp.pull_back(np.broadcast_to(cc[c], (400, 8, 3)), pts)
        hit = ok & np.all((X >= -1e-9) & (X <= 1 + 1e-9), axis=1) & (found < 0)
        found[hit] = c
    assert np.array_equal(np.nonzero(found >= 0)[0], np.nonzero(np.isin(pts, xp).all(axis=1))[0])
    assert np.array_equal(found[found >= 0], np.asarray(cells))
    # polynomial of degree <= P in each variable on an affine mesh: reproduced to rounding
    P = 4
    tb = S.element_tables(P)
    box = S.create_box((4, 3, 2), (1.0, 0.8, 0.6))
    dm = S.tensor_dofmap(box, P)
    xd = S.dof_coordinates(box, dm, tb)
    f = lambda x: 1 + x[:, 0] ** 4 * x[:, 1] - x[:, 2] ** 3 + x[:, 0] * x[:, 1] ** 2 * x[:, 2] ** 4  # noqa: E731
    xp, cells = sp.compute_eval_params(box, pts.T, np.float64)
    X, phi = sp.reference_basis(box, xp, cells, tb.pts_1d)
    assert np.abs(phi.sum(axis=2) - 1).max() < 1e-13  # partition of unity
    assert np.abs(orc.eval_points(f(xd), dm, cells, phi) - f(xp)).max() < 1e-13
    # nodes are hit exactly: sampling at dof coordinates returns the dof values
    some = rng.choice(xd.shape[0], 50, replace=False)
    xp2, c2 = sp.compute_eval_params(box, xd[some].T, np.float64)
    assert len(c2) == 50
    _, phi2 = sp.reference_basis(box, xp2, c2, tb.pts_1d)
    u = rng.standard_normal(xd.shape[0])
    assert np.abs(orc.eval_points(u, dm, c2, phi2) - u[some]).max() < 1e-12
    # nothing to find / nothing to search
    e, c = sp.compute_eval_params(box, np.array([[5.0], [5.0], [5.0]]), np.float32)
    assert e.shape == (0, 3) and e.dtype == np.float32 and c == []
    assert sp.compute_eval_params(box, np.zeros((3, 0)), np.float64)[1] == []


def test_shim_modules_export_every_name_the_reference_scripts_import():
    """shim/{operators,scatterer,precompute,utils}.py first on sys.path: the bare-name imports of the
    reference's cuda/ scripts (demo_linear_box.py:21-38, demo_linear_piston.py, demo_nonlinear_bowl.py,
    time_operators.py, test_operators.py, test_scatterer.py) resolve to this package."""
    import importlib
    import os
    import sys

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "shim")
    wanted = {
        "operators": ["mass_operator", "stiffness_operator", "axpy", "copy", "fill", "pointwise_divide", "square"],
        "scatterer": ["scatter_forward", "scatter_reverse", "pack_fwd", "unpack_fwd", "pack_rev", "unpack_rev"],
        "precompute": ["compute_scaled_jacobian_determinant", "compute_scaled_geometrical_factor",
                       "compute_boundary_facets_scaled_jacobian_determinant"],
        "utils": ["compute_scatterer_data", "facet_integration_domain", "compute_eval_params",
                  "compute_diffusivity_of_sound"],
    }
    saved = {m: sys.modules.pop(m, None) for m in wanted}
    sys.path.insert(0, shim)
    try:
        for mod, names in wanted.items():
            m = importlib.import_module(mod)
            assert os.path.dirname(os.path.abspath(m.__file__)) == shim
            for n in names:
                assert hasattr(m, n), f"{mod}.{n}"
    finally:
        sys.path.remove(shim)
        for mod in wanted:
            sys.modules.pop(mod, None)
            if saved[mod] is not None:
                sys.modules[mod] = saved[mod]


def test_eval_params_keep_only_the_points_of_this_rank():
    """compute_eval_params on the parts of a partitioned box: every interior point is found by exactly
    the ranks whose cells contain it (shared faces: both), as `points_on_proc` of cuda/utils.py:139-150."""
    from fenicsx_fus_gpu_b200 import sampling as sp

    parts = S.partition_box((4, 4, 4), 2, 8, lengths=(1.0, 1.0, 1.0))
    rng = np.random.default_rng(2)
    pts = rng.uniform(0.01, 0.99, (200, 3))
    pts = pts[np.all(np.abs(pts - 0.5) > 1e-3, axis=1)]  # keep clear of the rank interfaces
    count = np.zeros(pts.shape[0], int)
    for p in parts:
        xp, cells = sp.compute_eval_params(p.mesh, pts.T, np.float64)
        assert len(cells) == xp.shape[0] and all(0 <= c < p.mesh.num_cells for c in cells)
        lo = np.array(p.mesh.cell_origin) / 4.0
        hi = lo + np.array(p.mesh.ncells) / 4.0
        inside = np.all((pts > lo) & (pts < hi), axis=1)
        assert np.array_equal(xp, pts[inside])
        count += inside
    assert np.all(count == 1)


def test_partition_properties_on_random_grids():
    """Random cell counts / rank grids: owned ranges tile the global numbering, every dof has one
    owner, ghost owners really own their dofs, dest-rank lists mirror the ghost lists."""
    rng = np.random.default_rng(11)
    for _ in range(6):
        grid = tuple(int(v) for v in rng.integers(1, 4, 3))
        ncells = tuple(int(g * rng.integers(1, 3) + rng.integers(0, 2)) for g in grid)
        P = int(rng.integers(1, 4))
        R = grid[0] * grid[1] * grid[2]
        parts = S.partition_box(ncells, P, R, grid=grid)
        ranges = [p.index_map.local_range for p in parts]
        assert ranges[0][0] == 0 and ranges[-1][1] == parts[0].index_map.size_global == S.num_dofs(ncells, P)
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        ghosted_by = {}
        for p in parts:
            im = p.index_map
            for g, o in zip(im.ghosts, im.owners):
                assert ranges[o][0] <= g < ranges[o][1] and o != p.rank
                ghosted_by.setdefault((int(o), int(g) - ranges[o][0]), set()).add(p.rank)
            assert p.dofmap.min() >= 0 and p.dofmap.max() == im.size_local + im.num_ghosts - 1
        for p in parts:
            dest = p.index_map.index_to_dest_ranks()
            for i in range(p.index_map.size_local):
                assert set(int(r) for r in dest.links(i)) == ghosted_by.get((p.rank, i), set())


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_tensor_tables(dt):
    """(K1, w1) of a tensor-product rule; None (rect_tables: ValueError) for any other weights."""
    from fenicsx_fus_gpu_b200 import operators as ops

    tb = S.element_tables(4, "basix", dt)
    k1, w1 = ops.tensor_tables(tb.dphi_1D, tb.wts, dt)
    assert k1.dtype == w1.dtype == dt and k1.shape == (5, 5)
    tol = 1e-12 if dt == np.float64 else 1e-5
    np.testing.assert_allclose(np.einsum("i,j,k->ijk", w1, w1, w1).ravel(), tb.wts, rtol=tol)
    np.testing.assert_allclose(k1, k1.T, rtol=tol, atol=tol)
    np.testing.assert_allclose(k1.sum(axis=1), 0.0, atol=100 * tol)  # K1 annihilates constants
    rng = np.random.default_rng(0)
    for w in (rng.uniform(1, 2, 125), np.zeros(125), -np.asarray(tb.wts)):
        assert ops.tensor_tables(tb.dphi_1D, w, dt) is None
        with pytest.raises(ValueError):
            ops.rect_tables(tb.dphi_1D, w, dt)
