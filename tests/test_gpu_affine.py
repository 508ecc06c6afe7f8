"""GPU parity of the affine-cell path: cells with a constant Jacobian keep 6 (+1)
geometric factors instead of 6 (+1) n^3 (``precompute.compress_geometry``, the
``fus_stiffness_affine`` / ``fus_stiffness_westervelt_affine`` kernels, the solvers'
``geometry="auto"``).  The reference has no such path: the oracle is the reference
algorithm with the FULL tables (numba-cpu/operators.py:71-227), same tolerances
(rel-L2 <= 1e-12 float64, <= 1e-5 float32)."""

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

TOL = {"f64": 1e-12, "f32": 1e-5}
SHEAR = np.array([[1.0, 0.15, -0.1], [0.05, 0.9, 0.2], [-0.12, 0.07, 1.1]])


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def sheared_box(ncells, L, dt, jitter_below=None, seed=0, shear=True):
    """Box of parallelepipeds (every cell affine, all six entries of G non-zero); with
    ``jitter_below`` the vertices with x < jitter_below * L are perturbed, which makes the
    cells touching them non-affine.  Returns (mesh, expected affine mask)."""
    from fenicsx_fus_gpu_b200 import substrate as S

    mesh = S.create_box(ncells, L, dtype=np.float64)
    x = mesh.x_g.copy()
    moved = np.zeros(x.shape[0], bool)
    if jitter_below is not None:
        rng = np.random.default_rng(seed)
        h = L / max(mesh.ncells)
        moved = x[:, 0] < jitter_below * L
        x[moved] += rng.uniform(-0.15, 0.15, (int(moved.sum()), 3)) * h
    mesh.x_g = np.ascontiguousarray(x @ SHEAR.T if shear else x, dtype=dt)
    return mesh, ~moved[mesh.x_dofs].any(axis=1)


def test_compress_geometry_classifies_and_reproduces():
    import problems
    from fenicsx_fus_gpu_b200 import precompute as pre, substrate as S

    P = 3
    tb = S.element_tables(P, "basix", np.float64)
    mesh, expect = sheared_box((5, 4, 3), 1.0, np.float64, jitter_below=0.45)
    assert 0 < expect.sum() < expect.size
    G, detJ = problems.geometry(mesh, tb, np.float64)
    affine, Gc, detJc = pre.compress_geometry(d(G), d(detJ), d(tb.wts))
    affine, Gc, detJc = affine.cpu().numpy().astype(bool), Gc.cpu().numpy(), detJc.cpu().numpy()
    assert np.array_equal(affine, expect)
    assert rel_l2(Gc[affine][:, None, :] * tb.wts[None, :, None], G[affine]) < 1e-14
    assert rel_l2(detJc[affine][:, None] * tb.wts[None, :], detJ[affine]) < 1e-14
    assert np.abs(Gc[affine][:, [1, 2, 4]]).min() > 0  # the shear exercises the off-diagonal factors
    # without detJ, and in float32
    a2, Gc2, _ = pre.compress_geometry(d(G.astype(np.float32)), None, d(tb.wts.astype(np.float32)))
    assert np.array_equal(a2.cpu().numpy().astype(bool), expect)
    assert rel_l2(Gc2.cpu().numpy(), Gc) < 1e-6


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_affine_stiffness_vs_oracle(P, tag):
    import problems
    from fenicsx_fus_gpu_b200 import operators as ops, precompute as pre, substrate as S
    from oracle import oracle as orc

    dt = np.float64 if tag == "f64" else np.float32
    tb = S.element_tables(P, "basix", dt)
    N = (9, 5, 4) if P <= 4 else (4, 3, 3)  # several persistent-CTA batches + a ragged last one
    mesh, expect = sheared_box(N, 1.0, dt)
    assert expect.all()
    dofmap = S.tensor_dofmap(mesh, P)
    nd, Nc, n = int(dofmap.max()) + 1, dofmap.shape[0], P + 1
    G, _ = problems.geometry(mesh, tb, dt)
    rng = np.random.default_rng(P)
    x = rng.standard_normal(nd).astype(dt)
    coeff = rng.uniform(0.5, 2.0, Nc).astype(dt)
    y_ref = np.zeros(nd, dt)
    orc.stiffness_operator(P, x, coeff, y_ref, G, dofmap, tb.dphi_1D)

    affine, Gc, _ = pre.compress_geometry(d(G), None, d(tb.wts))
    assert bool(affine.all())
    y = torch.zeros(nd, dtype=d(x).dtype, device="cuda")
    K = ops.stiffness_operator_affine(P, dt)
    K[Nc, (n, n, n)](d(x), d(coeff), y, Gc, d(tb.wts), d(dofmap), tb.dphi_1D)
    assert rel_l2(y.cpu().numpy(), y_ref) < TOL[tag]
    K[Nc, (n, n, n)](d(x), d(coeff), y, Gc, d(tb.wts), d(dofmap), d(tb.dphi_1D))  # accumulates
    assert rel_l2(0.5 * y.cpu().numpy(), y_ref) < TOL[tag]
    with pytest.raises(Exception):
        K[Nc, (n, n, n)](d(x), d(coeff), y, Gc[:-1], d(tb.wts), d(dofmap), tb.dphi_1D)


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_rect_stiffness_vs_oracle(P, tag):
    """Axis-aligned cells of unequal sizes: the decoupled 1-D-stiffness kernel against the
    reference algorithm with the full tables."""
    import problems
    from fenicsx_fus_gpu_b200 import operators as ops, precompute as pre, substrate as S
    from oracle import oracle as orc

    dt = np.float64 if tag == "f64" else np.float32
    tb = S.element_tables(P, "basix", dt)
    N = (9, 5, 4) if P <= 4 else (4, 3, 3)
    mesh = S.create_box(N, (1.0, 0.7, 1.9), dtype=np.float64)
    x = mesh.x_g.copy()  # grade the grid: still axis-aligned, every cell a different box
    for ax in range(3):
        x[:, ax] = x[:, ax] + 0.08 * np.sin(2.5 * x[:, ax])
    mesh.x_g = np.ascontiguousarray(x, dtype=dt)
    dofmap = S.tensor_dofmap(mesh, P)
    nd, Nc, n = int(dofmap.max()) + 1, dofmap.shape[0], P + 1
    G, _ = problems.geometry(mesh, tb, dt)
    rng = np.random.default_rng(P)
    xv = rng.standard_normal(nd).astype(dt)
    coeff = rng.uniform(0.5, 2.0, Nc).astype(dt)
    y_ref = np.zeros(nd, dt)
    orc.stiffness_operator(P, xv, coeff, y_ref, G, dofmap, tb.dphi_1D)
    affine, Gc, _ = pre.compress_geometry(d(G), None, d(tb.wts))
    assert bool(affine.all())
    assert float(Gc[:, [1, 2, 4]].abs().max()) <= 1e-5 * float(Gc[:, [0, 3, 5]].abs().max())
    y = torch.zeros(nd, dtype=d(xv).dtype, device="cuda")
    K = ops.stiffness_operator_rect(P, dt)
    K[Nc, (n, n, n)](d(xv), d(coeff), y, Gc, tb.wts, d(dofmap), tb.dphi_1D)
    assert rel_l2(y.cpu().numpy(), y_ref) < TOL[tag]
    K[Nc, (n, n, n)](d(xv), d(coeff), y, Gc, tb.wts, d(dofmap), tb.dphi_1D)  # accumulates
    assert rel_l2(0.5 * y.cpu().numpy(), y_ref) < TOL[tag]
    with pytest.raises(ValueError):
        ops.rect_tables(tb.dphi_1D, rng.uniform(1, 2, n**3), dt)  # not a tensor-product rule


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_solver_rect_tables_match_operator(P, tag):
    """The (K1, w1) a geometry='auto' solver uploads for its rectilinear cells are bit for bit those
    of ``operators.rect_tables`` on the weights and derivative table in the solver's float type."""
    import problems
    import test_gpu_solver as tgs
    from fenicsx_fus_gpu_b200 import operators as ops

    dtt = np.float64 if tag == "f64" else np.float32
    dd = problems.linear_problem(P, 2, 0.01, dtt, perturb=0.0)  # axis-aligned: every cell rectilinear
    s = tgs._linear_solver(dd, dtt, geometry="auto", weights=dd.tb.wts, use_graph=False)
    assert s.nrect == s.ncells > 0
    k1, w1 = ops.rect_tables(np.asarray(dd.tb.dphi_1D, dtt), np.asarray(dd.tb.wts, dtt), dtt)
    for got, want in zip(s._rect_tables, (k1, w1)):
        assert got.dtype == want.dtype == dtt and got.tobytes() == want.tobytes()


@pytest.mark.parametrize("P,N,tag,jitter,shear", [(4, 5, "f64", None, True), (4, 5, "f64", 0.5, True),
                                                  (3, 6, "f32", 0.5, True), (5, 3, "f64", 0.4, True),
                                                  (2, 7, "f64", 1.1, True), (4, 5, "f64", None, False),
                                                  (4, 5, "f64", 0.5, False), (6, 3, "f32", 0.4, False)])
def test_linear_rk4_auto_geometry_vs_oracle(P, N, tag, jitter, shear):
    """All-affine, mixed and no-affine-cell meshes through geometry='auto'; without the shear
    the affine cells are rectilinear and take the decoupled kernel."""
    import problems
    import test_gpu_solver as tgs
    from fenicsx_fus_gpu_b200 import substrate as S

    dtt = np.float64 if tag == "f64" else np.float32
    L = 0.01
    mesh, expect = sheared_box(N, L, dtt, jitter_below=jitter, seed=P, shear=shear)
    dofmap = S.tensor_dofmap(mesh, P)
    dd = problems.linear_problem(P, N, L, dtt, mesh=mesh, dofmap=dofmap, ndofs=int(dofmap.max()) + 1)
    dt = problems.cfl_dt(P, 0.8 * L / N, dd.c0, dd.f0)
    nsteps = 10
    u_ref, v_ref = tgs._oracle_linear(dd, dt, nsteps, dtt)
    assert np.linalg.norm(u_ref) > 0
    for use_graph in (True, False):
        s = tgs._linear_solver(dd, dtt, geometry="auto", weights=dd.tb.wts, use_graph=use_graph)
        assert s.naff == int(expect.sum()) and s.nrect == (0 if shear else s.naff)
        s.init()
        s.rk4(0.0, dt, nsteps)
        assert rel_l2(s.u.cpu().numpy(), u_ref) < TOL[tag]
        assert rel_l2(s.v.cpu().numpy(), v_ref) < TOL[tag]
    with pytest.raises(ValueError):
        tgs._linear_solver(dd, dtt, geometry="auto")  # needs the quadrature weights


@pytest.mark.parametrize("P,N,tag,jitter,shear", [(4, 4, "f64", None, True), (4, 4, "f64", 0.5, True),
                                                  (3, 5, "f32", 0.5, True), (4, 4, "f64", None, False),
                                                  (4, 4, "f64", 0.5, False), (5, 3, "f32", None, False)])
def test_westervelt_rk4_auto_geometry_vs_oracle(P, N, tag, jitter, shear):
    import problems
    from fenicsx_fus_gpu_b200 import substrate as S
    from fenicsx_fus_gpu_b200.solver import WesterveltSpectral3D, westervelt_source
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32
    L = 0.006
    mesh, expect = sheared_box(N, L, dtt, jitter_below=jitter, seed=3, shear=shear)
    dofmap = S.tensor_dofmap(mesh, P)
    q = problems.westervelt_problem(P, N, L, dtt, mesh=mesh, dofmap=dofmap, ndofs=int(dofmap.max()) + 1)
    dt = problems.cfl_dt(P, 0.8 * L / N, q.c0, q.f0, cfl=0.4)
    nsteps = 8
    ones = np.ones(q.ndofs, dtt)
    m0 = np.zeros(q.ndofs, dtt)
    orc.mass_operator(ones, q.cell_coeff1, m0, q.detJ, q.dofmap)
    orc.mass_operator(ones, q.facet_coeff1_2, m0, q.detJ_f2, q.bfacet_dofmap2)
    prob = orc.WesterveltProblem(q.P, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff2, q.cell_coeff3,
                                 q.cell_coeff4, q.cell_coeff5, m0, q.bfacet_dofmap1, q.detJ_f1,
                                 q.facet_coeff1_1, q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2,
                                 q.facet_coeff2_2, q.f0, q.p0, q.c0)
    u_ref, v_ref = np.zeros(q.ndofs, dtt), np.zeros(q.ndofs, dtt)
    orc.westervelt_rk4(prob, u_ref, v_ref, 0.0, dt, nsteps)
    assert np.linalg.norm(u_ref) > 0
    s = WesterveltSpectral3D(
        q.P, dtt, q.ndofs, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
        q.cell_coeff3, q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1,
        q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2,
        source=lambda t: westervelt_source(t, q.f0, q.p0, q.c0), geometry="auto", weights=q.tb.wts)
    assert s.naff == int(expect.sum()) and s.nrect == (0 if shear else s.naff)
    s.init()
    s.rk4(0.0, dt, nsteps)
    assert rel_l2(s.u.cpu().numpy(), u_ref) < TOL[tag]
    assert rel_l2(s.v.cpu().numpy(), v_ref) < TOL[tag]
    # the reference's data flow (cell-mass pair over the cells each stage) through the compressed kernels
    s = WesterveltSpectral3D(
        q.P, dtt, q.ndofs, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
        q.cell_coeff3, q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1,
        q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2,
        source=lambda t: westervelt_source(t, q.f0, q.p0, q.c0), geometry="auto", weights=q.tb.wts,
        mass_form="cells")
    s.init()
    s.rk4(0.0, dt, nsteps)
    assert rel_l2(s.u.cpu().numpy(), u_ref) < TOL[tag]
    assert rel_l2(s.v.cpu().numpy(), v_ref) < TOL[tag]
