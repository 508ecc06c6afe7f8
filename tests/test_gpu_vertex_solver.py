"""The time loops with geometry="vertex": no (Nc, n^3) geometry table anywhere.

* host side (no GPU): ``precompute.compress_trilinear`` classifies and compresses the cells from
  the 36 trilinear coefficients exactly as ``compress_geometry`` plus the solvers' rectilinear
  rule do from the full ``G`` table;
* CUDA: the Westervelt cell form and the lumped mass on trilinear cells against their streamed
  twins and a float64 reference; the solvers against the oracle on fully trilinear meshes and on
  meshes that mix rectilinear, affine and trilinear cells; graph replay against eager steps;
  emulated ranks with the peer-memory halo in every split mode; the memory the mode saves; a demo.

Tolerances: rel-L2 <= 1e-12 (float64), <= 1e-5 (float32) for the solvers (as tests/test_gpu_affine.py).
"""

import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from fenicsx_fus_gpu_b200 import precompute as pre  # noqa: E402
from fenicsx_fus_gpu_b200 import substrate as S  # noqa: E402

torch = pytest.importorskip("torch")

TOL = {"f64": 1e-12, "f32": 1e-5}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _tc_host(tb, mesh, dt):
    M = pre.trilinear_expansion(tb.dphi, tb.pts)
    return np.einsum("dmv,cvk->cdmk", M, mesh.x_g[mesh.x_dofs].astype(np.float64)).reshape(-1, 36).astype(dt)


def _mesh(case, N, dt, seed=0):
    """(mesh, expected affine mask): 'sheared' (every cell affine), 'jittered' (vertices with
    x < 0.45 L moved: the cells touching them are trilinear), 'box' (unperturbed: rectilinear)."""
    from test_gpu_affine import sheared_box

    if case == "sheared":
        return sheared_box(N, 1.0, dt)
    if case == "jittered":
        return sheared_box(N, 1.0, dt, jitter_below=0.45, seed=seed)
    return sheared_box(N, 1.0, dt, shear=False)


def mixed_box(N, L, dt, seed=0):
    """Rectilinear, affine and trilinear cells in one mesh: the upper half (z above the middle
    grid plane) is sheared in x, which keeps its cells affine but not axis-aligned; vertices with
    x < 0.3 L are jittered, which makes the cells touching them trilinear."""
    mesh = S.create_box(N, L, dtype=np.float64)
    x = mesh.x_g.copy()
    z0 = (N[2] // 2) * L / N[2]
    x[:, 0] += 0.3 * np.maximum(x[:, 2] - z0, 0.0)
    rng = np.random.default_rng(seed)
    h = L / max(N)
    moved = x[:, 0] < 0.3 * L
    x[moved] += rng.uniform(-0.15, 0.15, (int(moved.sum()), 3)) * h
    mesh.x_g = np.ascontiguousarray(x, dtype=dt)
    return mesh


# --------------------------------------------------------------------------- #
# host side
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("case", ["sheared", "jittered", "box"])
@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_compress_trilinear_vs_geometry_tables(case, P, tag):
    """Masks identical to compress_geometry's rule applied to the oracle's G (and the solver's
    rectilinear rule on top); Gc and detJc equal to the weight-normalised tables."""
    import problems

    dt = np.float64 if tag == "f64" else np.float32
    tb = S.element_tables(P, "basix", dt)
    mesh, expect = _mesh(case, (5, 4, 3), dt, seed=P)
    G, detJ = problems.geometry(mesh, tb, dt)
    w = tb.wts.astype(np.float64)
    tol = 2048.0 * float(np.finfo(dt).eps)
    Gn, Jn = G.astype(np.float64) / w[None, :, None], detJ.astype(np.float64) / w[None, :]
    Gm, Jm = Gn.mean(axis=1), Jn.mean(axis=1)
    aff_ref = ((np.abs(Gn - Gm[:, None]).max(axis=(1, 2)) <= tol * np.abs(Gm).max(axis=1))
               & (np.abs(Jn - Jm[:, None]).max(axis=1) <= tol * np.abs(Jm)))
    assert np.array_equal(aff_ref, expect)

    affine, Gc, detJc = pre.compress_trilinear(torch.from_numpy(_tc_host(tb, mesh, dt)))
    affine, Gc, detJc = affine.numpy().astype(bool), Gc.numpy(), detJc.numpy()
    assert Gc.dtype == dt and detJc.dtype == dt
    assert np.array_equal(affine, aff_ref)

    def rect(g):
        return np.abs(g[:, [1, 2, 4]]).max(axis=1) <= tol * np.abs(g[:, [0, 3, 5]]).max(axis=1)

    assert np.array_equal(affine & rect(Gc), aff_ref & rect(Gm))
    if case == "box":
        assert rect(Gc).all()
    bar = 1e-14 if tag == "f64" else 1e-6
    if affine.any():
        assert rel_l2(Gc[affine], Gm[affine]) < bar
        assert rel_l2(detJc[affine], Jm[affine]) < bar


# --------------------------------------------------------------------------- #
# CUDA
# --------------------------------------------------------------------------- #
def _gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _kernel_problem(P, tag, N):
    dt = np.float64 if tag == "f64" else np.float32
    tb = S.element_tables(P, "basix", dt)
    n = P + 1
    mesh = S.create_box(N, (1.0, 0.7, 0.9), dtype=dt, perturb=0.25, seed=P)
    dofmap = S.tensor_dofmap(mesh, P)
    nc, nd = mesh.num_cells, S.num_dofs(N, P)
    tdt = torch.float64 if tag == "f64" else torch.float32
    G = torch.empty((nc, n**3, 6), dtype=tdt, device="cuda")
    detJ = torch.empty((nc, n**3), dtype=tdt, device="cuda")
    pre.compute_geometry(G, detJ, (d(mesh.x_dofs), d(mesh.x_g)), nc, d(tb.dphi), d(tb.wts))
    Tc = pre.trilinear_coefficients((mesh.x_dofs, mesh.x_g), nc, tb.dphi, tb.pts)
    return dt, tb, mesh, d(dofmap), nc, nd, G, detJ, Tc


def _tables(P, dt, tb):
    from fenicsx_fus_gpu_b200._lib import check, current_stream, fn

    x1, w1 = np.ascontiguousarray(tb.pts_1d, dt), np.ascontiguousarray(tb.wts_1d, dt)
    dphi = np.ascontiguousarray(tb.dphi_1D, dt)
    check(fn("fus_set_dphi", dt)(P, dphi.ctypes.data, current_stream()), "fus_set_dphi")
    check(fn("fus_set_vertex_tables", dt)(P, x1.ctypes.data, w1.ctypes.data, current_stream()), "fus_set_vertex_tables")
    torch.cuda.synchronize()


# cell ranges (c0, m) of one launch: single cells, around the batch sizes (1..14 cells), ragged sub-ranges
RANGES = [(0, 1), (2, 3), (1, 5), (0, 8), (3, 13), (0, 14), (5, 15), (0, 29)]


@pytest.mark.gpu
@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_westervelt_vertex_kernel_vs_streamed(P, tag):
    """b += K(c3; un) + K(c4; vn) + M(c5; vn^2), m += M(c2; un): trilinear form against the
    streamed form with G and detJ from compute_geometry, for both outputs, on cell sub-ranges."""
    from fenicsx_fus_gpu_b200._lib import FUS_TABLES_RESIDENT, check, current_stream, fn

    _gpu()
    dt, tb, mesh, dm, nc, nd, G, detJ, Tc = _kernel_problem(P, tag, (5, 4, 3) if P <= 4 else (4, 3, 3))
    _tables(P, dt, tb)
    rng = np.random.default_rng(P)
    un, vn = d(rng.standard_normal(nd).astype(dt)), d(rng.standard_normal(nd).astype(dt))
    c2, c3, c4, c5 = (d(rng.uniform(lo, hi, nc).astype(dt)) for lo, hi in ((-2, -1), (0.5, 2), (-1, 1), (1, 3)))
    bar = 1e-13 if tag == "f64" else 1e-5
    for c0, m in RANGES + [(0, nc), (nc // 3, nc - nc // 3 - 1)]:
        m = min(m, nc - c0)
        out = []
        for name, geo in (("fus_stiffness_westervelt", (G, detJ)), ("fus_stiffness_westervelt_vertex", (Tc,))):
            mv, b = torch.zeros(nd, dtype=un.dtype, device="cuda"), torch.zeros(nd, dtype=un.dtype, device="cuda")
            sp = lambda t: t[c0:].data_ptr()  # noqa: E731
            check(fn(name, dt)(un.data_ptr(), sp(c3), vn.data_ptr(), sp(c4), sp(c2), sp(c5), mv.data_ptr(), b.data_ptr(),
                               *(sp(t) for t in geo), sp(dm), None, m, P, FUS_TABLES_RESIDENT, current_stream()), name)
            out.append((mv.cpu().numpy(), b.cpu().numpy()))
        (m_ref, b_ref), (m_v, b_v) = out
        assert rel_l2(b_v, b_ref) < bar, (c0, m)
        assert rel_l2(m_v, m_ref) < bar, (c0, m)
    with pytest.raises(Exception):  # no uncoloured-scatter variant of the cell-mass pair
        check(fn("fus_stiffness_westervelt_vertex", dt)(un.data_ptr(), c3.data_ptr(), vn.data_ptr(), c4.data_ptr(),
                                                        c2.data_ptr(), c5.data_ptr(), un.data_ptr(), vn.data_ptr(),
                                                        Tc.data_ptr(), dm.data_ptr(), None, nc, P, 3,
                                                        current_stream()), "fus_stiffness_westervelt_vertex")


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 4, 7])
def test_westervelt_vertex_kernel_vs_float64_reference(P):
    """The f64 kernel against the oracle's streamed operators in float64 (numpy / C), on the same
    jittered mesh."""
    import problems
    from fenicsx_fus_gpu_b200._lib import check, current_stream, fn
    from oracle import oracle as orc

    _gpu()
    dt = np.float64
    tb = S.element_tables(P, "basix", dt)
    N = (4, 3, 3)
    mesh = S.create_box(N, (1.0, 0.7, 0.9), dtype=dt, perturb=0.25, seed=P)
    dofmap = S.tensor_dofmap(mesh, P)
    nc, nd = mesh.num_cells, S.num_dofs(N, P)
    G, detJ = problems.geometry(mesh, tb, dt)
    rng = np.random.default_rng(P + 10)
    un, vn = rng.standard_normal(nd), rng.standard_normal(nd)
    c2, c3, c4, c5 = (rng.uniform(lo, hi, nc) for lo, hi in ((-2, -1), (0.5, 2), (-1, 1), (1, 3)))
    b_ref, m_ref = np.zeros(nd), np.zeros(nd)
    orc.stiffness_operator(P, un, c3, b_ref, G, dofmap, tb.dphi_1D)
    orc.stiffness_operator(P, vn, c4, b_ref, G, dofmap, tb.dphi_1D)
    orc.mass_operator(vn * vn, c5, b_ref, detJ, dofmap)
    orc.mass_operator(un, c2, m_ref, detJ, dofmap)
    _tables(P, dt, tb)
    Tc = pre.trilinear_coefficients((mesh.x_dofs, mesh.x_g), nc, tb.dphi, tb.pts)
    m, b = torch.zeros(nd, dtype=torch.float64, device="cuda"), torch.zeros(nd, dtype=torch.float64, device="cuda")
    args = [d(a) for a in (un, c3, vn, c4, c2, c5)] + [m, b, Tc, d(dofmap), d(tb.dphi_1D)]  # alive until the launch
    check(fn("fus_stiffness_westervelt_vertex", dt)(*(a.data_ptr() for a in args), nc, P, 0, current_stream()),
          "fus_stiffness_westervelt_vertex")
    assert rel_l2(b.cpu().numpy(), b_ref) < 1e-13
    assert rel_l2(m.cpu().numpy(), m_ref) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_mass_vertex_vs_mass_with_detj(P, tag):
    from fenicsx_fus_gpu_b200._lib import FusError, check, current_stream, fn

    _gpu()
    dt, tb, mesh, dm, nc, nd, G, detJ, Tc = _kernel_problem(P, tag, (5, 4, 3) if P <= 4 else (4, 3, 3))
    _tables(P, dt, tb)
    rng = np.random.default_rng(P)
    x = d(rng.standard_normal(nd).astype(dt))
    c = d(rng.uniform(0.5, 2.0, nc).astype(dt))
    bar = 1e-13 if tag == "f64" else 1e-5
    for c0, m in [(0, nc), (3, 13), (1, 1)]:
        y_ref, y = torch.zeros(nd, dtype=x.dtype, device="cuda"), torch.zeros(nd, dtype=x.dtype, device="cuda")
        check(fn("fus_mass", dt)(x.data_ptr(), c[c0:].data_ptr(), y_ref.data_ptr(), detJ[c0:].data_ptr(),
                                 dm[c0:].data_ptr(), m, (P + 1) ** 3, current_stream()), "fus_mass")
        check(fn("fus_mass_vertex", dt)(x.data_ptr(), c[c0:].data_ptr(), y.data_ptr(), Tc[c0:].data_ptr(),
                                        dm[c0:].data_ptr(), m, P, current_stream()), "fus_mass_vertex")
        assert rel_l2(y.cpu().numpy(), y_ref.cpu().numpy()) < bar, (c0, m)
    with pytest.raises(FusError):
        check(fn("fus_mass_vertex", dt)(x.data_ptr(), c.data_ptr(), x.data_ptr(), Tc.data_ptr(), dm.data_ptr(), nc, 8,
                                        current_stream()), "fus_mass_vertex")


# --------------------------------------------------------------------------- #
# solvers
# --------------------------------------------------------------------------- #
def _trilinear(q, dtt):
    return (pre.trilinear_coefficients((q.mesh.x_dofs, q.mesh.x_g), q.mesh.num_cells, q.tb.dphi, q.tb.pts),
            q.tb.pts_1d, q.tb.wts_1d)


def _vertex_kw(q, dtt):
    return dict(geometry="vertex", weights=q.tb.wts, trilinear=_trilinear(q, dtt))


def _counts(s):
    return s.nrect, s.naff - s.nrect, s.ntri


MESHES = [("trilinear", 4, 4, "f64"), ("trilinear", 3, 4, "f32"), ("mixed", 4, 6, "f64"), ("mixed", 2, 6, "f32")]


def _problem(kind, P, N, dtt, L, westervelt=False):
    import problems

    if kind == "trilinear":
        mesh = S.create_box((N,) * 3, L, dtype=dtt, perturb=0.12, seed=P)
    else:
        mesh = mixed_box((N,) * 3, L, dtt, seed=P)
    dofmap = S.tensor_dofmap(mesh, P)
    build = problems.westervelt_problem if westervelt else problems.linear_problem
    return build(P, N, L, dtt, mesh=mesh, dofmap=dofmap, ndofs=int(dofmap.max()) + 1)


def _check_kinds(s, kind):
    nrect, naff, ntri = _counts(s)
    if kind == "trilinear":
        assert ntri == s.ncells
    else:
        assert nrect > 0 and naff > 0 and ntri > 0, (nrect, naff, ntri)
    assert s.G is None and s.detJ is None


@pytest.mark.gpu
@pytest.mark.parametrize("kind,P,N,tag", MESHES)
def test_linear_rk4_and_leapfrog_vertex_vs_oracle(kind, P, N, tag):
    import problems
    import test_gpu_leapfrog as tgl
    import test_gpu_solver as tgs
    from fenicsx_fus_gpu_b200.solver import LinearLeapfrog3D

    _gpu()
    dtt = np.float64 if tag == "f64" else np.float32
    L = 0.01
    q = _problem(kind, P, N, dtt, L)
    dt = problems.cfl_dt(P, 0.7 * L / N, q.c0, q.f0)
    nsteps = 10
    u_ref, v_ref = tgs._oracle_linear(q, dt, nsteps, dtt)
    assert np.linalg.norm(u_ref) > 0
    kw = _vertex_kw(q, dtt)
    s = tgs._linear_solver(q, dtt, **kw)
    _check_kinds(s, kind)
    s.init()
    s.rk4(0.0, dt, nsteps)
    assert rel_l2(s.u.cpu().numpy(), u_ref) < TOL[tag]
    assert rel_l2(s.v.cpu().numpy(), v_ref) < TOL[tag]
    # graph replay and eager launches run the same kernels; only the order of the scatter atomics
    # (which differs from run to run in every geometry mode) separates them
    e = tgs._linear_solver(q, dtt, use_graph=False, **kw)
    e.init()
    e.rk4(0.0, dt, nsteps)
    close = 1e-13 if tag == "f64" else 1e-6
    assert rel_l2(e.u.cpu().numpy(), s.u.cpu().numpy()) < close
    assert rel_l2(e.v.cpu().numpy(), s.v.cpu().numpy()) < close

    u_ref, v_ref = tgl._oracle(q, dt, nsteps, dtt)
    lf = tgl._solver(LinearLeapfrog3D, q, dtt, **kw)
    _check_kinds(lf, kind)
    lf.init()
    lf.rk4(0.0, dt, nsteps)
    assert rel_l2(lf.u.cpu().numpy(), u_ref) < TOL[tag]
    assert rel_l2(lf.v.cpu().numpy(), v_ref) < TOL[tag]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,P,N,tag", MESHES)
def test_westervelt_vertex_vs_oracle(kind, P, N, tag):
    import problems
    from fenicsx_fus_gpu_b200.solver import WesterveltSpectral3D, westervelt_source
    from oracle import oracle as orc

    _gpu()
    dtt = np.float64 if tag == "f64" else np.float32
    L = 0.006
    q = _problem(kind, P, N, dtt, L, westervelt=True)
    dt = problems.cfl_dt(P, 0.7 * L / N, q.c0, q.f0, cfl=0.4)
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
    for mass_form in ("pointwise", "cells"):
        s = WesterveltSpectral3D(
            q.P, dtt, q.ndofs, q.dofmap, None, None, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
            q.cell_coeff3, q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1,
            q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2,
            source=lambda t: westervelt_source(t, q.f0, q.p0, q.c0), mass_form=mass_form, **_vertex_kw(q, dtt))
        _check_kinds(s, kind)
        assert rel_l2(s.m0.cpu().numpy(), m0) < (1e-13 if tag == "f64" else 1e-6)
        s.init()
        s.rk4(0.0, dt, nsteps)
        assert rel_l2(s.u.cpu().numpy(), u_ref) < TOL[tag], mass_form
        assert rel_l2(s.v.cpu().numpy(), v_ref) < TOL[tag], mass_form


@pytest.mark.gpu
@pytest.mark.parametrize("split_mode", ["none", "two", "fused"])
def test_linear_rk4_vertex_emulated_ranks_vs_serial_oracle(split_mode):
    """Blob partition, shared-last numbering, peer-memory halo, ranks emulated on one GPU: the
    halo-wait (WAIT) instantiations of the trilinear kernels in split modes "two" and "fused"."""
    import problems
    import test_gpu_solver as tgs
    from test_unstructured_partition import _renumbered
    from fenicsx_fus_gpu_b200 import utils
    from fenicsx_fus_gpu_b200.scatterer import LocalCluster, P2PHaloExchange, local_fabric
    from fenicsx_fus_gpu_b200.solver import LinearSpectral3D, linear_source

    _gpu()
    dtt = np.float64
    P, N, L, R, nsteps = 3, (4, 4, 4), (0.012, 0.01, 0.011), 4, 8
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0)
    u_ref, v_ref = tgs._oracle_linear(serial, dt, nsteps, dtt)
    parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                              shuffle_seed=2, owner_rule="hash")
    ren = _renumbered(parts, utils.compute_scatterer_data_all([p.index_map for p in parts]))
    ndmax = max(q.index_map.size_local + q.index_map.num_ghosts for q in parts)

    def body(r, transport):
        p = parts[r]
        dm, _, od, gd, _ = ren[r]
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        q = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=dm, ndofs=nl + ng)
        h = P2PHaloExchange(local_fabric(transport.cluster, r, P2PHaloExchange.arena_bytes(ndmax, dtt)), od, gd, nl, ng,
                            dtt)
        s = LinearSpectral3D(q.P, dtt, q.ndofs, q.dofmap, None, None, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
                             q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff2,
                             halo=h, source=lambda t: linear_source(t, q.f0, q.p0, q.c0), use_graph=False,
                             **_vertex_kw(q, dtt))
        s.split_mode = split_mode
        assert s.ntri == s.ncells and 0 < s.ninterface
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
    assert rel_l2(u, u_ref) < TOL["f64"]
    assert rel_l2(v, v_ref) < TOL["f64"]


@pytest.mark.gpu
def test_vertex_mode_holds_no_point_tables_and_saves_their_memory():
    from fenicsx_fus_gpu_b200 import problem

    _gpu()
    P, N, L = 4, 12, 0.012
    peak = {}
    for geometry in ("stream", "vertex"):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        su = problem.box_setup(P, N, L, np.float64, perturb=0.1, seed=2, geometry=geometry)
        s = problem.linear_solver(su, (2,), (3,), geometry=geometry)
        torch.cuda.synchronize()
        peak[geometry] = torch.cuda.max_memory_allocated() - base
        if geometry == "stream":
            table_bytes = su.dev["G"].nbytes + su.dev["detJ"].nbytes
        else:
            assert "G" not in su.dev and "detJ" not in su.dev and su.dev["Tc"].shape == (N**3, 36)
            assert s.G is None and s.detJ is None and s.ntri == s.ncells
        del su, s
    assert peak["stream"] - peak["vertex"] >= 0.9 * table_bytes, (peak, table_bytes)


@pytest.mark.gpu
@pytest.mark.parametrize("script,args", [("demo_linear_box.py", ["--cells", "6", "--steps", "2"]),
                                         ("demo_nonlinear_box.py", ["--cells", "4", "--steps", "2"])])
def test_demo_runs_with_vertex_geometry(script, args):
    _gpu()
    cmd = [sys.executable, os.path.join(ROOT, "demos", script), *args, "--geometry", "vertex"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "nan" not in r.stdout.lower()
