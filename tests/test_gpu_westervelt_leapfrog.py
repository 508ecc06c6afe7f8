"""The Westervelt leapfrog integrator (``WesterveltLeapfrog3D``; the reference has RK4 only, so there is
no reference twin): the CUDA steps against the numpy restatement of the scheme
(``westervelt_leapfrog_oracle``; rel-L2 <= 1e-12 in float64, <= 1e-5 in float32) in every geometry
mode, with graph replay and eager launches and with a run split over two calls; the convergence order
against the RK4 solver; a phased-array source; recorded rows; emulated ranks under both halos and
partitions; the launches of a captured step; and the partitioned solve on real GPUs."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"f64": 1e-12, "f32": 1e-5}


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _m0(q, dtt):
    from oracle import oracle as orc

    ones = np.ones(q.ndofs, dtt)
    m0 = np.zeros(q.ndofs, dtt)
    orc.mass_operator(ones, q.cell_coeff1, m0, q.detJ, q.dofmap)
    orc.mass_operator(ones, q.facet_coeff1_2, m0, q.detJ_f2, q.bfacet_dofmap2)
    return m0


def _prob(q, dtt):
    from oracle import oracle as orc

    return orc.WesterveltProblem(q.P, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff2, q.cell_coeff3,
                                 q.cell_coeff4, q.cell_coeff5, _m0(q, dtt), q.bfacet_dofmap1, q.detJ_f1,
                                 q.facet_coeff1_1, q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff2_2,
                                 q.f0, q.p0, q.c0)


def _oracle(q, dt, nsteps, dtt, source=None):
    import westervelt_leapfrog_oracle as wlo

    u, v = np.zeros(q.ndofs, dtt), np.zeros(q.ndofs, dtt)
    wlo.westervelt_leapfrog(_prob(q, dtt), u, v, 0.0, dt, nsteps, source)
    return u, v


def _solver(q, dtt, cls=None, geo=True, **kw):
    """The solver of ``q`` (``geo=False``: no G / detJ, for geometry="vertex")."""
    from fenicsx_fus_gpu_b200.solver import WesterveltLeapfrog3D, westervelt_source

    kw.setdefault("source", lambda t: westervelt_source(t, q.f0, q.p0, q.c0))
    return (cls or WesterveltLeapfrog3D)(
        q.P, dtt, q.ndofs, q.dofmap, q.G if geo else None, q.detJ if geo else None, q.tb.dphi_1D, q.cell_coeff1,
        q.cell_coeff2, q.cell_coeff3, q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1,
        q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2, **kw)


def _split_run(s, dt, nsteps):
    s.init()
    t = s.rk4(0.0, dt, nsteps // 2)
    t = s.steps(t, dt, nsteps - nsteps // 2)  # a second call continues (no second kick-off)
    assert abs(t - nsteps * dt) < 1e-15
    return s.u.cpu().numpy(), s.v.cpu().numpy()


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("P,N", [(3, 5), (4, 4), (6, 3)])
def test_leapfrog_vs_oracle(P, N, tag):
    import problems

    dtt = np.float64 if tag == "f64" else np.float32
    L, nsteps = 0.006, 24
    q = problems.westervelt_problem(P, N, L, dtt, perturb=0.12, seed=P)
    dt = problems.cfl_dt(P, L / N, q.c0, q.f0, cfl=0.4)
    u_ref, v_ref = _oracle(q, dt, nsteps, dtt)
    assert np.linalg.norm(u_ref) > 0
    for use_graph in (True, False):
        s = _solver(q, dtt, use_graph=use_graph)
        assert s.integrator == "leapfrog" and s._absb is None  # the absorbing term is the close's
        u, v = _split_run(s, dt, nsteps)
        assert rel_l2(u, u_ref) < TOL[tag], use_graph
        assert rel_l2(v, v_ref) < TOL[tag], use_graph


@pytest.mark.parametrize("geometry", ["auto", "vertex"])
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_geometry_modes_vs_oracle(geometry, tag):
    """A box that mixes rectilinear, affine and trilinear cells."""
    import problems
    import test_gpu_vertex_solver as tvs

    dtt = np.float64 if tag == "f64" else np.float32
    P, N, L, nsteps = 4, 6, 0.006, 12
    q = tvs._problem("mixed", P, N, dtt, L, westervelt=True)
    dt = problems.cfl_dt(P, 0.7 * L / N, q.c0, q.f0, cfl=0.4)
    u_ref, v_ref = _oracle(q, dt, nsteps, dtt)
    assert np.linalg.norm(u_ref) > 0
    if geometry == "vertex":
        s = _solver(q, dtt, geo=False, **tvs._vertex_kw(q, dtt))
    else:
        s = _solver(q, dtt, geometry="auto", weights=q.tb.wts)
    assert s.nrect > 0 and s.naff > s.nrect and s.naff < s.ncells
    u, v = _split_run(s, dt, nsteps)
    assert rel_l2(u, u_ref) < TOL[tag]
    assert rel_l2(v, v_ref) < TOL[tag]


def test_second_order_against_rk4():
    """Same problem, same final time: the leapfrog solution converges to the RK4 one (at dt/4) with dt^2."""
    import problems
    from fenicsx_fus_gpu_b200.solver import WesterveltSpectral3D

    P, N, L, dtt = 3, 5, 0.006, np.float64
    q = problems.westervelt_problem(P, N, L, dtt, perturb=0.1, seed=2, p0=3.0e6)
    dt0 = problems.cfl_dt(P, L / N, q.c0, q.f0, cfl=0.1)
    ref = _solver(q, dtt, WesterveltSpectral3D)
    ref.init()
    ref.rk4(0.0, dt0 / 4, 4 * 64)
    u_ref = ref.u.cpu().numpy()
    assert np.linalg.norm(u_ref) > 0
    errs = []
    for k in (1, 2, 4):
        s = _solver(q, dtt)
        s.init()
        s.rk4(0.0, dt0 / k, 64 * k)
        assert abs(s.t - 64 * dt0) < 1e-14
        errs.append(rel_l2(s.u.cpu().numpy(), u_ref))
    assert errs[2] < 0.02, errs
    assert 3.5 < errs[0] / errs[1] < 4.6 and 3.5 < errs[1] / errs[2] < 4.6, errs


def test_phased_array_vs_element_resolved_oracle():
    import test_gpu_phased_array as tpa
    from oracle import oracle as orc

    dtt = np.float64
    q, ids, E, src, dt = tpa._array_problem(dtt, westervelt=True)
    sel = tpa._split(q, ids, E)

    def source(t, b):
        g, dg = src(t)
        tpa._elem_mass(orc, sel, g, q.facet_coeff1_1, q.detJ_f1, q.bfacet_dofmap1, b, b.dtype)
        tpa._elem_mass(orc, sel, dg, q.facet_coeff2_1, q.detJ_f1, q.bfacet_dofmap1, b, b.dtype)

    nsteps = 20
    u_ref, v_ref = _oracle(q, dt, nsteps, dtt, source)
    assert np.linalg.norm(u_ref) > 0
    for use_graph in (True, False):
        s = _solver(q, dtt, source=src, source_elements=ids, num_elements=E, use_graph=use_graph)
        s.init()
        s.rk4(0.0, dt, nsteps)
        assert rel_l2(s.u.cpu().numpy(), u_ref) <= 1e-12, use_graph
        assert rel_l2(s.v.cpu().numpy(), v_ref) <= 1e-12, use_graph


@pytest.mark.parametrize("geometry", ["stream", "auto", "vertex"])
def test_recorded_rows_equal_the_evaluator(geometry):
    """Points and array elements recorded inside the captured steps equal the evaluators applied to
    ``u`` after every one-step call."""
    import test_gpu_phased_array as tpa
    import test_gpu_record_points as trp
    from fenicsx_fus_gpu_b200 import problem

    dtt = np.float64
    runs = []
    for _ in range(2):
        su, s, dt = tpa._bowl(3, 5, dtt, geometry, "pointwise", integrator="leapfrog")
        runs.append(s)
    s, ref = runs
    ev = trp._points_evaluator(su)
    rx = problem.element_receiver(su, [2], problem.TileArray((0.0, 0.0025, 0.0025), 2, 2, 0.0025, axes=(1, 2)))
    nsteps = 12
    ref.init()
    rows_p, rows_e = [ev(ref.u).cpu().numpy()], [rx(ref.u).cpu().numpy()]
    for k in range(nsteps):
        ref.rk4(ref.t if k else 0.0, dt, 1)
        rows_p.append(ev(ref.u).cpu().numpy())
        rows_e.append(rx(ref.u).cpu().numpy())
    rec_p = s.record_points(ev, first=0, rows=nsteps + 1)
    rec_e = s.record_elements(rx, first=0, rows=nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    got_p, got_e = rec_p.cpu().numpy(), rec_e.cpu().numpy()
    assert np.isfinite(got_p).all() and np.isfinite(got_e).all() and np.linalg.norm(rows_p) > 0
    assert rel_l2(got_p, np.array(rows_p)) <= 1e-13
    assert rel_l2(got_e, np.array(rows_e)) <= 1e-13
    assert got_p[-1].tobytes() == ev(s.u).cpu().numpy().tobytes()
    assert got_e[-1].tobytes() == rx(s.u).cpu().numpy().tobytes()


def test_cells_mass_form_raises():
    import problems

    q = problems.westervelt_problem(3, 3, 0.006, np.float64)
    with pytest.raises(ValueError, match="pointwise"):
        _solver(q, np.float64, mass_form="cells")
    from fenicsx_fus_gpu_b200 import problem

    su = problem.box_setup(3, 3, 0.006, np.float64)
    with pytest.raises(ValueError, match="pointwise"):
        problem.westervelt_solver(su, [2], [3], integrator="leapfrog", mass_form="cells")
    with pytest.raises(ValueError, match="integrator"):
        problem.westervelt_solver(su, [2], [3], integrator="euler")


@pytest.mark.parametrize("halo", ["nccl-shaped", "p2p"])
@pytest.mark.parametrize("partition", ["block", "blob"])
def test_emulated_ranks_vs_serial_oracle(partition, halo):
    import problems
    from test_unstructured_partition import _renumbered
    from fenicsx_fus_gpu_b200 import substrate as S
    from fenicsx_fus_gpu_b200 import utils
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, LocalCluster, P2PHaloExchange, local_fabric

    dtt, P, N, L, R, nsteps = np.float64, 3, (4, 4, 3), (0.006, 0.005, 0.0055), 4, 16
    serial = problems.westervelt_problem(P, N, L, dtt, perturb=0.1, seed=11)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0, cfl=0.3)
    u_ref, v_ref = _oracle(serial, dt, nsteps, dtt)
    if partition == "blob":
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                                  shuffle_seed=2, owner_rule="hash")
    else:
        parts = S.partition_box(N, P, R, lengths=L, dtype=dtt, perturb=0.1, seed=11)
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    ren = _renumbered(parts, sdata)
    ndmax = max(p.index_map.size_local + p.index_map.num_ghosts for p in parts)

    def body(r, transport):
        p = parts[r]
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        if halo == "nccl-shaped":
            dm, od, gd = p.dofmap, *sdata[r]
            h = HaloExchange(transport, od, gd, nl, dtt)
        else:
            dm, _, od, gd, _ = ren[r]
            h = P2PHaloExchange(local_fabric(transport.cluster, r, P2PHaloExchange.arena_bytes(ndmax, dtt)), od, gd,
                                nl, ng, dtt)
        q = problems.westervelt_problem(P, None, None, dtt, mesh=p.mesh, dofmap=dm, ndofs=nl + ng)
        s = _solver(q, dtt, halo=h, use_graph=False)
        s.init()
        s.rk4(0.0, dt, nsteps // 2)
        s.rk4(s.t, dt, nsteps - nsteps // 2)
        torch.cuda.synchronize()
        return s.u.cpu().numpy(), s.v.cpu().numpy()

    out = LocalCluster(R).run(body)
    u, v = np.full_like(u_ref, np.nan), np.full_like(v_ref, np.nan)
    for r, p in enumerate(parts):
        nl = p.index_map.size_local
        l2s = p.local_to_serial if halo == "nccl-shaped" else ren[r][1]
        u[l2s[:nl]] = out[r][0][:nl]
        v[l2s[:nl]] = out[r][1][:nl]
    assert np.linalg.norm(u_ref) > 0
    assert rel_l2(u, u_ref) <= 1e-12
    assert rel_l2(v, v_ref) <= 1e-12


@pytest.mark.parametrize("record", [False, True])
def test_captured_step_launches(record):
    """A step is the cell-kernel launches (one per geometry kind), the boundary launch (sources only) and
    the close, plus the record launch when a recorder is attached: counted over the capture (two
    warm-up steps, two captured ones) and over an eager step."""
    import problems
    import test_gpu_vertex_solver as tvs
    from fenicsx_fus_gpu_b200 import _lib as L
    from fenicsx_fus_gpu_b200 import sampling as sp

    lib = L.lib()
    P, N, L_ = 3, 6, 0.006
    q = tvs._problem("mixed", P, N, np.float64, L_, westervelt=True)
    dt = problems.cfl_dt(P, 0.7 * L_ / N, q.c0, q.f0, cfl=0.4)
    s = _solver(q, np.float64, geometry="auto", weights=q.tb.wts)
    assert len(s._segs) == 3 and s._absb is None and s._bdofs.numel() > 0
    if record:
        pts = np.random.default_rng(1).uniform(0.1 * L_, 0.9 * L_, (40, 3))
        xp, cells = sp.compute_eval_params(q.mesh, pts.T, np.float64)
        s.record_points(sp.PointEvaluator(P, np.float64, q.dofmap, q.mesh, xp, cells, q.tb.pts_1d), first=0, rows=8)
    per_step = len(s._segs) + 2 + int(record)
    s.init()
    s.rk4(0.0, dt, 2)
    before = lib.fus_launch_count()
    s._capture(dt)
    assert s._graph is not None and lib.fus_launch_count() - before == 4 * per_step
    u = s.u.clone()
    s._replay_step(dt)  # the replay makes no host launch
    assert lib.fus_launch_count() - before == 4 * per_step and not torch.equal(u, s.u)
    s.use_graph = False
    before = lib.fus_launch_count()
    s.rk4(s.t, dt, 1)
    assert lib.fus_launch_count() - before == per_step + int(record)  # + the record after the call


def test_partitioned_solve_on_real_gpus_matches_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    out = tmp_path / "wl.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29613",
           os.path.join(ROOT, "tests", "mgpu_westervelt_leapfrog_worker.py"), "--out", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.load(open(out))
    assert res["ok"] and len(res["parity"]) == 5, res
