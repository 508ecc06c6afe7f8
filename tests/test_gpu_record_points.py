"""Point recorders: ``u`` at fixed points recorded at every step inside the captured step graphs
(``fus_record_points_*``, ``sampling.PointEvaluator.record``, ``solver.record_points`` and the
demos' ``PlaneSampler``).

A recorded row is the sum of ``fus_eval_points_*`` on the state at the start of a step, so the
references are ``PointEvaluator`` on one-step-at-a-time runs and the oracle's solution
interpolated at the points on the host."""

import glob
import os
import subprocess
import sys

import numpy as np
import pytest

from fenicsx_fus_gpu_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (nb if nb > 0 else 1.0))


def _torch():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# --------------------------------------------------------------------------- #
# CPU: argument rejection
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_record_points_rejects_bad_arguments_without_gpu(tag):
    lib = _lib.lib()
    f = getattr(lib, f"fus_record_points_{tag}")
    p = 256  # a non-null address: validation happens before any pointer is used
    ok = dict(u=p, dm=p, cells=p, phi=p, out=p, npts=7, P=4, step=None, base=p, first=0, rows=3)

    def call(**kw):
        a = {**ok, **kw}
        return f(a["u"], a["dm"], a["cells"], a["phi"], a["out"], a["npts"], a["P"], a["step"], a["base"],
                 a["first"], a["rows"], None)

    before = lib.fus_launch_count()
    assert call(npts=-1) == 100002
    assert call(rows=0) == 100002 and b"rows" in lib.fus_last_error()
    assert call(rows=-5) == 100002
    assert call(first=-1) == 100002 and b"first" in lib.fus_last_error()
    assert call(P=0) == 100001 and b"degree" in lib.fus_last_error()
    assert call(P=16) == 100001
    for name in ("u", "dm", "cells", "phi", "out", "base"):
        assert call(**{name: None}) == 100002, name
        assert b"null" in lib.fus_last_error()
    assert call(npts=0, u=None, dm=None, cells=None, phi=None, out=None, base=None) == 0  # nothing to launch
    assert lib.fus_launch_count() == before


# --------------------------------------------------------------------------- #
# GPU: the kernel
# --------------------------------------------------------------------------- #
def _box_evaluator(P, dt, npts=400, seed=0):
    torch = _torch()
    from fenicsx_fus_gpu_b200 import sampling as sp, substrate as S

    tb = S.element_tables(P, "basix", dt)
    mesh = S.create_box((3, 4, 3), (1.0, 1.1, 0.9), dtype=dt, perturb=0.12, seed=P)
    dm = S.tensor_dofmap(mesh, P)
    rng = np.random.default_rng(seed + P)
    pts = rng.uniform([0.0, 0.0, 0.0], [1.0, 1.1, 0.9], (npts, 3))
    xp, cells = sp.compute_eval_params(mesh, pts.T, dt)
    assert len(cells) > npts // 2
    return sp.PointEvaluator(P, dt, torch.from_numpy(dm).cuda(), mesh, xp, cells, tb.pts_1d), dm, cells


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("P", [2, 3, 4, 5, 6, 7])
def test_record_kernel_vs_float64_reference(P, tag):
    torch = _torch()
    from oracle import oracle as orc

    dt = np.float64 if tag == "f64" else np.float32
    ev, dm, cells = _box_evaluator(P, dt)
    n, rows, first = ev.npts, 5, 3
    rng = np.random.default_rng(P)
    u = torch.from_numpy(rng.standard_normal(int(dm.max()) + 1).astype(dt)).cuda()
    ref = orc.eval_points(u.cpu().numpy().astype(np.float64), dm, cells, ev.phi.cpu().numpy().astype(np.float64))
    sentinel = 12345.0
    buf = torch.full(((rows + 2) * n,), sentinel, dtype=ev.T, device="cuda")  # one guard row either side
    out = buf[n:(rows + 1) * n].view(rows, n)
    i64 = dict(dtype=torch.int64, device="cuda")
    step, base = torch.tensor([2], **i64), torch.tensor([4], **i64)
    ev.record(u, out, step, base, first, rows)  # row 4 + 2 - 3 = 3
    ev.record(u * 2, out, None, base, first, rows)  # without step_dev: row 4 - 3 = 1
    for b, s in ((first - 1, None), (first + rows, None), (first - 3, step), (first + rows - 2, step)):
        ev.record(u * 3, out, s, torch.tensor([b], **i64), first, rows)  # row -1 or rows: no write
    got = buf.cpu().numpy().reshape(rows + 2, n)
    tol = 1e-13 if tag == "f64" else 1e-5
    assert np.linalg.norm(ref) > 0
    assert rel_l2(got[4], ref) <= tol
    assert got[4].tobytes() == ev(u).cpu().numpy().tobytes()
    assert got[2].tobytes() == ev(u * 2).cpu().numpy().tobytes()
    for r in (0, 1, 3, 5, 6):
        assert (got[r] == sentinel).all(), r


# --------------------------------------------------------------------------- #
# GPU: solvers
# --------------------------------------------------------------------------- #
def _points_evaluator(su, npts=60, seed=5):
    from fenicsx_fus_gpu_b200 import sampling as sp

    x_g = su.mesh.x_g.astype(np.float64)
    lo, hi = x_g.min(axis=0), x_g.max(axis=0)
    pts = np.random.default_rng(seed).uniform(lo + 0.02 * (hi - lo), hi - 0.02 * (hi - lo), (npts, 3))
    xp, cells = sp.compute_eval_params(su.mesh, pts.T, su.dtype)  # a point near a jittered face may fall outside
    assert len(cells) > npts * 0.9
    return sp.PointEvaluator(su.P, su.dtype, su.dev["dofmap"], su.mesh, xp, cells, su.tables.pts_1d)


def _make(kind, geometry, dtt, tile=None):
    """Two identical solvers of ``kind`` and an evaluator of points inside their box."""
    import test_gpu_phased_array as tpa

    out = []
    for _ in range(2):
        if kind in ("rk4", "leapfrog"):
            t = tpa._whole_face(0.006, (0, 1)) if tile else None
            su, s, dt = tpa._piston(3, 5, dtt, geometry, kind, t)
        else:
            t = tpa._whole_face(0.005, (1, 2)) if tile else None
            su, s, dt = tpa._bowl(3, 5, dtt, geometry, kind, t)
        out.append(s)
    return out[0], out[1], _points_evaluator(su), dt


def _stepwise(s, ev, dt, nsteps):
    """Rows of ``ev(u)`` after 0, 1, ..., nsteps steps of one-step calls."""
    s.init()
    rows = [ev(s.u).cpu().numpy().copy()]
    for k in range(nsteps):
        s.rk4(s.t if k else 0.0, dt, 1)
        rows.append(ev(s.u).cpu().numpy().copy())
    return np.array(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("geometry", ["stream", "auto", "vertex"])
@pytest.mark.parametrize("kind", ["rk4", "leapfrog", "pointwise", "cells"])
def test_recorded_rows_equal_stepwise_evaluation(kind, geometry, tag):
    _torch()
    dtt = np.float64 if tag == "f64" else np.float32
    tol = 1e-13 if tag == "f64" else 1e-6
    s, ref_solver, ev, dt = _make(kind, geometry, dtt)
    nsteps = 16
    ref = _stepwise(ref_solver, ev, dt, nsteps)
    rec = s.record_points(ev, first=0, rows=nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    got = rec.cpu().numpy()
    assert np.isfinite(got).all() and np.linalg.norm(ref) > 0
    assert rel_l2(got, ref) <= tol
    assert got[-1].tobytes() == ev(s.u).cpu().numpy().tobytes()  # the state after the last step


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["rk4", "leapfrog", "pointwise"])
def test_recorded_rows_with_a_phased_array_source(kind):
    _torch()
    s, ref_solver, ev, dt = _make(kind, "auto", np.float64, tile="one")
    assert s.num_elements == 1
    ref = _stepwise(ref_solver, ev, dt, 12)
    rec = s.record_points(ev, first=0, rows=13)
    s.init()
    s.rk4(0.0, dt, 12)
    assert np.linalg.norm(ref) > 0 and rel_l2(rec.cpu().numpy(), ref) <= 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_linear_rk4_rows_match_the_oracle(tag):
    _torch()
    import problems
    import test_gpu_solver as tgs
    from fenicsx_fus_gpu_b200 import sampling as sp
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32
    P, N, L, nsteps = 3, 5, 0.008, 12
    d = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=4)
    pts = np.random.default_rng(1).uniform(0.05 * L, 0.95 * L, (50, 3))
    xp, cells = sp.compute_eval_params(d.mesh, pts.T, dtt)
    ev = sp.PointEvaluator(P, dtt, d.dofmap, d.mesh, xp, cells, d.tb.pts_1d)
    dt = problems.cfl_dt(P, L / N, d.c0, d.f0)
    m = np.zeros(d.ndofs, dtt)
    orc.mass_operator(np.ones(d.ndofs, dtt), d.cell_coeff1, m, d.detJ, d.dofmap)
    prob = orc.LinearProblem(P, d.dofmap, d.G, d.tb.dphi_1D, d.cell_coeff2, m, d.bfacet_dofmap1, d.detJ_f1,
                             d.facet_coeff1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff2, d.f0, d.p0, d.c0)
    u, v = np.zeros(d.ndofs, dtt), np.zeros(d.ndofs, dtt)
    phi = ev.phi.cpu().numpy()
    ref, t = [orc.eval_points(u, d.dofmap, cells, phi)], 0.0
    for _ in range(nsteps):
        orc.linear_rk4(prob, u, v, t, dt, 1)
        t += dt
        ref.append(orc.eval_points(u, d.dofmap, cells, phi))
    s = tgs._linear_solver(d, dtt)
    rec = s.record_points(ev, 0, nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    assert np.linalg.norm(ref) > 0
    assert rel_l2(rec.cpu().numpy(), np.array(ref)) <= (1e-12 if tag == "f64" else 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["graph", "eager"])
def test_rows_bit_identical_to_the_evaluator(mode):
    """After each one-step call, ``ev(u)`` equals the row of that step bit for bit."""
    _torch()
    s, _, ev, dt = _make("rk4", "auto", np.float64)
    s.use_graph = mode == "graph"
    rec = s.record_points(ev, first=2, rows=20)
    s.init()
    for k in range(10):
        s.rk4(s.t if k else 0.0, dt, 1)
        if s.nstep >= 2:
            assert rec[s.nstep - 2].cpu().numpy().tobytes() == ev(s.u).cpu().numpy().tobytes(), s.nstep
    for _ in range(3):
        s.step_eager(dt)
        assert rec[s.nstep - 2].cpu().numpy().tobytes() == ev(s.u).cpu().numpy().tobytes(), s.nstep
    got = rec.cpu().numpy()
    assert np.isfinite(got[:12]).all() and np.isnan(got[12:]).all()


@pytest.mark.gpu
def test_runs_split_over_calls():
    """Calls of 1, 3, 1, 5 and 2 steps: a window straddling calls and reaching past the run; the
    capture warm-up of a one-step call leaks no row; re-attaching recaptures; detaching restores
    the launches of a solver that never had a recorder."""
    _torch()
    from fenicsx_fus_gpu_b200 import _lib as L

    s, ref_solver, ev, dt = _make("rk4", "stream", np.float64)
    ref = _stepwise(ref_solver, ev, dt, 12)
    rec = s.record_points(ev, first=3, rows=15)  # rows 0..9 reached by the 12 steps, 10..14 not
    s.init()
    for k, n in enumerate((1, 3, 1, 5, 2)):
        s.rk4(s.t if k else 0.0, dt, n)
        got = rec.cpu().numpy()
        done = s.nstep - 3 + 1  # rows filled so far
        assert np.isnan(got[max(done, 0):]).all(), s.nstep
        if done > 0:
            assert rel_l2(got[:done], ref[3:s.nstep + 1]) <= 1e-13, s.nstep
            assert got[done - 1].tobytes() == ev(s.u).cpu().numpy().tobytes()
    assert s.nstep == 12 and np.isnan(rec[10:].cpu().numpy()).all()

    # re-attach at step 12: the graphs are recaptured, and the warm-up steps (from the current state)
    # write none of the rows before the window's first reached step
    graphs = s._graph
    rec2 = s.record_points(ev, first=0, rows=20)
    s.rk4(s.t, dt, 1)
    assert s._graph is not graphs
    got = rec2.cpu().numpy()
    assert np.isnan(got[:12]).all() and np.isnan(got[14:]).all()
    assert np.isfinite(got[12:14]).all()
    assert got[13].tobytes() == ev(s.u).cpu().numpy().tobytes()

    # detach: the eager launches per step are those of a solver that never had a recorder
    lib = L.lib()

    def launches(solver, n):
        before = lib.fus_launch_count()
        solver.rk4(solver.t, dt, n)
        return lib.fus_launch_count() - before

    s.use_graph = ref_solver.use_graph = False
    plain = launches(ref_solver, 3)
    assert launches(s, 3) == plain + 3 + 1  # one record per step and one after the last (rows 13..16)
    s.record_points(None)
    assert launches(s, 3) == plain
    got = rec2.cpu().numpy()
    assert np.isfinite(got[12:17]).all() and np.isnan(got[17:]).all()


@pytest.mark.gpu
def test_bad_recorder_arguments_raise_before_any_launch():
    _torch()
    from fenicsx_fus_gpu_b200 import _lib as L

    s, _, ev, dt = _make("rk4", "stream", np.float64)
    ev32 = _points_evaluator(_make_su32())
    lib = L.lib()
    before = lib.fus_launch_count()
    for bad in (dict(evaluator=ev32), dict(evaluator=ev, first=-1), dict(evaluator=ev, rows=0)):
        with pytest.raises(ValueError):
            s.record_points(**bad)
    assert s._rec is None and lib.fus_launch_count() == before


def _make_su32():
    from fenicsx_fus_gpu_b200 import problem

    return problem.box_setup(3, 5, 0.006, np.float32, perturb=0.08, seed=1)


@pytest.mark.gpu
def test_evaluator_of_another_degree_is_rejected():
    _torch()
    from fenicsx_fus_gpu_b200 import problem

    s, _, _, _ = _make("rk4", "stream", np.float64)
    ev4 = _points_evaluator(problem.box_setup(4, 3, 0.006, np.float64, perturb=0.08, seed=1))
    with pytest.raises(ValueError):
        s.record_points(ev4)


# --------------------------------------------------------------------------- #
# GPU: emulated ranks
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
@pytest.mark.parametrize("halo", ["nccl-shaped", "p2p-none", "p2p-two", "p2p-fused"])
@pytest.mark.parametrize("partition", ["block", "blob"])
def test_emulated_ranks_vs_single_rank(partition, halo):
    """Every rank records the points of its own cells; the rows equal the single-rank recorder's
    rows for the same points.  The run is split into two calls, and the window straddles them."""
    torch = _torch()
    import problems
    import test_gpu_phased_array as tpa
    from test_unstructured_partition import _renumbered
    from fenicsx_fus_gpu_b200 import sampling as sp, substrate as S, utils
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, LocalCluster, P2PHaloExchange, local_fabric
    from fenicsx_fus_gpu_b200.solver import linear_source

    dtt = np.float64
    P, N, L, R = 3, (4, 4, 4), (0.012, 0.01, 0.011), 4
    first, rows, calls = 2, 9, (4, 6)
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0)
    src = lambda t: linear_source(t, serial.f0, serial.p0, serial.c0)  # noqa: E731
    pts = np.random.default_rng(8).uniform(0.02, 0.98, (120, 3)) * np.array(L)

    def run(s, ev):
        rec = s.record_points(ev, first, rows)
        s.init()
        for k, n in enumerate(calls):
            s.rk4(s.t if k else 0.0, dt, n)
        torch.cuda.synchronize()
        return rec.cpu().numpy()

    xs, cs = sp.compute_eval_params(serial.mesh, pts.T, dtt)
    assert len(cs) == len(pts)
    ref = run(tpa._linear(serial, dtt, source=src),
              sp.PointEvaluator(P, dtt, serial.dofmap, serial.mesh, xs, cs, serial.tb.pts_1d))
    assert np.isfinite(ref).all() and np.linalg.norm(ref) > 0
    if partition == "blob":
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                                  shuffle_seed=2, owner_rule="hash")
    else:
        parts = S.partition_box(N, P, R, lengths=L, dtype=dtt, perturb=0.1, seed=11)
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    ren = _renumbered(parts, sdata)
    ndmax = max(p.index_map.size_local + p.index_map.num_ghosts for p in parts)
    where = {tuple(x): i for i, x in enumerate(xs)}

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
        q = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=dm, ndofs=nl + ng)
        s = tpa._linear(q, dtt, halo=h, source=src, use_graph=False)
        if halo != "nccl-shaped":
            s.split_mode = halo.split("-")[1]
        xp, cells = sp.compute_eval_params(p.mesh, pts.T, dtt)
        ev = sp.PointEvaluator(P, dtt, dm, p.mesh, xp, cells, q.tb.pts_1d)
        return [where[tuple(x)] for x in xp], run(s, ev)

    out = LocalCluster(R).run(body)
    seen = set()
    for idx, got in out:
        seen.update(idx)
        if idx:
            assert np.isfinite(got).all()
            assert rel_l2(got, ref[:, idx]) <= 1e-12
    assert len(seen) == len(pts) and sum(1 for idx, _ in out if idx) > 1


# --------------------------------------------------------------------------- #
# GPU: demos
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
def test_piston_demo_writes_the_recorded_window(tmp_path):
    """A window that lies inside the run: one file per recorded step, rows ``x, z, p``, finite."""
    _torch()
    from fenicsx_fus_gpu_b200 import problem

    P, cells, f0, c0 = 3, 5, 0.5e6, 1500.0
    h = 0.12 / 93
    dt = problem.cfl_time_step(P, h, c0, f0, 0.65)
    t_from = cells * h / c0 + 6.0 / f0
    period_steps = int(round(1.0 / f0 / dt))
    nsteps = int(t_from / dt) + period_steps + 10
    cmd = [sys.executable, os.path.join(ROOT, "demos", "demo_linear_piston.py"), "--cells", str(cells), "--degree",
           str(P), "--steps", str(nsteps), "--sample-dir", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "nan" not in r.stdout.lower()
    files = sorted(glob.glob(os.path.join(str(tmp_path), "pressure_field_*_rank0.txt")))
    assert len(files) == period_steps + 2
    last = None
    for k in range(period_steps + 2):
        d = np.loadtxt(os.path.join(str(tmp_path), f"pressure_field_{k}_rank0.txt"), delimiter=",")
        assert d.ndim == 2 and d.shape[1] == 3 and d.shape[0] > 100 and np.isfinite(d).all()
        if last is not None:
            assert np.array_equal(d[:, :2], last[:, :2])
        last = d
    assert np.abs(last[:, 2]).max() > 0
