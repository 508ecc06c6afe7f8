"""Element receivers: what each element of a transducer array receives, ``r_e = int_{Gamma_e} u dS``,
evaluated and recorded at every step inside the captured step graphs (``fus_eval_elements_*``,
``fus_record_elements_*``, ``sampling.ElementReceiver``, ``problem.element_receiver`` and
``solver.record_elements``).

The references are float64 sums on the host over the same facet rows (``detJ_f`` weights), the oracle's
linear RK4 states reduced that way, one-step-at-a-time runs, and reciprocity between two elements."""

import os
import subprocess
import sys

import numpy as np
import pytest

from fenicsx_fus_gpu_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARGUMENT = 100002


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
def test_element_entries_reject_bad_arguments_without_gpu(tag):
    lib = _lib.lib()
    p = 256  # a non-null address: validation happens before any pointer is used
    ok = dict(u=p, dof=p, w=p, cb=p, ec=p, part=p, out=p, nchunks=5, E=3, step=None, base=p, first=0, rows=3)
    ev, rec = getattr(lib, f"fus_eval_elements_{tag}"), getattr(lib, f"fus_record_elements_{tag}")

    def head(a):
        return a["u"], a["dof"], a["w"], a["cb"], a["ec"], a["part"], a["out"], a["nchunks"], a["E"]

    def call_rec(**kw):
        a = {**ok, **kw}
        return rec(*head(a), a["step"], a["base"], a["first"], a["rows"], None)

    def call_ev(**kw):
        return ev(*head({**ok, **kw}), None)

    before = lib.fus_launch_count()
    for call in (call_ev, call_rec):
        assert call(nchunks=-1) == BAD_ARGUMENT and b"nchunks" in lib.fus_last_error()
        assert call(E=-1) == BAD_ARGUMENT and b"E < 0" in lib.fus_last_error()
        for name in ("u", "dof", "w", "cb", "ec", "part", "out"):
            assert call(**{name: None}) == BAD_ARGUMENT, name
            assert b"null" in lib.fus_last_error()
        nulls = dict(u=None, dof=None, w=None, cb=None, ec=None, part=None, out=None, base=None)
        assert call(E=0, **nulls) == 0  # nothing to launch
        assert call(nchunks=0, **nulls) == 0  # no entries on this rank
    assert call_rec(rows=0) == BAD_ARGUMENT and b"rows" in lib.fus_last_error()
    assert call_rec(rows=-4) == BAD_ARGUMENT
    assert call_rec(first=-1) == BAD_ARGUMENT and b"first" in lib.fus_last_error()
    assert call_rec(base=None) == BAD_ARGUMENT and b"null" in lib.fus_last_error()
    assert b"record_elements" in lib.fus_last_error()
    assert lib.fus_launch_count() == before


# --------------------------------------------------------------------------- #
# GPU: the kernels
# --------------------------------------------------------------------------- #
def _random_rows(rng, E, nd, big=None):
    """Element-major (dof, w) rows, dofs distinct and sorted inside a row; every third element empty,
    element ``big`` (if any) with more than 100 k entries."""
    dof, w, elem = [], [], []
    for e in range(E):
        n = 0 if e % 3 == 2 else int(rng.integers(1, 700))
        if e == big:
            n = 150_000
        d = np.sort(rng.choice(nd, n, replace=False))
        dof.append(d)
        w.append(rng.uniform(0.1, 2.0, n))
        elem.append(np.full(n, e))
    return np.concatenate(dof), np.concatenate(w), np.concatenate(elem)


def _chunk_tables(elem, E, chunk):
    """Chunk table of element-major rows, built independently of ElementReceiver."""
    cnt = np.bincount(elem, minlength=E)
    start = np.concatenate([[0], np.cumsum(cnt)])
    beg, ech = [], [0]
    for e in range(E):
        beg += list(range(start[e], start[e + 1], chunk))
        ech.append(len(beg))
    return np.array(beg + [start[-1]], np.int32), np.array(ech, np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("E", [1, 7, 64, 1024])
def test_kernel_vs_float64_reference(E, tag):
    torch = _torch()
    from fenicsx_fus_gpu_b200 import sampling as sp

    dt = np.float64 if tag == "f64" else np.float32
    rng = np.random.default_rng(E)
    nd = 400_000
    dof, w, elem = _random_rows(rng, E, nd, big=0 if E in (1, 7) else None)
    w = w.astype(dt)
    # one facet row per entry: the receiver's rows are then exactly these entries
    r = sp.ElementReceiver(dt, dof.astype(np.int32)[:, None], w[:, None], elem, E)
    cb, ec = _chunk_tables(elem, E, sp.CHUNK)
    assert np.array_equal(r.dof.cpu().numpy(), dof) and r.w.cpu().numpy().tobytes() == w.tobytes()
    assert np.array_equal(r.chunk_beg.cpu().numpy(), cb) and np.array_equal(r.elem_chunk.cpu().numpy(), ec)
    u = torch.from_numpy(rng.standard_normal(nd).astype(dt)).cuda()
    ref = np.bincount(elem, weights=w.astype(np.float64) * u.cpu().numpy().astype(np.float64)[dof], minlength=E)
    got = r(u).cpu().numpy()
    assert np.linalg.norm(ref) > 0 and rel_l2(got, ref) <= (1e-13 if tag == "f64" else 1e-5)
    assert np.all(got[2::3] == 0.0)  # empty elements
    assert r(u).cpu().numpy().tobytes() == got.tobytes()  # two runs, the same bits

    rows, first, sentinel = 5, 3, 12345.0
    buf = torch.full(((rows + 2) * E,), sentinel, dtype=r.T, device="cuda")  # one guard row either side
    out = buf[E:(rows + 1) * E].view(rows, E)
    i64 = dict(dtype=torch.int64, device="cuda")
    step, base = torch.tensor([2], **i64), torch.tensor([4], **i64)
    r.record(u, out, step, base, first, rows)  # row 4 + 2 - 3 = 3
    r.record(u * 2, out, None, base, first, rows)  # without step_dev: row 4 - 3 = 1
    for b, s in ((first - 1, None), (first + rows, None), (first - 3, step), (first + rows - 2, step)):
        r.record(u * 3, out, s, torch.tensor([b], **i64), first, rows)  # row -1 or rows: no write
    g = buf.cpu().numpy().reshape(rows + 2, E)
    assert g[4].tobytes() == got.tobytes()
    assert g[2].tobytes() == r(u * 2).cpu().numpy().tobytes()
    for k in (0, 1, 3, 5, 6):
        assert (g[k] == sentinel).all(), k


# --------------------------------------------------------------------------- #
# GPU: rows and areas
# --------------------------------------------------------------------------- #
def _host_rows(bdm, dJ, ids, E):
    """(element, dof) -> sum of detJ_f in float64, in facet order, as sorted arrays."""
    acc = {}
    for f in range(bdm.shape[0]):
        for q in range(bdm.shape[1]):
            k = (int(ids[f]), int(bdm[f, q]))
            acc[k] = acc.get(k, 0.0) + float(dJ[f, q])
    keys = sorted(acc)
    return np.array([k[0] for k in keys]), np.array([k[1] for k in keys]), np.array([acc[k] for k in keys])


@pytest.mark.gpu
@pytest.mark.parametrize("perturb", [0.0, 0.1])
def test_rows_and_areas_of_a_tile_array(perturb):
    _torch()
    from fenicsx_fus_gpu_b200 import problem

    P, N, L = 3, 6, 0.006
    su = problem.box_setup(P, N, L, np.float64, perturb=perturb, seed=3)
    pitch = L / N
    tile = problem.TileArray((0.5 * L, 0.5 * L, 0.0), 4, 4, pitch)  # one facet per element
    r = problem.element_receiver(su, [0], tile)
    fd, dJ, bd = problem.facet_group(su, [0], lambda cen: tile.element_of(cen) >= 0)
    ids = tile.element_of(problem.facet_centroids(su.mesh, bd))
    assert r.E == 16 and np.array_equal(np.sort(np.unique(ids)), np.arange(16))
    e_h, d_h, w_h = _host_rows(fd.cpu().numpy(), dJ.cpu().numpy(), ids, 16)
    count = np.bincount(e_h, minlength=16)
    assert np.array_equal(r.dof.cpu().numpy(), d_h)
    assert rel_l2(r.w.cpu().numpy(), w_h) <= 1e-15
    assert np.array_equal(np.diff(r.elem_chunk.cpu().numpy()), (count + 255) // 256)
    areas = r.areas.cpu().numpy()
    host = np.bincount(ids, weights=dJ.cpu().numpy().sum(axis=1), minlength=16)
    assert rel_l2(areas, host) <= 1e-13
    if perturb == 0.0:
        assert np.abs(areas / pitch**2 - 1.0).max() <= 1e-13
    # an id list with one index per facet row gives the same receiver
    r2 = problem.element_receiver(su, [0], ids, predicate=lambda cen: tile.element_of(cen) >= 0, num_elements=16)
    assert r2.areas.cpu().numpy().tobytes() == areas.tobytes()


@pytest.mark.gpu
def test_source_rows_bit_identical_to_the_inline_reduction():
    """The phased-array source's CSR rows through ``sampling.reduce_by_key`` equal those of the
    reduction the solver carried inline before, bit for bit."""
    torch = _torch()
    import test_gpu_phased_array as tpa

    for west in (False, True):
        q, ids, E, src, dt = tpa._array_problem(np.float64, west)
        if west:
            from fenicsx_fus_gpu_b200.solver import WesterveltSpectral3D

            s = WesterveltSpectral3D(
                q.P, np.float64, q.ndofs, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
                q.cell_coeff3, q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1,
                q.facet_coeff2_1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2, source=src,
                source_elements=ids, num_elements=E)
            coeffs = (q.facet_coeff1_1, q.facet_coeff2_1)
        else:
            s = tpa._linear(q, np.float64, source=src, source_elements=ids)
            coeffs = (q.facet_coeff1,)
        dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
        bdm, dJ = dv(q.bfacet_dofmap1), dv(q.detJ_f1)
        i64 = dict(dtype=torch.int64, device="cuda")
        key = bdm.reshape(-1).to(torch.int64) * E + dv(ids).repeat_interleave(bdm.shape[1])
        key, order = torch.sort(key, stable=True)
        vals = [(dv(c)[:, None] * dJ).reshape(-1)[order] for c in coeffs]
        ukey, inv, counts = torch.unique_consecutive(key, return_inverse=True, return_counts=True)
        pos = torch.arange(key.numel(), **i64) - (torch.cumsum(counts, 0) - counts)[inv]
        sums = [torch.zeros(ukey.numel(), dtype=torch.float64, device="cuda") for _ in vals]
        for j in range(int(counts.max().item())):
            sel = pos == j
            for acc, v in zip(sums, vals):
                acc.index_add_(0, inv[sel], v[sel])
        assert s._eelem.cpu().numpy().tobytes() == (ukey % E).to(torch.int32).cpu().numpy().tobytes()
        assert s._ew.cpu().numpy().tobytes() == sums[0].cpu().numpy().tobytes()
        if west:
            assert s._ew2.cpu().numpy().tobytes() == sums[1].cpu().numpy().tobytes()


@pytest.mark.gpu
def test_bad_receiver_input_raises_before_any_kernel():
    _torch()
    from fenicsx_fus_gpu_b200 import problem, sampling as sp

    lib = _lib.lib()
    su = problem.box_setup(3, 4, 0.006, np.float64, perturb=0.05, seed=1)
    fd, dJ, _ = problem.facet_group(su, [0])
    nf = fd.shape[0]
    ids = np.arange(nf) % 3
    before = lib.fus_launch_count()
    for bad in (dict(elements=ids, num_elements=2), dict(elements=ids - 1, num_elements=3),
                dict(elements=ids[:-1], num_elements=3), dict(elements=ids, num_elements=0)):
        with pytest.raises(ValueError):
            sp.ElementReceiver(np.float64, fd, dJ, **bad)
    with pytest.raises(ValueError):
        sp.ElementReceiver(np.float64, fd, dJ[:, :-1], ids, 3)
    assert lib.fus_launch_count() == before
    r = sp.ElementReceiver(np.float64, fd, dJ, ids, 3)
    s = problem.linear_solver(su, [0], [1, 2, 3, 4, 5])
    s32 = problem.linear_solver(problem.box_setup(3, 4, 0.006, np.float32, perturb=0.05, seed=1), [0], [1])
    for solver, kw in ((s32, dict(receiver=r)), (s, dict(receiver=r, first=-1)), (s, dict(receiver=r, rows=0))):
        with pytest.raises(ValueError):
            solver.record_elements(**kw)
    assert not s._recs and not s32._recs


# --------------------------------------------------------------------------- #
# GPU: solvers
# --------------------------------------------------------------------------- #
def _make(kind, geometry, dtt):
    """Two identical solvers of ``kind`` and a 3 x 3 receiver on their source face."""
    import test_gpu_phased_array as tpa
    from fenicsx_fus_gpu_b200 import problem

    out = []
    for _ in range(2):
        if kind in ("rk4", "leapfrog"):
            su, s, dt = tpa._piston(3, 5, dtt, geometry, kind)
            tile, face = problem.TileArray((0.003, 0.003, 0.0), 3, 3, 0.0015), 0
        else:
            su, s, dt = tpa._bowl(3, 5, dtt, geometry, kind)
            tile, face = problem.TileArray((0.0, 0.0025, 0.0025), 3, 3, 0.0012, axes=(1, 2)), 2
        out.append(s)
    return out[0], out[1], problem.element_receiver(su, [face], tile), dt


def _stepwise(s, r, dt, nsteps):
    """Rows of ``r(u)`` after 0, 1, ..., nsteps steps of one-step calls."""
    s.init()
    rows = [r(s.u).cpu().numpy().copy()]
    for k in range(nsteps):
        s.rk4(s.t if k else 0.0, dt, 1)
        rows.append(r(s.u).cpu().numpy().copy())
    return np.array(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("geometry", ["stream", "auto", "vertex"])
@pytest.mark.parametrize("kind", ["rk4", "leapfrog", "pointwise", "cells"])
def test_recorded_rows_equal_stepwise_evaluation(kind, geometry, tag):
    _torch()
    dtt = np.float64 if tag == "f64" else np.float32
    tol = 1e-13 if tag == "f64" else 1e-6
    s, ref_solver, r, dt = _make(kind, geometry, dtt)
    nsteps = 16
    ref = _stepwise(ref_solver, r, dt, nsteps)
    rec = s.record_elements(r, first=0, rows=nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    got = rec.cpu().numpy()
    assert got.shape == (nsteps + 1, 9) and np.isfinite(got).all() and np.linalg.norm(ref) > 0
    assert rel_l2(got, ref) <= tol
    assert got[-1].tobytes() == r(s.u).cpu().numpy().tobytes()  # the state after the last step


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_linear_rk4_rows_match_the_oracle(tag):
    _torch()
    import problems
    import test_gpu_solver as tgs
    from fenicsx_fus_gpu_b200 import sampling as sp
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32
    P, N, L, nsteps, E = 3, 5, 0.008, 12, 3
    d = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=4)
    bdm, dJ = np.asarray(d.bfacet_dofmap1), np.asarray(d.detJ_f1)
    ids = np.arange(bdm.shape[0]) % E
    r = sp.ElementReceiver(dtt, bdm, dJ, ids, E)
    dt = problems.cfl_dt(P, L / N, d.c0, d.f0)
    m = np.zeros(d.ndofs, dtt)
    orc.mass_operator(np.ones(d.ndofs, dtt), d.cell_coeff1, m, d.detJ, d.dofmap)
    prob = orc.LinearProblem(P, d.dofmap, d.G, d.tb.dphi_1D, d.cell_coeff2, m, d.bfacet_dofmap1, d.detJ_f1,
                             d.facet_coeff1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff2, d.f0, d.p0, d.c0)
    u, v = np.zeros(d.ndofs, dtt), np.zeros(d.ndofs, dtt)

    def reduce(x):
        return np.bincount(ids, weights=(dJ.astype(np.float64) * x.astype(np.float64)[bdm]).sum(axis=1),
                           minlength=E)

    ref, t = [reduce(u)], 0.0
    for _ in range(nsteps):
        orc.linear_rk4(prob, u, v, t, dt, 1)
        t += dt
        ref.append(reduce(u))
    s = tgs._linear_solver(d, dtt)
    rec = s.record_elements(r, 0, nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    assert np.linalg.norm(ref) > 0
    assert rel_l2(rec.cpu().numpy(), np.array(ref)) <= (1e-12 if tag == "f64" else 1e-5)


@pytest.mark.gpu
def test_runs_split_over_calls_reattach_and_detach():
    """Calls of 1, 3, 1, 5 and 2 steps with a window straddling them; eager steps; re-attaching
    recaptures; detaching restores the launches of a solver that never had a receiver."""
    _torch()
    s, ref_solver, r, dt = _make("rk4", "stream", np.float64)
    ref = _stepwise(ref_solver, r, dt, 12)
    rec = s.record_elements(r, first=3, rows=15)
    s.init()
    for k, n in enumerate((1, 3, 1, 5, 2)):
        s.rk4(s.t if k else 0.0, dt, n)
        got = rec.cpu().numpy()
        done = s.nstep - 3 + 1
        assert np.isnan(got[max(done, 0):]).all(), s.nstep
        if done > 0:
            assert rel_l2(got[:done], ref[3:s.nstep + 1]) <= 1e-13, s.nstep
            assert got[done - 1].tobytes() == r(s.u).cpu().numpy().tobytes()
    graphs = s._graph
    rec2 = s.record_elements(r, first=0, rows=20)
    s.rk4(s.t, dt, 1)
    assert s._graph is not graphs
    got = rec2.cpu().numpy()
    assert np.isnan(got[:12]).all() and np.isnan(got[14:]).all() and np.isfinite(got[12:14]).all()
    s.step_eager(dt)
    assert rec2[14].cpu().numpy().tobytes() == r(s.u).cpu().numpy().tobytes()

    lib = _lib.lib()

    def launches(solver, n):
        before = lib.fus_launch_count()
        solver.rk4(solver.t, dt, n)
        return lib.fus_launch_count() - before

    s.use_graph = ref_solver.use_graph = False
    plain = launches(ref_solver, 3)
    assert launches(s, 3) == plain + 2 * (3 + 1)  # a launch pair per step and after the last
    s.record_elements(None)
    assert launches(s, 3) == plain and not s._recs


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["graph", "eager"])
def test_point_recorder_and_receiver_together(mode):
    """Both attached: each gives the rows it gives alone, and both record the final state."""
    _torch()
    import test_gpu_record_points as trp

    from fenicsx_fus_gpu_b200 import problem

    s, alone, r, dt = _make("rk4", "auto", np.float64)
    _, alone2, _, _ = _make("rk4", "auto", np.float64)
    # the set-up of the solvers' box (test_gpu_phased_array._piston)
    ev = trp._points_evaluator(problem.box_setup(3, 5, 0.006, np.float64, perturb=0.0, seed=1, geometry="auto"))
    for x in (s, alone, alone2):
        x.use_graph = mode == "graph"
    both = (s.record_points(ev, 2, 10), s.record_elements(r, 1, 12))
    only_p = alone.record_points(ev, 2, 10)
    only_e = alone2.record_elements(r, 1, 12)
    for x in (s, alone, alone2):
        x.init()
        x.rk4(0.0, dt, 6)
        x.rk4(x.t, dt, 5)
    # separate solvers: the stiffness atomics may sum in another order, so rounding apart
    got_p, got_e = both[0].cpu().numpy(), both[1].cpu().numpy()
    assert np.isfinite(got_e[:11]).all() and np.isnan(got_e[11:]).all() and np.isfinite(got_p).all()
    assert rel_l2(got_p, only_p.cpu().numpy()) <= 1e-13 and rel_l2(got_e[:11], only_e.cpu().numpy()[:11]) <= 1e-13
    assert got_p[-1].tobytes() == ev(s.u).cpu().numpy().tobytes()
    assert got_e[10].tobytes() == r(s.u).cpu().numpy().tobytes()


# --------------------------------------------------------------------------- #
# GPU: physics - reciprocity and echo timing
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["rk4", "leapfrog"])
def test_reciprocity_between_two_elements(integrator):
    """Transmit on a, receive on b = transmit on b, receive on a (symmetric stiffness, diagonal mass
    and damping, source weights = receive weights / rho).  RK4 with absorbing facets, leapfrog with
    none."""
    _torch()
    from fenicsx_fus_gpu_b200 import problem

    P, N, L = 3, 6, 0.006
    su = problem.box_setup(P, N, L, np.float64, perturb=0.08, seed=5)
    tile = problem.TileArray((0.5 * L, 0.5 * L, 0.0), 4, 4, L / 5)
    r = problem.element_receiver(su, [0], tile)
    dt = problem.cfl_time_step(P, L / N, 1500.0, 0.5e6, 0.5)
    nsteps = 160
    a, b = 0, 6  # a corner element, an off-axis one
    traces = {}
    for e in (a, b):
        if integrator == "rk4":
            absorbing = dict(absorbing_facets=[0, 1, 2, 3, 4, 5],
                             absorbing_predicate=lambda cen: ~((cen[:, 2] < 0.5 * L / N) & (tile.element_of(cen) >= 0)))
        else:
            absorbing = dict(absorbing_facets=[])
        s = problem.linear_solver(su, [0], integrator=integrator, source_elements=tile,
                                  element_amplitudes=(np.arange(16) == e).astype(float), **absorbing)
        rec = s.record_elements(r, 0, nsteps + 1)
        s.init()
        s.rk4(0.0, dt, nsteps)
        traces[e] = rec.cpu().numpy()
    ab, ba = traces[a][:, b], traces[b][:, a]
    err = rel_l2(ab, ba)
    print(f"\nreciprocity ({integrator}): rel-L2 {err:.3e} over {nsteps} steps, |r| max {np.abs(ab).max():.3e}")
    assert np.linalg.norm(ab) > 0
    assert err <= 1e-12


@pytest.mark.gpu
def test_echo_from_the_back_wall_arrives_at_the_round_trip():
    """A 3 x 3 array on z = 0 transmits; the back wall z = L reflects.  The echo at the centre element
    is the difference from a run with an absorbing back wall.  Its onset, the first step where it
    exceeds 5 % of its peak, must fall in [2L/c - T/4, 2L/c + 4T]: the waveform's envelope ramps up
    over 4 periods T, and the envelope reaches 5 % 0.57 T after the start."""
    _torch()
    from fenicsx_fus_gpu_b200 import problem

    P, N, L, f0, c0 = 3, 8, 0.008, 0.5e6, 1500.0
    T = 1.0 / f0
    su = problem.box_setup(P, N, L, np.float64, geometry="auto")
    tile = problem.TileArray((0.5 * L, 0.5 * L, 0.0), 3, 3, 0.002)
    aperture = lambda cen: (cen[:, 2] < 0.5 * L / N) & (tile.element_of(cen) >= 0)  # noqa: E731
    r = problem.element_receiver(su, [0], tile)
    dt = problem.cfl_time_step(P, L / N, c0, f0, 0.65)
    round_trip = 2 * L / c0
    nsteps = int((round_trip + 5 * T) / dt)
    traces = []
    for back in ("reflecting", "absorbing"):
        faces = [0, 1, 2, 3, 4] + ([5] if back == "absorbing" else [])
        s = problem.linear_solver(su, [0], faces, f0=f0, c0=c0, source_elements=tile, geometry="auto",
                                  absorbing_predicate=lambda cen: ~aperture(cen))
        rec = s.record_elements(r, 0, nsteps + 1)
        s.init()
        s.rk4(0.0, dt, nsteps)
        traces.append(rec.cpu().numpy()[:, 4])
    echo = traces[0] - traces[1]
    t = np.arange(nsteps + 1) * dt
    onset = t[np.argmax(np.abs(echo) > 0.05 * np.abs(echo).max())]
    print(f"\necho onset at the centre element: {onset * 1e6:.3f} us, round trip 2L/c = {round_trip * 1e6:.3f} us")
    assert np.isfinite(echo).all() and np.abs(echo).max() > 0
    assert round_trip - 0.25 * T <= onset <= round_trip + 4 * T


# --------------------------------------------------------------------------- #
# GPU: emulated ranks
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
@pytest.mark.parametrize("halo", ["nccl-shaped", "p2p"])
@pytest.mark.parametrize("partition", ["block", "blob"])
def test_emulated_ranks_sum_to_the_single_rank_rows(partition, halo):
    """Every rank receives on the array facets of its own cells; the rows and areas summed over the
    ranks equal the single-rank ones.  Some ranks hold no facet of some elements, or of any."""
    torch = _torch()
    import problems
    import test_gpu_phased_array as tpa
    from test_unstructured_partition import _renumbered
    from fenicsx_fus_gpu_b200 import problem, sampling as sp, substrate as S, utils
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, LocalCluster, P2PHaloExchange, local_fabric
    from fenicsx_fus_gpu_b200.solver import linear_source

    dtt = np.float64
    P, N, L, R = 3, (4, 4, 4), (0.012, 0.01, 0.011), 4
    first, rows, calls = 2, 9, (4, 6)
    tile = problem.TileArray((0.0, 0.35 * L[1], 5.0 / 11.0 * L[2]), 2, 2, 0.8 * L[1], axes=(1, 2))
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0)
    src = lambda t: linear_source(t, serial.f0, serial.p0, serial.c0)  # noqa: E731

    def receiver(q):
        ids = tile.element_of(problem.facet_centroids(q.mesh, S.boundary_facets(q.mesh, 2)))
        return sp.ElementReceiver(dtt, q.bfacet_dofmap1, q.detJ_f1, ids, 4)

    def run(s, r):
        rec = s.record_elements(r, first, rows)
        s.init()
        for k, n in enumerate(calls):
            s.rk4(s.t if k else 0.0, dt, n)
        torch.cuda.synchronize()
        return rec.cpu().numpy(), r.areas.cpu().numpy()

    ref, ref_areas = run(tpa._linear(serial, dtt, source=src), receiver(serial))
    assert np.isfinite(ref).all() and np.linalg.norm(ref) > 0
    if partition == "blob":
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                                  shuffle_seed=2, owner_rule="hash")
    else:
        parts = S.partition_box(N, P, R, lengths=L, dtype=dtt, perturb=0.1, seed=11)
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    ren = _renumbered(parts, sdata)
    ndmax = max(p.index_map.size_local + p.index_map.num_ghosts for p in parts)

    def body(rk, transport):
        p = parts[rk]
        nl, ng = p.index_map.size_local, p.index_map.num_ghosts
        if halo == "nccl-shaped":
            dm, od, gd = p.dofmap, *sdata[rk]
            h = HaloExchange(transport, od, gd, nl, dtt)
        else:
            dm, _, od, gd, _ = ren[rk]
            h = P2PHaloExchange(local_fabric(transport.cluster, rk, P2PHaloExchange.arena_bytes(ndmax, dtt)), od, gd,
                                nl, ng, dtt)
        q = problems.linear_problem(P, None, None, dtt, mesh=p.mesh, dofmap=dm, ndofs=nl + ng)
        s = tpa._linear(q, dtt, halo=h, source=src, use_graph=False)
        r = receiver(q)
        return r.nchunks, run(s, r)

    out = LocalCluster(R).run(body)
    assert any(n == 0 for n, _ in out) or any(not (a > 0).all() for _, (_, a) in out), "every rank sees every element"
    got = sum(o[1][0] for o in out)
    areas = sum(o[1][1] for o in out)
    assert rel_l2(areas, ref_areas) <= 1e-13
    assert rel_l2(got, ref) <= 1e-13


# --------------------------------------------------------------------------- #
# GPU: demo
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
def test_pulse_echo_demo(tmp_path):
    _torch()
    cmd = [sys.executable, os.path.join(ROOT, "demos", "demo_pulse_echo.py"), "--cells", "8", "--degree", "3",
           "--elements", "3,3", "--length", "0.008", "--sample-dir", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "nan" not in r.stdout.lower() and "echo" in r.stdout and "2L/c" in r.stdout
    traces = np.load(os.path.join(str(tmp_path), "element_traces.npy"))
    assert traces.ndim == 2 and traces.shape[1] == 9 and np.isfinite(traces).all() and np.abs(traces).max() > 0
