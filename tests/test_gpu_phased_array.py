"""Phased-array sources: one waveform, amplitude and delay per array element
(``fus_boundary_terms_elements_*``, the ``source_elements`` keyword of the solvers, and
``problem.TileArray`` / ``focus_delays`` / ``element_source``).

The element-resolved oracle below is ``oracle.linear_rk4`` / ``linear_leapfrog`` /
``westervelt_rk4`` with the source facet mass applied per element: the reference
``mass_operator`` on the facets of element e with ``fill(g_e)``, in the order of the elements."""

import os
import subprocess
import sys

import numpy as np
import pytest

import test_stage_kernels as tsk
from fenicsx_fus_gpu_b200 import problem
from fenicsx_fus_gpu_b200 import substrate as S
from fenicsx_fus_gpu_b200.solver import linear_source, westervelt_source

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPES = [np.float64, np.float32]


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / (nb if nb > 0 else 1.0))


# --------------------------------------------------------------------------- #
# CPU: waveforms and array geometry
# --------------------------------------------------------------------------- #
def test_vectorised_sources_bit_identical_to_scalar_calls():
    t = np.concatenate([np.linspace(-1e-6, 2e-5, 2001), [0.0, 8e-6, 4.0 / 0.5e6, 4.0 / 1.1e6]])
    for f in (lambda x: linear_source(x, 0.5e6, 6e4, 1500.0), lambda x: westervelt_source(x, 1.1e6, 5.7e5, 1480.0)):
        g, dg = f(t)
        for i, ti in enumerate(t):
            gs, dgs = f(float(ti))
            assert np.float64(gs).tobytes() == g[i].tobytes(), ti
            assert np.float64(dgs).tobytes() == np.broadcast_to(dg, t.shape)[i].tobytes(), ti


def test_element_source_is_silent_before_its_delay():
    A = np.array([1.0, 0.5, 2.0, -1.0])
    tau = np.array([0.0, 1e-6, 3e-6, 2.5e-6])
    src = problem.element_source(lambda t: westervelt_source(t, 1.1e6, 5.7e5, 1480.0), A, tau)
    for t in np.linspace(0.0, 6e-6, 301):
        g, dg = src(t)
        assert g.shape == dg.shape == (4,)
        off = t < tau
        assert np.all(g[off] == 0.0) and np.all(dg[off] == 0.0)
        g0, dg0 = westervelt_source(t - tau, 1.1e6, 5.7e5, 1480.0)
        assert np.array_equal(g[~off], (A * g0)[~off]) and np.array_equal(dg[~off], (A * dg0)[~off])
    one = problem.element_source(lambda t: linear_source(t, 0.5e6, 6e4, 1500.0), [1.0], [0.0])
    for t in np.linspace(0.0, 1e-5, 57):  # one element, A = 1, tau = 0: the single source, bit for bit
        assert one(t)[0][0] == linear_source(t, 0.5e6, 6e4, 1500.0)[0]
    with pytest.raises(ValueError):
        problem.element_source(linear_source, [1.0, 2.0], [0.0])


def test_tile_array_ids_and_centres():
    tile = problem.TileArray((0.01, 0.02, 0.0), 3, 4, 0.002)
    assert tile.E == 12 and tile.centres.shape == (12, 3)
    for e, c in enumerate(tile.centres):
        ia, ib = divmod(e, 4)
        assert np.allclose(c, (0.01 + (ia - 1) * 0.002, 0.02 + (ib - 1.5) * 0.002, 0.0), rtol=0, atol=1e-15)
    # the centres, and points anywhere inside an element, map to that element
    rng = np.random.default_rng(0)
    jit = rng.uniform(-0.49, 0.49, (12, 3)) * 0.002
    jit[:, 2] = 0.0
    assert np.array_equal(tile.element_of(tile.centres), np.arange(12))
    assert np.array_equal(tile.element_of(tile.centres + jit), np.arange(12))
    outside = np.array([[0.01 - 0.0031, 0.02, 0.0], [0.01, 0.02 + 0.0041, 0.0], [0.0, 0.0, 0.0]])
    assert np.all(tile.element_of(outside) == -1)
    side = problem.TileArray((0.0, 0.005, 0.006), 2, 2, 0.001, axes=(1, 2))
    assert np.allclose(side.centres[:, 0], 0.0) and side.element_of([[0.0, 0.0052, 0.0061]])[0] == 3


def test_focus_delays_equalise_path_plus_delay():
    tile = problem.TileArray((0.01, 0.01, 0.0), 8, 6, 0.0015)
    c0 = 1500.0
    for focus in ((0.01, 0.01, 0.02), (0.014, 0.007, 0.015)):
        tau = problem.focus_delays(tile.centres, focus, c0)
        assert np.all(tau >= 0) and tau.min() == 0.0
        arrival = tau + np.linalg.norm(tile.centres - np.asarray(focus), axis=1) / c0
        assert np.ptp(arrival) <= 1e-15 * arrival.max() + 1e-22


# --------------------------------------------------------------------------- #
# GPU: the kernel against a float64 reference
# --------------------------------------------------------------------------- #
def _torch():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def elements_ref(b, vn, dof, row, elem, w, w2, absb, G, DG):
    """(value, Y): b[dof[i]] + sum_k (w G[elem] + w2 DG[elem]) + vn[dof] absb in float64, and Y the
    sum of the absolute values of every term (b included)."""
    n = dof.size
    rid = np.repeat(np.arange(n), np.diff(row))
    t1 = w * G[elem]
    t2 = w2 * DG[elem] if w2 is not None else np.zeros_like(t1)
    acc = np.bincount(rid, weights=t1 + t2, minlength=n)
    Y = np.bincount(rid, weights=np.abs(t1) + np.abs(t2), minlength=n)
    if absb is not None:
        acc = acc + vn[dof] * absb
        Y = Y + np.abs(vn[dof] * absb)
    out, Yo = b.copy(), np.zeros_like(b)
    out[dof] = b[dof] + acc
    Yo[dof] = np.abs(b[dof]) + Y
    return out, Yo


def _csr(rng, n, E, maxlen):
    """Row lengths 0..maxlen (every length present), distinct elements inside a row."""
    lens = rng.integers(0, maxlen + 1, n)
    lens[: min(n, maxlen + 1)] = np.arange(min(n, maxlen + 1))
    row = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    elem = np.concatenate([rng.choice(E, ln, replace=E < ln) for ln in lens] or [np.zeros(0)]).astype(np.int32)
    return row, elem


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_elements_kernel_vs_float64_reference(dt):
    torch = _torch()
    L = tsk._lib()
    rng = np.random.default_rng(21)
    st = torch.cuda.current_stream().cuda_stream
    f = lambda a: np.asarray(a, np.float64)  # noqa: E731
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    nd = 9000
    b0, vn = rng.standard_normal(nd).astype(dt), rng.standard_normal(nd).astype(dt)
    vnd = dv(vn)
    maxlen = 4
    k = maxlen + 3
    name = "fus_boundary_terms_elements"
    checked_mutants = 0
    for E in (1, 4096):
        rows = 3
        tab = rng.standard_normal((rows, 4, 2, E)).astype(dt)
        tabd = dv(tab)
        for n in (0, 1, 255, 256, 257, 1023, 1024, 1025, 5000):
            dof = rng.choice(nd, n, replace=False).astype(np.int32)
            row, elem = _csr(rng, n, E, maxlen)
            nk = int(row[-1])
            w, w2, absb = (rng.standard_normal(nk).astype(dt), rng.standard_normal(nk).astype(dt),
                           rng.standard_normal(n).astype(dt))
            dd, rd, ed, wd, w2d, ad = dv(dof), dv(row), dv(elem if nk else np.zeros(1, np.int32)), \
                dv(w if nk else np.zeros(1, dt)), dv(w2 if nk else np.zeros(1, dt)), dv(absb if n else np.zeros(1, dt))
            for use_w2, use_absb in ((True, True), (False, True), (True, False), (False, False)):
                for s, stage in ((None, 0), (None, 3), (2, 1), (1, 2)):
                    b = tsk.Dev(torch, b0, seed=stage)
                    step = torch.tensor([s], dtype=torch.int64, device="cuda") if s is not None else None
                    rc = L.fn(name, dt)(b.ptr, vnd.data_ptr(), dd.data_ptr(), rd.data_ptr(), ed.data_ptr(),
                                        wd.data_ptr(), w2d.data_ptr() if use_w2 else None,
                                        ad.data_ptr() if use_absb else None, tabd.data_ptr(),
                                        step.data_ptr() if step is not None else None, E, stage, n, st)
                    assert rc == 0, L.lib().fus_last_error()
                    torch.cuda.synchronize()
                    out = b.get()
                    r = s if s is not None else 0
                    G, DG = f(tab[r, stage, 0]), f(tab[r, stage, 1])
                    args = (f(b0), f(vn), dof, row, elem, f(w), f(w2) if use_w2 else None,
                            f(absb) if use_absb else None)
                    ref, Y = elements_ref(*args, G, DG)
                    off = np.ones(nd, bool)
                    off[dof] = False
                    assert tsk._bits_equal(out[off], b0[off])
                    tsk.check_bound(out, ref, Y, k, dt, "boundary_elements")
                    if E > 1 and n >= 1000 and use_w2:
                        mutants = [
                            elements_ref(*args[:4], (elem + 1) % E, *args[5:], G, DG),        # element ids shifted
                            elements_ref(*args, f(tab[r, (stage + 1) % 4, 0]), f(tab[r, (stage + 1) % 4, 1])),
                            elements_ref(*args, G, G),                                        # DG read as G
                        ]
                        if s is not None:
                            mutants.append(elements_ref(*args, f(tab[0, stage, 0]), f(tab[0, stage, 1])))
                        for mref, _ in mutants:
                            assert tsk.violates(out, mref, Y, k, dt)
                            checked_mutants += 1
    assert checked_mutants >= 3 * 3 * 2


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_elements_kernel_rejects_bad_arguments_before_launch(dt):
    torch = _torch()
    L = tsk._lib()
    st = torch.cuda.current_stream().cuda_stream
    x = torch.zeros(8, dtype=torch.float64 if dt == np.float64 else torch.float32, device="cuda")
    i = torch.zeros(8, dtype=torch.int32, device="cuda")
    p, q = x.data_ptr(), i.data_ptr()
    fn = L.fn("fus_boundary_terms_elements", dt)
    good = [p, p, q, q, q, p, p, p, p, None, 1, 0, 4, st]
    before = L.lib().fus_launch_count()
    for pos, bad in ((12, -1), (10, 0), (10, -3), (11, 4), (11, -1), (8, None), (3, None), (4, None), (5, None),
                     (2, None)):
        args = list(good)
        args[pos] = bad
        assert fn(*args) == tsk.BAD_ARGUMENT, (pos, bad)
    assert L.lib().fus_launch_count() == before
    assert fn(None, None, None, None, None, None, None, None, None, None, 5, 0, 0, st) == 0  # empty: no launch
    assert L.lib().fus_launch_count() == before
    sig = L.fn("fus_boundary_terms_elements_signal", dt)
    assert sig(None, *good[:-1], 0, st) == tsk.BAD_ARGUMENT
    assert fn(*good) == 0
    torch.cuda.synchronize()


# --------------------------------------------------------------------------- #
# GPU: solvers
# --------------------------------------------------------------------------- #
def _piston(P, N, dtt, geometry, integrator="rk4", tile=None, **kw):
    L = 0.006
    su = problem.box_setup(P, N, L, dtt, perturb=0.08 if geometry != "auto" else 0.0, seed=1, geometry=geometry)
    disc = problem.disc(0, 1, (0.5 * L, 0.5 * L), 0.35 * L)
    s = problem.linear_solver(su, [0], [1, 2, 3, 4, 5], source_predicate=disc, geometry=geometry,
                              integrator=integrator, source_elements=tile, **kw)
    return su, s, problem.cfl_time_step(P, L / N, 1500.0, 0.5e6, 0.5)


def _bowl(P, N, dtt, geometry, mass_form, tile=None, **kw):
    L = 0.005
    su = problem.box_setup(P, N, L, dtt, perturb=0.08 if geometry != "auto" else 0.0, seed=2, geometry=geometry)
    disc = problem.disc(1, 2, (0.5 * L, 0.5 * L), 0.3 * L)
    s = problem.westervelt_solver(su, [2], [0, 1, 3, 4, 5], f0=1.1e6, alpha_dB=20.0, source_predicate=disc,
                                  geometry=geometry, mass_form=mass_form, source_elements=tile, **kw)
    return su, s, problem.cfl_time_step(P, L / N, 1480.0, 1.1e6, 0.4)


def _whole_face(L, axes):
    """One element covering a whole box face."""
    c = [0.5 * L] * 3
    c[({0, 1, 2} - set(axes)).pop()] = 0.0
    return problem.TileArray(c, 1, 1, 4 * L, axes=axes)


def _run(s, dt, nsteps, mode):
    s.init()
    if mode == "graph":
        s.rk4(0.0, dt, nsteps)
    elif s.integrator == "leapfrog":
        s.use_graph = False
        s.rk4(0.0, dt, nsteps)
    else:
        for _ in range(nsteps):
            s.step_eager(dt)
    return s.u.cpu().numpy(), s.v.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("geometry", ["stream", "auto", "vertex"])
@pytest.mark.parametrize("kind", ["rk4", "leapfrog", "pointwise", "cells"])
def test_one_element_equals_the_single_source(kind, geometry, tag):
    """One element, A = 1, tau = 0, covering every source facet: the run of today's single-source
    solver, graph replay and eager steps."""
    _torch()
    dtt = np.float64 if tag == "f64" else np.float32
    tol = 1e-13 if tag == "f64" else 1e-6
    P, N, nsteps = 3, 5, 20
    for mode in ("graph", "eager"):
        out = []
        for tile in (None, "one"):
            if kind in ("rk4", "leapfrog"):
                t = _whole_face(0.006, (0, 1)) if tile else None
                su, s, dt = _piston(P, N, dtt, geometry, kind, t)
            else:
                t = _whole_face(0.005, (1, 2)) if tile else None
                su, s, dt = _bowl(P, N, dtt, geometry, kind, t)
            assert (s.num_elements == 1) == (tile is not None)
            out.append(_run(s, dt, nsteps, mode))
        assert np.linalg.norm(out[0][0]) > 0
        assert rel_l2(out[1][0], out[0][0]) <= tol, mode
        assert rel_l2(out[1][1], out[0][1]) <= tol, mode


# ---- the element-resolved oracle ------------------------------------------- #
def _split(q, ids, E):
    """Per element: (facet coefficient(s), detJ_f, facet dofmap) rows of its source facets."""
    return [np.flatnonzero(ids == e) for e in range(E)]


def _elem_mass(orc, sel, vals, coeff, dJ, fdm, b, dtp):
    g = np.zeros(b.size, dtp)
    for e, rows in enumerate(sel):
        if rows.size:
            g[:] = dtp.type(vals[e])
            orc.mass_operator(g, np.ascontiguousarray(coeff[rows]), b, np.ascontiguousarray(dJ[rows]),
                              np.ascontiguousarray(fdm[rows]))


def oracle_linear_rk4_elements(q, m, ids, E, src, u_, v_, t, dt, nsteps):
    """``oracle.linear_rk4`` with the per-element source."""
    from oracle import oracle as orc

    dtp = u_.dtype
    nd = u_.size
    sel = _split(q, ids, E)
    un, vn, u0, v0, b = (np.zeros(nd, dtp) for _ in range(5))
    ku, kv = u_.copy(), v_.copy()
    for _ in range(nsteps):
        u0[:], v0[:] = u_, v_
        for i in range(4):
            un[:], vn[:] = u0, v0
            un += dtp.type(orc.A_RUNGE[i] * dt) * ku
            vn += dtp.type(orc.A_RUNGE[i] * dt) * kv
            ku[:] = vn
            b[:] = 0.0
            orc.stiffness_operator(q.P, un, q.cell_coeff2, b, q.G, q.dofmap, q.tb.dphi_1D)
            _elem_mass(orc, sel, src(t + orc.C_RUNGE[i] * dt)[0], q.facet_coeff1, q.detJ_f1, q.bfacet_dofmap1, b, dtp)
            orc.mass_operator(vn, q.facet_coeff2, b, q.detJ_f2, q.bfacet_dofmap2)
            kv[:] = b / m
            u_ += dtp.type(orc.B_RUNGE[i] * dt) * ku
            v_ += dtp.type(orc.B_RUNGE[i] * dt) * kv
        t += dt


def oracle_linear_leapfrog_elements(q, m, ids, E, src, u_, v_, t, dt, nsteps):
    """``oracle.linear_leapfrog`` with the per-element source."""
    from oracle import oracle as orc

    dtp = u_.dtype
    nd = u_.size
    sel = _split(q, ids, E)
    b = np.zeros(nd, dtp)
    absd = np.zeros(nd, dtp)
    orc.mass_operator(np.ones(nd, dtp), q.facet_coeff2, absd, q.detJ_f2, q.bfacet_dofmap2)

    def assemble(tt):
        b[:] = 0.0
        orc.stiffness_operator(q.P, u_, q.cell_coeff2, b, q.G, q.dofmap, q.tb.dphi_1D)
        _elem_mass(orc, sel, src(tt)[0], q.facet_coeff1, q.detJ_f1, q.bfacet_dofmap1, b, dtp)
        orc.mass_operator(v_, q.facet_coeff2, b, q.detJ_f2, q.bfacet_dofmap2)

    assemble(t)
    v_ += dtp.type(-0.5 * dt) * (b / m)
    mlf = m - dtp.type(0.5 * dt) * absd
    for _ in range(nsteps):
        assemble(t)
        v_ += dtp.type(dt) * (b / mlf)
        u_ += dtp.type(dt) * v_
        t += dt


def oracle_westervelt_rk4_elements(q, m0, ids, E, src, u_, v_, t, dt, nsteps):
    """``oracle.westervelt_rk4`` with the per-element source (g and dg per element)."""
    from oracle import oracle as orc

    dtp = u_.dtype
    nd = u_.size
    sel = _split(q, ids, E)
    un, vn, u0, v0, b, m = (np.zeros(nd, dtp) for _ in range(6))
    ku, kv = u_.copy(), v_.copy()
    for _ in range(nsteps):
        u0[:], v0[:] = u_, v_
        for i in range(4):
            un[:], vn[:] = u0, v0
            un += dtp.type(orc.A_RUNGE[i] * dt) * ku
            vn += dtp.type(orc.A_RUNGE[i] * dt) * kv
            ku[:] = vn
            g, dg = src(t + orc.C_RUNGE[i] * dt)
            m[:] = 0.0
            orc.mass_operator(un, q.cell_coeff2, m, q.detJ, q.dofmap)
            m += m0
            b[:] = 0.0
            orc.stiffness_operator(q.P, un, q.cell_coeff3, b, q.G, q.dofmap, q.tb.dphi_1D)
            orc.stiffness_operator(q.P, vn, q.cell_coeff4, b, q.G, q.dofmap, q.tb.dphi_1D)
            orc.mass_operator(vn * vn, q.cell_coeff5, b, q.detJ, q.dofmap)
            _elem_mass(orc, sel, g, q.facet_coeff1_1, q.detJ_f1, q.bfacet_dofmap1, b, dtp)
            _elem_mass(orc, sel, dg, q.facet_coeff2_1, q.detJ_f1, q.bfacet_dofmap1, b, dtp)
            orc.mass_operator(vn, q.facet_coeff2_2, b, q.detJ_f2, q.bfacet_dofmap2)
            kv[:] = b / m
            u_ += dtp.type(orc.B_RUNGE[i] * dt) * ku
            v_ += dtp.type(orc.B_RUNGE[i] * dt) * kv
        t += dt


def _array_problem(dtt, westervelt=False, N=5, P=3):
    """Box with the source on the whole face x = 0 split into a 2 x 3 array, every element with its
    own amplitude and delay (the delays fall inside the run)."""
    import problems

    L = 0.006
    build = problems.westervelt_problem if westervelt else problems.linear_problem
    q = build(P, N, L, dtt, perturb=0.1, seed=7)
    bd1 = np.concatenate([S.boundary_facets(q.mesh, 2)])
    tile = problem.TileArray((0.0, 0.55 * L, 0.5 * L), 2, 3, L / 1.9, axes=(1, 2))  # covers the face
    ids = tile.element_of(problem.facet_centroids(q.mesh, bd1))
    assert (ids >= 0).all() and np.unique(ids).size == 6
    dt = problems.cfl_dt(P, L / N, q.c0, q.f0, cfl=0.4 if westervelt else 0.65)
    A = np.array([1.0, -0.6, 1.7, 0.3, 0.9, -1.2])
    tau = np.array([0.0, 3.0, 7.5, 1.2, 11.0, 5.0]) * dt
    base = (lambda t: westervelt_source(t, q.f0, q.p0, q.c0)) if westervelt else (
        lambda t: linear_source(t, q.f0, q.p0, q.c0))
    return q, ids, 6, problem.element_source(base, A, tau), dt


def _linear(q, dtt, cls=None, **kw):
    from fenicsx_fus_gpu_b200.solver import LinearSpectral3D

    cls = cls or LinearSpectral3D
    return cls(q.P, dtt, q.ndofs, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2,
               q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1, q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff2, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("kind", ["rk4", "leapfrog", "pointwise", "cells"])
def test_array_vs_element_resolved_oracle(kind, tag):
    _torch()
    from fenicsx_fus_gpu_b200.solver import LinearLeapfrog3D, WesterveltSpectral3D
    from oracle import oracle as orc

    dtt = np.float64 if tag == "f64" else np.float32
    west = kind in ("pointwise", "cells")
    q, ids, E, src, dt = _array_problem(dtt, west)
    nsteps = 20
    ones = np.ones(q.ndofs, dtt)
    u_ref, v_ref = np.zeros(q.ndofs, dtt), np.zeros(q.ndofs, dtt)
    m = np.zeros(q.ndofs, dtt)
    orc.mass_operator(ones, q.cell_coeff1, m, q.detJ, q.dofmap)
    if west:
        orc.mass_operator(ones, q.facet_coeff1_2, m, q.detJ_f2, q.bfacet_dofmap2)
        oracle_westervelt_rk4_elements(q, m, ids, E, src, u_ref, v_ref, 0.0, dt, nsteps)
        s = WesterveltSpectral3D(
            q.P, dtt, q.ndofs, q.dofmap, q.G, q.detJ, q.tb.dphi_1D, q.cell_coeff1, q.cell_coeff2, q.cell_coeff3,
            q.cell_coeff4, q.cell_coeff5, q.bfacet_dofmap1, q.detJ_f1, q.facet_coeff1_1, q.facet_coeff2_1,
            q.bfacet_dofmap2, q.detJ_f2, q.facet_coeff1_2, q.facet_coeff2_2, source=src, mass_form=kind,
            source_elements=ids, num_elements=E)
    elif kind == "rk4":
        oracle_linear_rk4_elements(q, m, ids, E, src, u_ref, v_ref, 0.0, dt, nsteps)
        s = _linear(q, dtt, source=src, source_elements=ids)
    else:
        oracle_linear_leapfrog_elements(q, m, ids, E, src, u_ref, v_ref, 0.0, dt, nsteps)
        s = _linear(q, dtt, LinearLeapfrog3D, source=src, source_elements=ids)
    assert s.num_elements == E
    s.init()
    s.rk4(0.0, dt, nsteps)
    tol = 1e-12 if tag == "f64" else 1e-5
    assert np.linalg.norm(u_ref) > 0
    assert rel_l2(s.u.cpu().numpy(), u_ref) <= tol
    assert rel_l2(s.v.cpu().numpy(), v_ref) <= tol


@pytest.mark.gpu
def test_superposition_of_elements():
    _torch()
    dtt = np.float64
    q, ids, E, src, dt = _array_problem(dtt)
    A = np.array([1.0, -0.6, 1.7, 0.3, 0.9, -1.2])
    tau = np.array([0.0, 3.0, 7.5, 1.2, 11.0, 5.0]) * dt
    base = lambda t: linear_source(t, q.f0, q.p0, q.c0)  # noqa: E731
    nsteps = 24

    def run(amps):
        s = _linear(q, dtt, source=problem.element_source(base, amps, tau), source_elements=ids, num_elements=E)
        s.init()
        s.rk4(0.0, dt, nsteps)
        return s.u.cpu().numpy(), s.v.cpu().numpy()

    u_all, v_all = run(A)
    parts = [run(np.where(np.arange(E) == e, A, 0.0)) for e in range(E)]
    assert all(np.linalg.norm(p[0]) > 0 for p in parts)
    assert rel_l2(sum(p[0] for p in parts), u_all) <= 1e-12
    assert rel_l2(sum(p[1] for p in parts), v_all) <= 1e-12


@pytest.mark.gpu
def test_time_invariance_under_a_common_delay():
    _torch()
    dtt = np.float64
    q, ids, E, _, dt = _array_problem(dtt)
    A = np.array([1.0, -0.6, 1.7, 0.3, 0.9, -1.2])
    tau = np.array([0.0, 3.0, 7.5, 1.2, 11.0, 5.0]) * dt
    base = lambda t: linear_source(t, q.f0, q.p0, q.c0)  # noqa: E731
    N, k = 20, 7
    out = []
    for shift, steps in ((0.0, N), (k * dt, N + k)):
        s = _linear(q, dtt, source=problem.element_source(base, A, tau + shift), source_elements=ids)
        s.init()
        s.rk4(0.0, dt, steps)
        out.append((s.u.cpu().numpy(), s.v.cpu().numpy()))
    assert np.linalg.norm(out[0][0]) > 0
    assert rel_l2(out[1][0], out[0][0]) <= 1e-10
    assert rel_l2(out[1][1], out[0][1]) <= 1e-10


@pytest.mark.gpu
def test_resteering_reuses_the_captured_graphs():
    """New delays on the same solver: the captured graphs replay the new table (no recapture) and
    the result is that of a solver built with the new delays."""
    _torch()
    dtt = np.float64
    q, ids, E, src, dt = _array_problem(dtt)
    base = lambda t: linear_source(t, q.f0, q.p0, q.c0)  # noqa: E731
    A = np.ones(E)
    s = _linear(q, dtt, source=src, source_elements=ids, num_elements=E)
    s.init()
    s.rk4(0.0, dt, 12)
    graphs, tab = list(s._graph), s.gtab.data_ptr()
    u_first = s.u.cpu().numpy()
    tau2 = np.array([9.0, 0.0, 2.0, 4.0, 1.0, 6.5]) * dt
    s.source = problem.element_source(base, A, tau2)
    s.init()
    s.rk4(0.0, dt, 12)
    assert all(a is b for a, b in zip(s._graph, graphs)) and s.gtab.data_ptr() == tab
    fresh = _linear(q, dtt, source=problem.element_source(base, A, tau2), source_elements=ids)
    fresh.init()
    fresh.rk4(0.0, dt, 12)
    assert rel_l2(s.u.cpu().numpy(), u_first) > 1e-3
    assert rel_l2(s.u.cpu().numpy(), fresh.u.cpu().numpy()) <= 1e-13
    assert rel_l2(s.v.cpu().numpy(), fresh.v.cpu().numpy()) <= 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("halo", ["nccl-shaped", "p2p-none", "p2p-two", "p2p-fused"])
@pytest.mark.parametrize("partition", ["block", "blob"])
def test_emulated_ranks_vs_single_rank(partition, halo):
    """Ranks emulated on one GPU; the elements' facets span several ranks, and some ranks hold no
    source facet at all."""
    torch = _torch()
    import problems
    from test_unstructured_partition import _renumbered
    from fenicsx_fus_gpu_b200 import utils
    from fenicsx_fus_gpu_b200.scatterer import HaloExchange, LocalCluster, P2PHaloExchange, local_fabric

    dtt = np.float64
    P, N, L, R, nsteps = 3, (4, 4, 4), (0.012, 0.01, 0.011), 4, 10
    # 2 x 2 elements over the whole face x = 0, their seams off the middle, where block partitions cut
    tile = problem.TileArray((0.0, 0.35 * L[1], 5.0 / 11.0 * L[2]), 2, 2, 0.8 * L[1], axes=(1, 2))
    serial = problems.linear_problem(P, N, L, dtt, perturb=0.1, seed=11)
    dt = problems.cfl_dt(P, min(L[i] / N[i] for i in range(3)), serial.c0, serial.f0)
    A, tau = np.array([1.0, 0.4, -0.8, 1.3]), np.array([0.0, 2.0, 5.0, 3.5]) * dt
    src = problem.element_source(lambda t: linear_source(t, serial.f0, serial.p0, serial.c0), A, tau)

    def ids_of(q):
        return tile.element_of(problem.facet_centroids(q.mesh, S.boundary_facets(q.mesh, 2)))

    ref = _linear(serial, dtt, source=src, source_elements=ids_of(serial), num_elements=4)
    ref.init()
    ref.rk4(0.0, dt, nsteps)
    u_ref, v_ref = ref.u.cpu().numpy(), ref.v.cpu().numpy()
    if partition == "blob":
        parts = S.partition_cells(N, P, S.blob_cell_ranks(N, R, seed=3), lengths=L, dtype=dtt, perturb=0.1, seed=11,
                                  shuffle_seed=2, owner_rule="hash")
    else:
        parts = S.partition_box(N, P, R, lengths=L, dtype=dtt, perturb=0.1, seed=11)
    sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
    ren = _renumbered(parts, sdata)
    ndmax = max(p.index_map.size_local + p.index_map.num_ghosts for p in parts)
    seen = [set(np.unique(ids_of(p))) for p in parts]
    assert sum(e in sn for sn in seen for e in range(4)) > 4, "no element spans two ranks"

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
        s = _linear(q, dtt, halo=h, source=src, source_elements=ids_of(q), num_elements=4, use_graph=False)
        if halo != "nccl-shaped":
            s.split_mode = halo.split("-")[1]
        s.init()
        s.rk4(0.0, dt, nsteps)
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


@pytest.mark.gpu
def test_bad_element_input_raises_before_any_kernel():
    _torch()
    dtt = np.float64
    q, ids, E, src, dt = _array_problem(dtt)
    with pytest.raises(ValueError):
        _linear(q, dtt, source=src, source_elements=ids, num_elements=5)  # ids up to 5
    bad = ids.copy()
    bad[3] = -1
    with pytest.raises(ValueError):
        _linear(q, dtt, source=src, source_elements=bad)
    with pytest.raises(ValueError):
        _linear(q, dtt, source=src, source_elements=ids[:-1])  # not one per facet row
    s = _linear(q, dtt, source=lambda t: (np.zeros(E + 1), np.zeros(E + 1)), source_elements=ids)
    s.init()
    with pytest.raises(ValueError):
        s.rk4(0.0, dt, 2)
    with pytest.raises(ValueError):
        s.step_eager(dt)


@pytest.mark.gpu
def test_steered_array_focuses_off_axis():
    """A 12 mm (4 wavelength) 8 x 8 array, pitch lambda / 2, on z = 0 of a water box, focused at
    10 mm depth and 3 mm off axis: over the last period, |p| at the focus is larger than at its
    mirror point across the array axis.  Measured on an NVIDIA B200 (1000 W power limit): 13.8
    (peaks 2.22e5 and 1.61e4).  No threshold above 1 is assumed."""
    torch = _torch()
    from fenicsx_fus_gpu_b200 import sampling

    dtt, P, N, Lb = np.float64, 4, 16, 0.016
    f0, c0 = 0.5e6, 1500.0
    h = Lb / N
    su = problem.box_setup(P, N, Lb, dtt, geometry="auto")
    tile = problem.TileArray((0.5 * Lb, 0.5 * Lb, 0.0), 8, 8, 0.0015)
    focus = np.array([0.5 * Lb + 0.003, 0.5 * Lb, 0.010])
    mirror = focus - [0.006, 0.0, 0.0]
    tau = problem.focus_delays(tile.centres, focus, c0)
    s = problem.linear_solver(su, [0], [0, 1, 2, 3, 4, 5], f0=f0, c0=c0, source_elements=tile, element_delays=tau,
                              absorbing_predicate=lambda cen: ~((cen[:, 2] < 0.5 * h) & (tile.element_of(cen) >= 0)),
                              geometry="auto")
    x_eval, cell_eval = sampling.compute_eval_params(su.mesh, np.stack([focus, mirror], axis=1), dtt)
    ev = sampling.PointEvaluator(P, dtt, su.dev["dofmap"], su.mesh, x_eval, cell_eval, su.tables.pts_1d)
    dt = problem.cfl_time_step(P, h, c0, f0, 0.65)
    arrival = np.linalg.norm(tile.centres - focus, axis=1).max() / c0  # the same for every element
    nsteps = int((arrival + 4.5 / f0) / dt) + 1  # past the 4-period ramp of the waveform
    s.init()
    s.rk4(0.0, dt, nsteps)
    peak = np.zeros(2)
    for _ in range(int(round(1.0 / f0 / dt))):
        s.rk4(s.t, dt, 1)
        peak = np.maximum(peak, np.abs(ev.to_host(s.u)))
    torch.cuda.synchronize()
    ratio = peak[0] / peak[1]
    print(f"\nfocus / mirror amplitude ratio: {ratio:.3f} (peaks {peak})")
    assert np.all(np.isfinite(peak)) and ratio > 1.0


@pytest.mark.gpu
def test_demo_phased_array_runs():
    _torch()
    cmd = [sys.executable, os.path.join(ROOT, "demos", "demo_phased_array.py"), "--cells", "8", "--degree", "3",
           "--elements", "4,4", "--focus", "0.002,0,0.006", "--periods", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "nan" not in r.stdout.lower() and "peak" in r.stdout
