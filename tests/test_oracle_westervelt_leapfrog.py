"""CPU: the numpy restatement of the Westervelt leapfrog scheme (``westervelt_leapfrog_oracle``, what
the product's WesterveltLeapfrog3D implements; the reference has RK4 only) converges to the oracle's
Westervelt RK4 solution with dt^2, on a problem whose nonlinear (beta) and diffusive (delta) terms
both change the solution by far more than the leapfrog error."""

import numpy as np

import problems
import westervelt_leapfrog_oracle as wlo
from oracle import oracle as orc

P, N, L, P0, NSTEPS = 2, 4, 0.012, 3.0e6, 48


def _prob(d):
    ones = np.ones(d.ndofs)
    m0 = np.zeros(d.ndofs)
    orc.mass_operator(ones, d.cell_coeff1, m0, d.detJ, d.dofmap)
    orc.mass_operator(ones, d.facet_coeff1_2, m0, d.detJ_f2, d.bfacet_dofmap2)
    return orc.WesterveltProblem(d.P, d.dofmap, d.G, d.detJ, d.tb.dphi_1D, d.cell_coeff2, d.cell_coeff3,
                                 d.cell_coeff4, d.cell_coeff5, m0, d.bfacet_dofmap1, d.detJ_f1, d.facet_coeff1_1,
                                 d.facet_coeff2_1, d.bfacet_dofmap2, d.detJ_f2, d.facet_coeff2_2, d.f0, d.p0, d.c0)


def _rk4(d, dt, nsteps):
    u, v = np.zeros(d.ndofs), np.zeros(d.ndofs)
    orc.westervelt_rk4(_prob(d), u, v, 0.0, dt, nsteps)
    return u


def test_oracle_westervelt_leapfrog_second_order_against_oracle_rk4():
    kw = dict(perturb=0.1, seed=2, p0=P0)  # alpha_dB = 20 (the test problems' default)
    d = problems.westervelt_problem(P, N, L, np.float64, **kw)
    prob = _prob(d)
    dt0 = problems.cfl_dt(P, L / N, d.c0, d.f0, cfl=0.4)
    # RK4 at dt0/32: its time error is orders of magnitude below the finest leapfrog one
    u_ref = _rk4(d, dt0 / 32, NSTEPS * 32)
    assert np.linalg.norm(u_ref) > 0
    errs = []
    for k in (32, 64, 128):
        u, v = np.zeros(d.ndofs), np.zeros(d.ndofs)
        t, w = wlo.westervelt_leapfrog(prob, u, v, 0.0, dt0 / k, NSTEPS * k)
        assert abs(t - NSTEPS * dt0) < 1e-14
        assert np.isfinite(w).all()
        errs.append(orc.rel_l2(u, u_ref))
    assert 3.5 < errs[0] / errs[1] < 4.6 and 3.5 < errs[1] / errs[2] < 4.6, errs
    # the terms the leapfrog treats explicitly at the extrapolated velocity (and the mass at u^n) matter:
    # dropping either changes the reference by more than 10x the finest leapfrog error
    no_beta = _rk4(problems.westervelt_problem(P, N, L, np.float64, beta=0.0, **kw), dt0 / 32, NSTEPS * 32)
    no_delta = _rk4(problems.westervelt_problem(P, N, L, np.float64, alpha_dB=0.0, **kw), dt0 / 32, NSTEPS * 32)
    assert orc.rel_l2(no_beta, u_ref) > 10 * errs[2], (orc.rel_l2(no_beta, u_ref), errs)
    assert orc.rel_l2(no_delta, u_ref) > 10 * errs[2], (orc.rel_l2(no_delta, u_ref), errs)
