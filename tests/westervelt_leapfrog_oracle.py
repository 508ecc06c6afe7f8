"""numpy restatement of the Westervelt leapfrog scheme of ``solver.WesterveltLeapfrog3D`` (pointwise
mass form), built from the oracle's operators beside ``oracle.westervelt_rk4`` as
``oracle.linear_leapfrog`` sits beside ``oracle.linear_rk4``.  The reference implements RK4 only, so
this restatement and its convergence to ``oracle.westervelt_rk4`` are what pin the scheme."""

import numpy as np

from oracle import oracle as orc


def diagonals(prob, nd, dtype):
    """``(m2, m5, absd)``: ``M(c2; 1)``, ``M(c5; 1)`` and the -1/(rho c) absorbing facets applied to
    ones."""
    ones = np.ones(nd, dtype)
    m2, m5, absd = (np.zeros(nd, dtype) for _ in range(3))
    orc.mass_operator(ones, prob.cell_coeff2, m2, prob.detJ, prob.dofmap)
    orc.mass_operator(ones, prob.cell_coeff5, m5, prob.detJ, prob.dofmap)
    if prob.bfacet_dofmap2.shape[0]:
        orc.mass_operator(ones, prob.facet_coeff2_2, absd, prob.detJ_f2, prob.bfacet_dofmap2)
    return m2, m5, absd


def westervelt_leapfrog(prob: orc.WesterveltProblem, u_, v_, t, dt, nsteps, source=None):
    """Operation for operation what the CUDA steps do (``prob.m0`` includes the absorbing facet term
    delta/(rho c^3)):

        kick-off  : w = v ; close with (m, bdt, cdt, adt) = (m0, -dt/2, dt/2, 0)
        each step : close with (m0 - dt/2 absd, dt, dt/2, dt)
        close     : b = K(c3; u) + K(c4; w) + g(t) src + dg(t) src2
                    a = (b + m5 w^2 + absd v) / (m + m2 u)
                    v += bdt a ; w = v + cdt a ; u += adt v

    ``source(t, b)`` (optional) adds the source terms to ``b`` instead of the single-waveform
    facets (an element-resolved phased array).  On return ``u_`` is u(t + nsteps dt) and ``v_`` is v
    half a step before; returns ``(t, w)``."""
    dtp = u_.dtype.type
    nd = u_.size
    m2, m5, absd = diagonals(prob, nd, u_.dtype)
    b, g, dg = (np.zeros(nd, u_.dtype) for _ in range(3))
    w = v_.copy()

    def step(tt, m, bdt, cdt, adt):
        b[:] = 0.0
        orc.stiffness_operator(prob.P, u_, prob.cell_coeff3, b, prob.G, prob.dofmap, prob.dphi_1D)
        orc.stiffness_operator(prob.P, w, prob.cell_coeff4, b, prob.G, prob.dofmap, prob.dphi_1D)
        if source is not None:
            source(tt, b)
        elif prob.bfacet_dofmap1.shape[0]:
            gv, dgv = orc.westervelt_source(tt, prob.f0, prob.p0, prob.c0)
            g[:] = gv
            dg[:] = dgv
            orc.mass_operator(g, prob.facet_coeff1_1, b, prob.detJ_f1, prob.bfacet_dofmap1)
            orc.mass_operator(dg, prob.facet_coeff2_1, b, prob.detJ_f1, prob.bfacet_dofmap1)
        a = (b + m5 * (w * w) + absd * v_) / (m + m2 * u_)
        v_[:] = v_ + dtp(bdt) * a
        w[:] = v_ + dtp(cdt) * a
        u_[:] = u_ + dtp(adt) * v_

    step(t, prob.m0, -0.5 * dt, 0.5 * dt, 0.0)
    mm = prob.m0 - dtp(0.5 * dt) * absd
    for _ in range(nsteps):
        step(t, mm, dt, 0.5 * dt, dt)
        t += dt
    return t, w
