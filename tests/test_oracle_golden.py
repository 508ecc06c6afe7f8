"""Pins oracle/ (the C restatement and the compiled reference templates)
against the fixtures the reference's own Python produced
(tests/golden/make_golden.py).  CPU only."""

import os

import numpy as np
import pytest

from oracle import oracle as orc

TOL = {"f64": 1e-13, "f32": 2e-6}


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_operators_match_reference(golden_dir, P, tag):
    g = _load(golden_dir, f"operators_P{P}_{tag}.npz")
    dt = g["x"].dtype
    nd = g["x"].size
    y = np.zeros(nd, dt)
    orc.mass_operator(g["x"], g["coeff"], y, g["detJ"], g["dofmap"])
    assert orc.rel_l2(y, g["y_mass"]) < TOL[tag]
    y = np.zeros(nd, dt)
    orc.stiffness_operator(P, g["x"], g["coeff"], y, g["G"], g["dofmap"], g["dphi_1D"])
    assert orc.rel_l2(y, g["y_stiff"]) < TOL[tag]
    y = np.zeros(nd, dt)
    orc.mass_operator(g["x"], g["fcoeff"], y, g["detJ_f"], g["bdofmap"])
    assert orc.rel_l2(y, g["y_fmass"]) < TOL[tag]


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_compiled_reference_templates_match(golden_dir, P, tag):
    if orc.ref_lib() is None:
        pytest.skip("oracle/_ref not built: needs the reference's C++ sources, which the repository does not hold")
    g = _load(golden_dir, f"operators_P{P}_{tag}.npz")
    y = np.zeros(g["x"].size, g["x"].dtype)
    orc.ref_stiffness_operator(P, g["x"], g["coeff"], y, g["G"], g["dofmap"], g["dphi_1D"])
    assert orc.rel_l2(y, g["y_stiff"]) < TOL[tag]
    y = np.zeros(g["x"].size, g["x"].dtype)
    orc.ref_mass_operator(g["x"], g["coeff"], y, g["detJ"], g["dofmap"])
    assert orc.rel_l2(y, g["y_mass"]) < TOL[tag]


@pytest.mark.parametrize("P", range(2, 8))
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_geometry_matches_reference(golden_dir, P, tag):
    g = _load(golden_dir, f"operators_P{P}_{tag}.npz")
    dt = g["x"].dtype
    tol = 1e-12 if tag == "f64" else 2e-4  # f32 LAPACK inverse vs adjugate on jittered cells
    mesh = (g["x_dofs"], g["x_g"])
    Nc = g["dofmap"].shape[0]
    detJ = np.zeros_like(g["detJ"])
    orc.compute_scaled_jacobian_determinant(detJ, mesh, Nc, g["dphi"], g["wts"])
    assert orc.rel_l2(detJ, g["detJ"]) < tol
    G = np.zeros_like(g["G"])
    orc.compute_scaled_geometrical_factor(G, mesh, Nc, g["dphi"], g["wts"])
    assert orc.rel_l2(G, g["G"]) < tol
    dJf = np.zeros_like(g["detJ_f"])
    orc.compute_boundary_facets_scaled_jacobian_determinant(dJf, mesh, g["bdata"], g["dphi_f"], g["wts_f"])
    assert orc.rel_l2(dJf, g["detJ_f"]) < tol
    assert dt == detJ.dtype


def test_vector_ops(golden_dir):
    g = _load(golden_dir, "vector_ops.npz")
    y = g["y"].copy()
    orc.axpy(float(g["alpha"]), g["a"], y)
    assert orc.rel_l2(y, g["y_axpy"]) < 1e-15
    c = np.zeros_like(y)
    orc.pointwise_divide(g["a"], g["b"], c)
    assert orc.rel_l2(c, g["c_div"]) < 1e-15
    orc.copy(g["a"], c)
    assert np.array_equal(c, g["b_copy"])
    orc.fill(2.5, c)
    assert np.array_equal(c, g["f_fill"])
    orc.square(g["a"], c)
    assert np.array_equal(c, g["a"] * g["a"])
