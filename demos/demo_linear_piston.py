"""Planar piston - the B200 twin of /root/reference/cuda/demo_linear_piston.py:
circular piston source (radius 10 mm) on z=0, every other exterior facet absorbing,
degree 5 (BASELINE.json configs[2]).  The reference reads the BM1-SC2 XDMF mesh,
which is not in its tree; here the domain is a box of hexahedra."""

import numpy as np

import _common

from fenicsx_fus_gpu_b200 import problem, substrate as S


def main():
    a = _common.parser(__doc__, degree=5, cells=93).parse_args()
    rank, world = _common.init()
    dtype = np.float64 if a.dtype == "f64" else np.float32
    f0, p0, c0, rho = 0.5e6, 60000.0, 1500.0, 1000.0  # demo_linear_piston.py:53-60
    L = 0.12
    h = L / 93
    grid = S.block_grid(world)
    ncells = tuple(a.cells * g for g in grid)
    lengths = tuple(h * n for n in ncells)
    su = problem.box_setup(a.degree, ncells, lengths, dtype, rank, world, grid=grid, geometry=a.geometry)
    centre = (0.5 * lengths[0], 0.5 * lengths[1])
    piston = problem.disc(0, 1, centre, 0.01)
    solver = problem.linear_solver(
        su, source_facets=[0], absorbing_facets=[0, 1, 2, 3, 4, 5], rho=rho, c0=c0, f0=f0, p0=p0,
        source_predicate=piston, absorbing_predicate=lambda cen: ~(piston(cen) & (cen[:, 2] < 0.5 * h)),
        geometry=a.geometry, integrator=a.integrator)
    dt = problem.cfl_time_step(a.degree, h, c0, f0, 0.65)
    tf = lengths[2] / c0 + 8.0 / f0  # :110
    nsteps = a.steps or int(tf / dt) + 1
    if rank == 0:
        print(f"Number of steps: {nsteps}; {su.global_dofs} dofs on {world} GPU(s)", flush=True)
    sampler = None
    if a.sample_dir:
        # the x-z sampling plane of cuda/demo_linear_piston.py:120-140 (141 x 241 points through the axis)
        from fenicsx_fus_gpu_b200 import sampling

        x_p = centre[0] + np.linspace(-0.035, 0.035, 141)
        z_p = np.linspace(0.0, lengths[2], 241)
        X_p, Z_p = np.meshgrid(x_p, z_p)
        points = np.zeros((3, X_p.size))
        points[0], points[1], points[2] = X_p.ravel(), centre[1], Z_p.ravel()
        x_eval, cell_eval = sampling.compute_eval_params(su.mesh, points, dtype)
        ev = sampling.PointEvaluator(a.degree, dtype, su.dev["dofmap"], su.mesh, x_eval, cell_eval, su.tables.pts_1d)
        period_steps = int(round(1.0 / f0 / dt))
        sampler = _common.PlaneSampler(ev, x_eval[:, [0, 2]], lengths[2] / c0 + 6.0 / f0, period_steps + 2,
                                       a.sample_dir, rank)
    _common.run(solver, 0.0, dt, nsteps, rank, sampler=sampler)
    _common.finish(world)


if __name__ == "__main__":
    main()
