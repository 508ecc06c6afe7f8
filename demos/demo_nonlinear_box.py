"""Westervelt equation in a box - the B200 twin of
/root/reference/cuda/demo_nonlinear_box.py (degree 6, beta = 100, alpha = 50 dB, CFL 0.7,
source on x=0, absorbing x=L)."""

import numpy as np

import _common

from fenicsx_fus_gpu_b200 import problem, substrate as S


def main():
    a = _common.parser(__doc__, degree=6, cells=40).parse_args()
    rank, world = _common.init()
    dtype = np.float64 if a.dtype == "f64" else np.float32
    f0, p0, c0, rho = 0.5e6, 60000.0, 1500.0, 1000.0  # demo_nonlinear_box.py:62-69
    L = 0.12
    h = L / int(1 * L / (c0 / f0))  # :97-99
    grid = S.block_grid(world)
    ncells = tuple(a.cells * g for g in grid)
    lengths = tuple(h * n for n in ncells)
    su = problem.box_setup(a.degree, ncells, lengths, dtype, rank, world, grid=grid, geometry=a.geometry)
    solver = problem.westervelt_solver(su, source_facets=[2], absorbing_facets=[3], rho=rho, c0=c0, f0=f0,
                                       p0=p0, beta=100.0, alpha_dB=50.0, geometry=a.geometry)
    dt = problem.cfl_time_step(a.degree, h, c0, f0, 0.70)  # :128
    tf = lengths[0] / c0 + 2.0 / f0
    nsteps = a.steps or int(tf / dt) + 1
    if rank == 0:
        print(f"Number of steps: {nsteps}; {su.global_dofs} dofs on {world} GPU(s)", flush=True)
    _common.run(solver, 0.0, dt, nsteps, rank)
    _common.finish(world)


if __name__ == "__main__":
    main()
