"""Focused transducer, Westervelt equation - the B200 twin of
/root/reference/cuda/demo_nonlinear_bowl.py (c = 1480 m/s, f = 1.1 MHz, beta = 3.5,
alpha = 0.2 dB, CFL 0.4; every exterior facet absorbing as :282-285 does).  The reference
reads the H131 bowl mesh, which is not in its tree; here the source is a disc on x=0 of a
box of hexahedra (BASELINE.json configs[3]: degree 4)."""

import numpy as np

import _common

from fenicsx_fus_gpu_b200 import problem, substrate as S


def main():
    a = _common.parser(__doc__, degree=4, cells=99).parse_args()
    rank, world = _common.init()
    dtype = np.float64 if a.dtype == "f64" else np.float32
    c0, rho, f0 = 1480.0, 1000.0, 1.1e6  # demo_nonlinear_bowl.py:61-64
    p0 = rho * c0 * 0.38557513826589934
    L = 0.08  # :77
    h = L / 198  # 198^3 cells of degree 4 = 498.7 M dofs on 8 GPUs (99 per direction per GPU)
    grid = S.block_grid(world)
    ncells = tuple(a.cells * g for g in grid)
    lengths = tuple(h * n for n in ncells)
    su = problem.box_setup(a.degree, ncells, lengths, dtype, rank, world, grid=grid, geometry=a.geometry)
    centre = (0.5 * lengths[1], 0.5 * lengths[2])
    solver = problem.westervelt_solver(
        su, source_facets=[2], absorbing_facets=[0, 1, 2, 3, 4, 5], rho=rho, c0=c0, f0=f0, p0=p0, beta=3.5,
        alpha_dB=0.2, source_predicate=problem.disc(1, 2, centre, 0.3 * lengths[1]), geometry=a.geometry)
    dt = problem.cfl_time_step(a.degree, h, c0, f0, 0.40)  # :122
    tf = lengths[0] / c0 + 8.0 / f0
    nsteps = a.steps or int(tf / dt) + 1
    if rank == 0:
        print(f"Number of steps: {nsteps}; {su.global_dofs} dofs on {world} GPU(s)", flush=True)
    _common.run(solver, 0.0, dt, nsteps, rank)
    _common.finish(world)


if __name__ == "__main__":
    main()
