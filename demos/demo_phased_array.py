"""Phased array - a planar array of na x nb square elements on z = 0 of a water box (linear
wave equation, f = 0.5 MHz), every other facet absorbing.  Each element fires with the delay
that focuses the array on ``--focus`` (metres from the centre of the array: lateral x, lateral
y, depth z; off-axis points steer the focus electronically, on the same mesh).  The x-z plane
through the focus is recorded every step of the last period; the script prints where |p| peaks there
and how far that is from the requested focus."""

import numpy as np

import _common

from fenicsx_fus_gpu_b200 import problem, substrate as S


def main():
    ap = _common.parser(__doc__, degree=4, cells=40)
    ap.add_argument("--length", type=float, default=0.03, help="box edge in metres (one GPU; scaled with the GPU grid)")
    ap.add_argument("--elements", default="16,16", help="NA,NB elements of the array")
    ap.add_argument("--pitch", type=float, default=0.0015, help="element pitch in metres (default: half a wavelength)")
    ap.add_argument("--focus", default="0.004,0,0.015", help="x,y,z of the focus from the array centre, metres")
    ap.add_argument("--periods", type=int, default=2, help="periods simulated after the focus is reached")
    a = ap.parse_args()
    rank, world = _common.init()
    dtype = np.float64 if a.dtype == "f64" else np.float32
    f0, c0, rho = 0.5e6, 1500.0, 1000.0
    h = a.length / a.cells
    grid = S.block_grid(world)
    ncells = tuple(a.cells * g for g in grid)
    lengths = tuple(h * n for n in ncells)
    su = problem.box_setup(a.degree, ncells, lengths, dtype, rank, world, grid=grid, geometry=a.geometry)
    na, nb = (int(v) for v in a.elements.split(","))
    centre = np.array([0.5 * lengths[0], 0.5 * lengths[1], 0.0])
    tile = problem.TileArray(centre, na, nb, a.pitch)
    focus = centre + np.array([float(v) for v in a.focus.split(",")])
    delays = problem.focus_delays(tile.centres, focus, c0)
    solver = problem.linear_solver(
        su, source_facets=[0], absorbing_facets=[0, 1, 2, 3, 4, 5], rho=rho, c0=c0, f0=f0,
        source_elements=tile, element_delays=delays,
        absorbing_predicate=lambda cen: ~((cen[:, 2] < 0.5 * h) & (tile.element_of(cen) >= 0)),
        geometry=a.geometry, integrator=a.integrator)
    dt = problem.cfl_time_step(a.degree, h, c0, f0, 0.65)
    period = int(round(1.0 / f0 / dt))
    # every element's wave reaches the focus at the same time; the waveform ramps up over 4 periods
    arrival = float(np.linalg.norm(tile.centres - focus, axis=1).max()) / c0
    nsteps = a.steps or int((arrival + (4 + a.periods) / f0) / dt) + 1
    nsteps = max(nsteps, period + 1)
    if rank == 0:
        print(f"Number of steps: {nsteps}; {su.global_dofs} dofs on {world} GPU(s); {tile.E} elements, "
              f"delays up to {delays.max() * 1e6:.3f} us", flush=True)
    from fenicsx_fus_gpu_b200 import sampling

    x_p = np.linspace(0.0, lengths[0], 121)
    z_p = np.linspace(0.0, lengths[2], 121)
    X_p, Z_p = np.meshgrid(x_p, z_p)
    points = np.zeros((3, X_p.size))
    points[0], points[1], points[2] = X_p.ravel(), focus[1], Z_p.ravel()
    x_eval, cell_eval = sampling.compute_eval_params(su.mesh, points, dtype)
    ev = sampling.PointEvaluator(a.degree, dtype, su.dev["dofmap"], su.mesh, x_eval, cell_eval, su.tables.pts_1d)

    sampler = _common.PlaneSampler(ev, x_eval[:, [0, 2]], (nsteps - period - 0.5) * dt, period, a.sample_dir, rank)
    _common.run(solver, 0.0, dt, nsteps, rank, sampler=sampler)
    peak = np.zeros(ev.npts) if sampler.values is None else np.abs(sampler.values).max(axis=0, initial=0.0)
    # the peak beyond one wavelength from the array (the elements' own near field is excluded)
    far = x_eval[:, 2] > c0 / f0
    best = (-1.0, 0.0, 0.0)
    if far.any():
        i = int(np.argmax(np.where(far, peak, -1.0)))
        best = (float(peak[i]), float(x_eval[i, 0]), float(x_eval[i, 2]))
    if world > 1:
        import torch.distributed as dist

        everyone = [None] * world
        dist.all_gather_object(everyone, best)
        best = max(everyone)
    if rank == 0:
        d = np.hypot(best[1] - focus[0], best[2] - focus[2])
        print(f"peak |p| over the last period in the plane y = {focus[1] * 1e3:.2f} mm: {best[0]:.6g} at "
              f"x = {best[1] * 1e3:.2f} mm, z = {best[2] * 1e3:.2f} mm; requested focus x = {focus[0] * 1e3:.2f} mm, "
              f"z = {focus[2] * 1e3:.2f} mm; distance {d * 1e3:.2f} mm", flush=True)
    _common.finish(world)


if __name__ == "__main__":
    main()
