"""Pulse echo - a planar array of na x nb square elements on z = 0 of a water box (linear wave
equation, f = 0.5 MHz) transmits (unfocused, or focused on ``--focus``) and the same array
receives: every step records what each element receives, the integral of p over its facets
(``solver.record_elements``).  The back wall z = L reflects, every other facet off the aperture
absorbs.

The run is made twice, the second time with an absorbing back wall; the echo is the difference of
the two recordings.  The script prints when the echo reaches the centre element (the first step at
which it exceeds 5 % of its peak) beside the round trip 2L/c, and writes the traces of the run with
the reflecting wall (``element_traces.npy``, (steps + 1, E), summed over the ranks) and the echo
(``element_echo.npy``) to ``--sample-dir``."""

import os

import numpy as np

import _common

from fenicsx_fus_gpu_b200 import problem, substrate as S


def main():
    ap = _common.parser(__doc__, degree=4, cells=40)
    ap.add_argument("--length", type=float, default=0.03, help="box edge in metres (one GPU; scaled with the GPU grid)")
    ap.add_argument("--elements", default="8,8", help="NA,NB elements of the array")
    ap.add_argument("--pitch", type=float, default=0.0015, help="element pitch in metres (default: half a wavelength)")
    ap.add_argument("--focus", default=None, help="x,y,z of a focus from the array centre, metres (default: unfocused)")
    ap.add_argument("--periods", type=float, default=5.0, help="periods simulated after the round trip 2L/c")
    a = ap.parse_args()
    rank, world = _common.init()
    import torch

    dtype = np.float64 if a.dtype == "f64" else np.float32
    f0, c0, rho = 0.5e6, 1500.0, 1000.0
    h = a.length / a.cells
    grid = S.block_grid(world)
    ncells = tuple(a.cells * g for g in grid)
    lengths = tuple(h * n for n in ncells)
    su = problem.box_setup(a.degree, ncells, lengths, dtype, rank, world, grid=grid, geometry=a.geometry)
    na, nb = (int(v) for v in a.elements.split(","))
    centre = np.array([0.5 * lengths[0], 0.5 * lengths[1], 0.0])
    pitch = min(a.pitch, 0.9 * min(lengths[0] / na, lengths[1] / nb))  # the aperture stays inside the face
    tile = problem.TileArray(centre, na, nb, pitch)
    delays = np.zeros(tile.E)
    if a.focus is not None:
        delays = problem.focus_delays(tile.centres, centre + np.array([float(v) for v in a.focus.split(",")]), c0)
    aperture = lambda cen: (cen[:, 2] < 0.5 * h) & (tile.element_of(cen) >= 0)  # noqa: E731
    receiver = problem.element_receiver(su, [0], tile)
    dt = problem.cfl_time_step(a.degree, h, c0, f0, 0.65)
    round_trip = 2.0 * lengths[2] / c0
    nsteps = a.steps or int((round_trip + delays.max() + a.periods / f0) / dt) + 1
    if rank == 0:
        print(f"Number of steps: {nsteps} (twice); {su.global_dofs} dofs on {world} GPU(s); {tile.E} elements of "
              f"{pitch * 1e3:.3f} mm", flush=True)
    traces = []
    for back in ("reflecting", "absorbing"):
        faces = [0, 1, 2, 3, 4] + ([5] if back == "absorbing" else [])
        solver = problem.linear_solver(su, source_facets=[0], absorbing_facets=faces, rho=rho, c0=c0, f0=f0,
                                       source_elements=tile, element_delays=delays,
                                       absorbing_predicate=lambda cen: ~aperture(cen), geometry=a.geometry,
                                       integrator=a.integrator)
        rows = solver.record_elements(receiver, first=0, rows=nsteps + 1)
        if rank == 0:
            print(f"back wall {back}:", flush=True)
        _common.run(solver, 0.0, dt, nsteps, rank, report=max(nsteps // 4, 1))
        if world > 1:
            import torch.distributed as dist

            dist.all_reduce(rows)  # each rank holds its part of every element's integral
        traces.append(rows.cpu().numpy().astype(np.float64))
        del solver
    echo = traces[0] - traces[1]
    c = int(tile.element_of(centre[None])[0])
    t = np.arange(nsteps + 1) * dt
    peak = np.abs(echo[:, c]).max()
    onset = float(t[np.argmax(np.abs(echo[:, c]) > 0.05 * peak)]) if peak > 0 else float("nan")
    if rank == 0:
        print(f"element areas: {receiver.areas.sum().item() * 1e6:.4f} mm^2 on rank 0 of {world}", flush=True)
        print(f"echo at the centre element {c}: onset {onset * 1e6:.3f} us (first step above 5 % of its peak "
              f"{peak:.6g} Pa m^2); round trip 2L/c = {round_trip * 1e6:.3f} us, plus the waveform's 4-period ramp "
              f"{4e6 / f0:.1f} us; delay of that element {delays[c] * 1e6:.3f} us", flush=True)
        if a.sample_dir:
            os.makedirs(a.sample_dir, exist_ok=True)
            np.save(os.path.join(a.sample_dir, "element_traces.npy"), traces[0])
            np.save(os.path.join(a.sample_dir, "element_echo.npy"), echo)
    torch.cuda.synchronize()
    _common.finish(world)


if __name__ == "__main__":
    main()
