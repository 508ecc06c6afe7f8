"""Developer tool: the cost of a point recorder (``solver.record_points``) on one GPU.

    python tools/record_points_bench.py [--P 4] [--N 80] [--steps 20] [--repeats 3]
                                        [--out profiles/r04_record_points.jsonl]

The linear RK4 piston problem of ``demos/demo_linear_piston.py`` on an N^3 box of degree P (the
demo's cell size).  For each float type (f64, f32) and point set - the demo's 141 x 241 sampling
plane through the piston axis (34 k points) and a 100^3 grid filling the box (1 M points) - it
writes one JSON line with

* ``ms_per_step`` / ``ms_per_step_plain``: graph-replayed steps of a solver with the recorder and
  of an identical solver without one, CUDA events around ``--steps`` steps, alternated in pairs
  ``--repeats`` times in the same process (the order inside a pair alternates too);
* ``record_us``: the time of one record launch, from CUDA events around every record launch of
  eager steps;
* ``ms_per_step_stepwise``: the step-by-step path over the same number of steps, ``rk4(..., 1)``
  then ``PointEvaluator.to_host`` per step, host clock (every step ends in a synchronise);
* ``npts``: the points kept (those whose pull-back to their cell converges to ``PointEvaluator``'s
  tolerance);
* the recorded rows are checked against ``PointEvaluator`` on the final state (``last_row_equal``);
* the GPU's name and power limit.
"""

import argparse
import gc
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fenicsx_fus_gpu_b200 import problem, sampling  # noqa: E402
from vertex_solver_bench import gpu_info  # noqa: E402


def steps_ms(s, dt, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.rk4(s.t, dt, steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def record_us(s, dt, steps):
    """Mean time of one record launch in eager steps (events around each launch)."""
    events = []
    launch = s._record

    def timed(*args):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch(*args)
        e1.record()
        events.append((e0, e1))

    s.use_graph = False
    s._record = timed
    s.rk4(s.t, dt, steps)
    torch.cuda.synchronize()
    del s._record
    s.use_graph = True
    return 1000.0 * float(np.mean([a.elapsed_time(b) for a, b in events]))


def stepwise_ms(s, ev, dt, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        s.rk4(s.t, dt, 1)
        ev.to_host(s.u)
    return 1000.0 * (time.perf_counter() - t0) / steps


def point_sets(lengths, centre):
    x_p = centre[0] + np.linspace(-0.035, 0.035, 141)
    z_p = np.linspace(0.0, lengths[2], 241)
    X, Z = np.meshgrid(x_p, z_p)
    plane = np.zeros((3, X.size))
    plane[0], plane[1], plane[2] = X.ravel(), centre[1], Z.ravel()
    g = [np.linspace(0.005 * L, 0.995 * L, 100) for L in lengths]
    cube = np.stack([a.ravel() for a in np.meshgrid(*g, indexing="ij")])
    return {"plane": plane, "grid": cube}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--P", type=int, default=4)
    ap.add_argument("--N", type=int, default=80)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--points", default="plane,grid")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_record_points.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("record_points_bench: no CUDA device")
    name, power = gpu_info()
    f0, c0 = 0.5e6, 1500.0
    h = 0.12 / 93
    L = h * a.N
    centre = (0.5 * L, 0.5 * L)
    piston = problem.disc(0, 1, centre, 0.01)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for tag in a.dtypes.split(","):
            dtype = np.float64 if tag == "f64" else np.float32
            su = problem.box_setup(a.P, a.N, L, dtype)
            dt = problem.cfl_time_step(a.P, h, c0, f0, 0.65)
            sets = point_sets((L, L, L), centre)
            for pname in a.points.split(","):
                xp, cells = sampling.compute_eval_params(su.mesh, sets[pname], dtype)
                # keep the points whose pull-back meets PointEvaluator's tolerance (1e-14 of the cell size: the
                # rounding of coordinates 80 cells from the origin can exceed it)
                ok = sampling.pull_back(su.mesh.x_g[su.mesh.x_dofs[np.asarray(cells)]], xp)[1]
                xp, cells = xp[ok], [c for c, k in zip(cells, ok) if k]
                ev = sampling.PointEvaluator(a.P, dtype, su.dev["dofmap"], su.mesh, xp, cells, su.tables.pts_1d)
                gc.collect()
                solvers = [problem.linear_solver(su, [0], [0, 1, 2, 3, 4, 5], f0=f0, c0=c0, source_predicate=piston,
                                                 absorbing_predicate=lambda cen: ~(piston(cen) & (cen[:, 2] < 0.5 * h)))
                           for _ in range(2)]
                plain, rec_s = solvers
                total = 3 + a.repeats * a.steps + 2 + a.steps  # every step of rec_s below lands in the window
                rows = rec_s.record_points(ev, first=0, rows=total + 1)
                for s in solvers:
                    s.init()
                    s.rk4(0.0, dt, 3)  # capture + warm-up
                ms = {id(plain): [], id(rec_s): []}
                for r in range(a.repeats):
                    for s in (solvers if r % 2 == 0 else solvers[::-1]):
                        ms[id(s)].append(round(steps_ms(s, dt, a.steps), 4))
                rus = round(record_us(rec_s, dt, 2), 2)
                # the step-by-step path over the same window, on the solver without a recorder
                sw = round(stepwise_ms(plain, ev, dt, a.steps), 4)
                rec_s.rk4(rec_s.t, dt, a.steps)
                torch.cuda.synchronize()
                last = rows[rec_s.nstep].cpu().numpy()
                rec = dict(gpu=name, power_limit=power, P=a.P, N=a.N, dtype=tag, points=pname, npts=ev.npts,
                           ndofs=su.global_dofs, steps=a.steps,
                           ms_per_step=ms[id(rec_s)], ms_per_step_plain=ms[id(plain)], record_us=rus,
                           ms_per_step_stepwise=sw, rows_bytes=int(rows.nbytes),
                           last_row_equal=bool(last.tobytes() == ev(rec_s.u).cpu().numpy().tobytes()),
                           rows_finite=bool(torch.isfinite(rows[:rec_s.nstep + 1]).all().item()))
                print(json.dumps(rec), flush=True)
                f.write(json.dumps(rec) + "\n")
                del solvers, plain, rec_s, rows, ev
            del su


if __name__ == "__main__":
    main()
