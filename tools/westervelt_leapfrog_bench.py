"""Developer tool: the Westervelt time loops, RK4 against leapfrog, on one GPU.

    python tools/westervelt_leapfrog_bench.py [--out profiles/r06_westervelt_leapfrog.jsonl]

Workloads (degree 4, pointwise mass form, geometry "stream", c = 1480 m/s, f = 1.1 MHz, beta = 3.5,
the dt of the demos at CFL 0.4):

* ``box``: 80^3 cells of h = 0.12/80 m, source on the whole face x = 0, every other face absorbing,
  p0 = 1 MPa, alpha = 20 dB;
* ``bowl``: the single-GPU part of demos/demo_nonlinear_bowl.py: 99^3 cells of h = 0.08/198 m, a
  disc source of radius 0.3 L on x = 0, every face absorbing, the demo's p0 and alpha = 0.2 dB.

For each workload and float type both solvers are built side by side, and per integrator the tool
writes one JSON line:

* accuracy: both run ``--sim-steps`` steps from rest (default: the time the wave takes to cross half
  the box plus 8 periods, so the focus sees the steady wave) and record the pressure at the "focus"
  (the point on the source axis at x = L/2) every step:
  ``peak_focus_pa`` is its largest |p|, ``rel_l2_vs_rk4`` the rel-L2 difference of the leapfrog ``u``
  against the RK4 ``u`` at the same simulated time, ``finite`` whether every value stayed finite;
* ``ms_per_step``: graph-replayed steps, CUDA events around ``--steps`` steps, RK4 and leapfrog
  alternated ``--rounds`` times in this process (one value per round);
* ``stage_kernel_ms``: the mean in-situ time of one cell-kernel group (``solver.probe``, eager
  steps): one per RK4 stage, one per leapfrog step;
* ``sim_us_per_wall_s``: simulated microseconds per wall-clock second at the median step time.

When the leapfrog run is not finite at CFL 0.4, it is repeated at lower CFL numbers and the largest
one that stays finite is recorded.  The GPU's name and power limit go into every line.
"""

import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fenicsx_fus_gpu_b200 import problem  # noqa: E402
from fenicsx_fus_gpu_b200 import sampling as sp  # noqa: E402

C0, RHO, F0, P = 1480.0, 1000.0, 1.1e6, 4
WORKLOADS = {
    "box": dict(n=80, h=0.12 / 80, p0=1.0e6, alpha_dB=20.0),
    "bowl": dict(n=99, h=0.08 / 198, p0=RHO * C0 * 0.38557513826589934, alpha_dB=0.2),
}


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        power = r.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception:
        power = "unknown"
    return name, power


def build(su, name, W, integrator):
    L = su.h * W["n"]
    kw = dict(rho=RHO, c0=C0, f0=F0, p0=W["p0"], beta=3.5, alpha_dB=W["alpha_dB"], integrator=integrator)
    if name == "bowl":
        return problem.westervelt_solver(su, [2], [0, 1, 2, 3, 4, 5],
                                         source_predicate=problem.disc(1, 2, (0.5 * L, 0.5 * L), 0.3 * L), **kw)
    return problem.westervelt_solver(su, [2], [0, 1, 3, 4, 5], **kw)


def focus(su, n):
    L = su.h * n
    xp, cells = sp.compute_eval_params(su.mesh, np.array([[0.5 * L], [0.5 * L + 1e-3 * su.h], [0.5 * L + 1e-3 * su.h]]),
                                       su.dtype)
    assert len(cells) == 1
    return sp.PointEvaluator(su.P, su.dtype, su.dev["dofmap"], su.mesh, xp, cells, su.tables.pts_1d)


def accuracy(s, ev, dt, nsteps):
    rows = s.record_points(ev, 0, nsteps + 1)
    s.init()
    s.rk4(0.0, dt, nsteps)
    torch.cuda.synchronize()
    s.record_points(None)
    finite = bool(torch.isfinite(s.u).all().item()) and bool(torch.isfinite(rows).all().item())
    return finite, float(rows.abs().max().item()) if finite else float("nan")


def time_steps(s, dt, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.rk4(s.t, dt, steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def stage_kernel(s, dt):
    s.use_graph = False
    s.rk4(s.t, dt, 1)
    s.probe = []
    s.rk4(s.t, dt, 3)
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in s.probe]))
    s.probe = None
    s.use_graph = True
    return ms


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", default="box,bowl")
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sim-steps", type=int, default=0, help="steps of the accuracy runs (default: half a box crossing + 8 periods)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_westervelt_leapfrog.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("westervelt_leapfrog_bench: no CUDA device")
    gpu, power = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for name in a.workloads.split(","):
            W = WORKLOADS[name]
            for tag in a.dtypes.split(","):
                dtype = np.float64 if tag == "f64" else np.float32
                gc.collect()
                torch.cuda.empty_cache()
                su = problem.box_setup(P, W["n"], W["h"] * W["n"], dtype)
                ev = focus(su, W["n"])
                solvers = {i: build(su, name, W, i) for i in ("rk4", "leapfrog")}
                cfl = 0.4
                dt = problem.cfl_time_step(P, su.h, C0, F0, cfl)
                nsim = a.sim_steps or int((0.5 * su.h * W["n"] / C0 + 8.0 / F0) / dt) + 1
                acc = {i: accuracy(s, ev, dt, nsim) for i, s in solvers.items()}
                u_rk = solvers["rk4"].u.clone()
                rel = float(((solvers["leapfrog"].u - u_rk).norm() / u_rk.norm()).item())
                stable_cfl = cfl
                while not acc["leapfrog"][0] and stable_cfl > 0.05:  # record the largest CFL that stays finite
                    stable_cfl = round(stable_cfl - 0.05, 2)
                    dts = problem.cfl_time_step(P, su.h, C0, F0, stable_cfl)
                    acc["leapfrog"] = accuracy(solvers["leapfrog"], ev, dts, int(nsim * dt / dts) + 1)
                    rel = float("nan")
                del u_rk
                ms = {i: [] for i in solvers}
                for i, s in solvers.items():  # start the timed windows from a running state, graphs captured
                    s.init()
                    s.rk4(0.0, dt, 3)
                for _ in range(a.rounds):
                    for i, s in solvers.items():
                        ms[i].append(round(time_steps(s, dt, a.steps), 4))
                for i, s in solvers.items():
                    med = float(np.median(ms[i]))
                    rec = dict(gpu=gpu, power_limit=power, workload=name, P=P, cells=W["n"], dtype=tag,
                               ndofs=su.global_dofs, integrator=i, cfl=cfl, dt=dt, steps=a.steps, rounds=a.rounds,
                               ms_per_step=ms[i], ms_per_step_median=round(med, 4),
                               stage_kernel_ms=round(stage_kernel(s, dt), 4),
                               sim_us_per_wall_s=round(dt * 1e6 / (med * 1e-3), 2),
                               stage_bytes=int(s.stage_bytes()), sim_steps=nsim, sim_time_us=round(nsim * dt * 1e6, 3),
                               peak_focus_pa=acc[i][1], finite=acc[i][0],
                               rel_l2_vs_rk4=(rel if i == "leapfrog" else 0.0),
                               largest_stable_cfl=(stable_cfl if i == "leapfrog" else None))
                    print(json.dumps(rec), flush=True)
                    f.write(json.dumps(rec) + "\n")
                del solvers, su, ev


if __name__ == "__main__":
    main()
