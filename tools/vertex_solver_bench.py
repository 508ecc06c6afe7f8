"""Developer tool: the time loops in the three geometry modes, on one GPU.

    python tools/vertex_solver_bench.py [--P 4] [--N 80] [--steps 20] [--out profiles/r03_vertex_solver.jsonl]

For each float type (f64, f32), mesh (a perturbed box: every cell trilinear; an unperturbed box:
every cell rectilinear, so "vertex" must equal "auto"), geometry ("stream", "auto", "vertex") and
solver (linear RK4, leapfrog, Westervelt pointwise and cells) it writes one JSON line:

* ``ms_per_step``: graph-replayed steps, CUDA events around ``--steps`` steps after 3 warm-up steps;
* ``stage_kernel_ms``: the mean in-situ time of one cell-kernel group of a stage (``solver.probe``,
  eager steps);
* ``peak_bytes`` / ``bytes_per_dof``: ``torch.cuda.max_memory_allocated`` from before the set-up
  (``problem.box_setup``) to the end of the solver's construction.

The GPU's name and power limit go into every line.
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

SOLVERS = [("linear", "rk4", None), ("linear", "leapfrog", None), ("westervelt", "rk4", "pointwise"),
           ("westervelt", "rk4", "cells")]


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        power = r.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception:
        power = "unknown"
    return name, power


def build(su, kind, integrator, mass_form, geometry, L):
    if kind == "linear":
        return problem.linear_solver(su, (2,), (3,), integrator=integrator, geometry=geometry)
    return problem.westervelt_solver(su, (2,), (0, 1, 3, 4, 5), geometry=geometry, mass_form=mass_form)


def run_one(s, dt, steps):
    s.init()
    s.rk4(0.0, dt, 3)  # capture + warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.rk4(s.t, dt, steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    # in-situ stage kernels: eager steps with events around every cell-kernel group
    s.use_graph = False
    s.rk4(s.t, dt, 1)
    s.probe = []
    s.rk4(s.t, dt, 3)
    torch.cuda.synchronize()
    probe = float(np.mean([a.elapsed_time(b) for a, b in s.probe]))
    s.probe = None
    s.use_graph = True
    return ms, probe, bool(torch.isfinite(s.u).all().item())


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--P", type=int, default=4)
    ap.add_argument("--N", type=int, default=80)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_vertex_solver.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vertex_solver_bench: no CUDA device")
    name, power = gpu_info()
    L = 0.12 / 80 * a.N
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for tag in a.dtypes.split(","):
            dtype = np.float64 if tag == "f64" else np.float32
            for mesh, perturb in (("perturbed", 0.1), ("box", 0.0)):
                for geometry in ("stream", "auto", "vertex"):
                    gc.collect()
                    torch.cuda.synchronize()
                    base = torch.cuda.memory_allocated()
                    torch.cuda.reset_peak_memory_stats()
                    su = problem.box_setup(a.P, a.N, L, dtype, perturb=perturb, seed=1, geometry=geometry)
                    setup_bytes = torch.cuda.memory_allocated() - base
                    for kind, integrator, mass_form in SOLVERS:
                        gc.collect()
                        if kind != SOLVERS[0][0] or integrator != "rk4":
                            torch.cuda.reset_peak_memory_stats()  # the set-up's own peak was counted first
                        s = build(su, kind, integrator, mass_form, geometry, L)
                        torch.cuda.synchronize()
                        peak = torch.cuda.max_memory_allocated() - base
                        c0 = 1480.0 if kind == "westervelt" else 1500.0
                        f0 = 1.1e6 if kind == "westervelt" else 0.5e6
                        dt = problem.cfl_time_step(a.P, su.h, c0, f0, 0.4 if kind == "westervelt" else 0.65)
                        ms, probe, finite = run_one(s, dt, a.steps)
                        rec = dict(gpu=name, power_limit=power, P=a.P, N=a.N, dtype=tag, mesh=mesh, geometry=geometry,
                                   solver=kind, integrator=integrator, mass_form=mass_form, ndofs=su.global_dofs,
                                   nrect=s.nrect, naff=s.naff, ntri=s.ntri, steps=a.steps, ms_per_step=round(ms, 4),
                                   stage_kernel_ms=round(probe, 4), setup_bytes=setup_bytes, peak_bytes=peak,
                                   bytes_per_dof=round(peak / su.global_dofs, 2), finite=finite)
                        print(json.dumps(rec), flush=True)
                        f.write(json.dumps(rec) + "\n")
                        del s
                    del su


if __name__ == "__main__":
    main()
