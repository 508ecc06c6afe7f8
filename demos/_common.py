"""Shared launcher bits of the demo scripts: one process per GPU under torchrun
(``python -m torch.distributed.run --nproc-per-node N demos/demo_*.py``) or a
plain ``python demos/demo_*.py`` on one GPU."""

import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def init():
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world


def parser(desc, degree, cells):
    ap = argparse.ArgumentParser(description=desc)
    ap.add_argument("--degree", type=int, default=degree)
    ap.add_argument("--cells", type=int, default=cells, help="cells per direction PER GPU (default: the reference demo's mesh)")
    ap.add_argument("--steps", type=int, default=0, help="number of steps (default: run to the demo's final time)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--geometry", default="stream", choices=["stream", "auto", "vertex"],
                    help="auto: affine cells keep 6 geometric factors instead of 6 n^3; vertex: as auto, and the "
                         "other cells rebuild their geometry from 36 values instead of streaming it (no per-point "
                         "tables; same results to rounding)")
    ap.add_argument("--integrator", default="rk4", choices=["rk4", "leapfrog"],
                    help="time integrator: rk4 (the reference's) or leapfrog (one stiffness action per step)")
    ap.add_argument("--sample-dir", default=None,
                    help="write pressure_field_<k>.txt dumps of the sampling plane here (device-side sampling)")
    return ap


class PlaneSampler:
    """The reference's "Collect data" block (cuda/demo_linear_piston.py:555-582): once
    ``t > t_from``, every step for ``ndumps`` steps, the field on the sampling points goes
    to ``pressure_field_<k>.txt`` as rows ``x, z, p``.  The reference copies the whole
    vector to the host and evaluates there; here the solver records the points inside its
    captured steps (``record_points``) and the rows are copied once, after the run.
    ``out_dir=None`` writes no files; ``values`` holds the rows (ndumps', npts) either way."""

    def __init__(self, evaluator, coords2, t_from, ndumps, out_dir, rank):
        self.ev, self.t_from, self.ndumps = evaluator, t_from, ndumps
        self.coords2, self.dir, self.rank = coords2, out_dir, rank
        self.rows = self.values = None
        if out_dir is not None:
            os.makedirs(out_dir, exist_ok=True)

    def attach(self, solver, t0, dt, nsteps):
        """Attach the recorder of the window to ``solver``: from the first step count whose time,
        accumulated as the solver does (``t += dt``), exceeds ``t_from``, ``ndumps`` rows clipped to
        the ``nsteps`` steps of the run.  Every rank attaches the same window."""
        t, first = t0, 0
        while first < nsteps:
            t += dt
            first += 1
            if t > self.t_from:
                break
        rows = min(self.ndumps, nsteps - first + 1) if t > self.t_from else 0
        self.rows = solver.record_points(self.ev, first, rows) if rows > 0 else None

    def collect(self):
        """After the run: the recorded rows to the host, one file per row."""
        import numpy as np

        if self.rows is None:
            return
        self.values = self.rows.cpu().numpy()
        if self.dir is None or not self.ev.npts:
            return
        data = np.zeros((self.ev.npts, 3))
        data[:, :2] = self.coords2
        for k, row in enumerate(self.values):
            data[:, 2] = row
            with open(os.path.join(self.dir, f"pressure_field_{k}_rank{self.rank}.txt"), "a") as f:
                np.savetxt(f, data, fmt="%.8f", delimiter=",")


def run(solver, t0, dt, nsteps, rank, report=100, sampler=None):
    """The demos' loop: print u[0] every ``report`` steps (cuda/demo_linear_box.py:569-570),
    then "Solve time" / "Solve time per step" (:579-581)."""
    import torch

    solver.init()
    if sampler is not None:
        sampler.attach(solver, t0, dt, nsteps)
    torch.cuda.synchronize()
    t_start = time.perf_counter()
    done = 0
    while done < nsteps:
        k = min(report - done % report, nsteps - done)
        solver.rk4(solver.t if done else t0, dt, k)
        done += k
        u0 = float(solver.u[0])  # device -> host read of one value (synchronises)
        if rank == 0:
            print(f"t: {solver.t:5.5},\t Steps: {done}/{nsteps}, \t u[0] = {u0}", flush=True)
    torch.cuda.synchronize()
    el = time.perf_counter() - t_start
    if sampler is not None:
        sampler.collect()
    if rank == 0:
        print(f"Solve time: {el}")
        print(f"Solve time per step: {el / max(1, nsteps)}")
    return el


def finish(world):
    if world > 1:
        import torch
        import torch.distributed as dist

        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)
