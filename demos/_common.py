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
                    help="time integrator of the linear demos: rk4 (the reference's) or leapfrog")
    ap.add_argument("--sample-dir", default=None,
                    help="write pressure_field_<k>.txt dumps of the sampling plane here (device-side sampling)")
    return ap


class PlaneSampler:
    """The reference's "Collect data" block (cuda/demo_linear_piston.py:555-582): once
    ``t > t_from``, every step for ``ndumps`` steps, the field on the sampling points goes
    to ``pressure_field_<k>.txt`` as rows ``x, z, p``.  The reference copies the whole
    vector to the host and evaluates there; here one kernel samples on the device and only
    the sampled values are copied."""

    def __init__(self, evaluator, coords2, t_from, ndumps, out_dir, rank):
        self.ev, self.t_from, self.ndumps, self.k = evaluator, t_from, ndumps, 0
        self.data = None
        self.dir, self.rank = out_dir, rank
        if evaluator.npts:
            import numpy as np

            self.data = np.zeros((evaluator.npts, 3))
            self.data[:, :2] = coords2
        os.makedirs(out_dir, exist_ok=True)

    def active(self, t):
        return t > self.t_from and self.k < self.ndumps

    def dump(self, solver):
        import numpy as np

        # ghost entries of the solution are made current by the same forward halo the next step
        # starts with - scatter_fwd(u_n_d) in the reference (:566).  Collective: every rank dumps
        # at the same steps.
        if solver.halo is not None:
            solver.halo.forward(solver.u, solver.v)
        if self.data is not None:
            self.data[:, 2] = self.ev.to_host(solver.u)
            with open(os.path.join(self.dir, f"pressure_field_{self.k}_rank{self.rank}.txt"), "a") as f:
                np.savetxt(f, self.data, fmt="%.8f", delimiter=",")
        self.k += 1


def run(solver, t0, dt, nsteps, rank, report=100, sampler=None):
    """The demos' loop: print u[0] every ``report`` steps (cuda/demo_linear_box.py:569-570),
    then "Solve time" / "Solve time per step" (:579-581)."""
    import torch

    solver.init()
    torch.cuda.synchronize()
    t_start = time.perf_counter()
    done = 0
    while done < nsteps:
        k = min(report - done % report, nsteps - done)
        if sampler is not None and sampler.k < sampler.ndumps:
            # stop at the first step of the sampling window, then go step by step through it
            t_next = solver.t if done else t0
            if sampler.active(t_next + dt):
                k = 1
            elif sampler.t_from > t_next:
                k = max(1, min(k, int((sampler.t_from - t_next) / dt)))
        solver.rk4(solver.t if done else t0, dt, k)
        done += k
        if sampler is not None and sampler.active(solver.t):
            sampler.dump(solver)
        if done % report and done < nsteps:
            continue
        u0 = float(solver.u[0])  # device -> host read of one value (synchronises)
        if rank == 0:
            print(f"t: {solver.t:5.5},\t Steps: {done}/{nsteps}, \t u[0] = {u0}", flush=True)
    torch.cuda.synchronize()
    el = time.perf_counter() - t_start
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
