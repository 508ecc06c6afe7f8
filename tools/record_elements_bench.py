"""Developer tool: the cost of an element receiver (``solver.record_elements``) on one GPU.

    python tools/record_elements_bench.py [--P 4] [--N 80] [--steps 20] [--repeats 3]
                                          [--out profiles/r05_record_elements.jsonl]

The problem of ``tools/phased_array_bench.py``: a linear RK4 solver on an N^3 box of degree P with a
square 60 mm source aperture on z = 0, every other facet absorbing.  For each float type (f64, f32)
and array of E = 1, 64, 256, 1024 square elements covering that aperture, the same array receives,
and the tool writes one JSON line with

* ``ms_per_step`` / ``ms_per_step_plain``: graph-replayed steps of a solver with the receiver and of
  an identical solver without one, CUDA events around ``--steps`` steps, alternated in pairs
  ``--repeats`` times in the same process (the order inside a pair alternates too);
* ``record_us``: the time of one record launch pair (chunk partials, then element sums), from CUDA
  events around every record of eager steps; ``boundary_us``: the boundary launch of the same
  solver, timed the same way in the same steps;
* ``receiver_bytes``: the receiver's device arrays (rows, chunk tables, scratch) and ``rows_bytes``
  the recording;
* ``entries`` / ``chunks``: the receiver's (element, dof) entries and chunks;
* the recorded last row against ``receiver(u)`` on the final state (``last_row_equal``);
* the GPU's name and power limit.
"""

import argparse
import gc
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fenicsx_fus_gpu_b200 import problem  # noqa: E402
from vertex_solver_bench import gpu_info  # noqa: E402


def steps_ms(s, dt, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.rk4(s.t, dt, steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def launch_us(s, dt, steps, names):
    """Mean time of one call of each solver method in ``names`` in eager steps (events around each)."""
    events = {n: [] for n in names}

    def timed(name, launch):
        def call(*args, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch(*args, **kw)
            e1.record()
            events[name].append((e0, e1))
        return call

    s.use_graph = False
    for n in names:
        setattr(s, n, timed(n, getattr(s, n)))
    s.rk4(s.t, dt, steps)
    torch.cuda.synchronize()
    for n in names:
        delattr(s, n)
    s.use_graph = True
    return {n: round(1000.0 * float(np.mean([a.elapsed_time(b) for a, b in ev])), 2) for n, ev in events.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--P", type=int, default=4)
    ap.add_argument("--N", type=int, default=80)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--elements", default="1,64,256,1024")
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_record_elements.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("record_elements_bench: no CUDA device")
    name, power = gpu_info()
    L = 0.12 / 80 * a.N
    aperture = 0.06 / 0.12 * L
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for tag in a.dtypes.split(","):
            dtype = np.float64 if tag == "f64" else np.float32
            su = problem.box_setup(a.P, a.N, L, dtype, seed=1)
            dt = problem.cfl_time_step(a.P, su.h, 1500.0, 0.5e6, 0.65)
            for E in (int(e) for e in a.elements.split(",")):
                na = int(round(np.sqrt(E)))
                assert na * na == E, "square arrays only"
                tile = problem.TileArray((0.5 * L, 0.5 * L, 0.0), na, na, aperture / na)
                absorbing = lambda cen: ~((cen[:, 2] < 0.5 * su.h) & (tile.element_of(cen) >= 0))  # noqa: E731
                gc.collect()
                solvers = [problem.linear_solver(su, [0], [0, 1, 2, 3, 4, 5], source_elements=tile,
                                                 absorbing_predicate=absorbing,
                                                 element_delays=np.linspace(0.0, 2e-6, E)) for _ in range(2)]
                plain, recv = solvers
                receiver = problem.element_receiver(su, [0], tile)
                total = 3 + a.repeats * a.steps + 2 + a.steps  # every step of recv below lands in the window
                rows = recv.record_elements(receiver, first=0, rows=total + 1)
                for s in solvers:
                    s.init()
                    s.rk4(0.0, dt, 3)  # capture + warm-up
                ms = {id(plain): [], id(recv): []}
                for r in range(a.repeats):
                    for s in (solvers if r % 2 == 0 else solvers[::-1]):
                        ms[id(s)].append(round(steps_ms(s, dt, a.steps), 4))
                us = launch_us(recv, dt, 2, ("_record", "_boundary"))
                recv.rk4(recv.t, dt, a.steps)
                torch.cuda.synchronize()
                last = rows[recv.nstep].cpu().numpy()
                rec = dict(gpu=name, power_limit=power, P=a.P, N=a.N, dtype=tag, E=E, ndofs=su.global_dofs,
                           entries=int(receiver.dof.numel()), chunks=receiver.nchunks, steps=a.steps,
                           ms_per_step=ms[id(recv)], ms_per_step_plain=ms[id(plain)],
                           record_us=us["_record"], boundary_us=us["_boundary"],
                           receiver_bytes=int(receiver.nbytes), rows_bytes=int(rows.nbytes),
                           last_row_equal=bool(last.tobytes() == receiver(recv.u).cpu().numpy().tobytes()),
                           rows_finite=bool(torch.isfinite(rows[:recv.nstep + 1]).all().item()))
                print(json.dumps(rec), flush=True)
                f.write(json.dumps(rec) + "\n")
                del solvers, plain, recv, rows, receiver
            del su


if __name__ == "__main__":
    main()
