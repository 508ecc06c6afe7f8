"""Developer tool: the cost of a phased-array source on one GPU.

    python tools/phased_array_bench.py [--P 4] [--N 80] [--steps 20] [--repeats 3]
                                       [--out profiles/r03_phased_array.jsonl]

A linear RK4 problem on an N^3 box of degree P, shaped like the piston demo: a square source
aperture of 60 mm on z = 0 (the disc of the piston demo is too small to hold 1024 elements of
at least one facet each), every other facet absorbing.  For each float type (f64, f32) and array
of E = 1, 64, 256, 1024 square elements covering that aperture, it writes one JSON line with

* ``ms_per_step`` / ``ms_per_step_single``: graph-replayed steps of the element solver and of the
  single-source solver on the same mesh and facets, CUDA events around ``--steps`` steps, the two
  alternated ``--repeats`` times in the same process (the lists keep every repeat);
* ``boundary_us`` / ``boundary_us_single``: the in-situ time of one boundary launch, from CUDA
  events the tool puts around every boundary launch of eager steps (``solver.probe`` brackets the
  cell kernels only);
* ``table_bytes``: the device source table (``rows * 8 E * itemsize``, rows >= 256);
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


def boundary_us(s, dt, steps):
    """Mean time of one boundary launch in eager steps (events around each launch)."""
    events = []
    launch = s._boundary

    def timed(*args, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch(*args, **kw)
        e1.record()
        events.append((e0, e1))

    s.use_graph = False
    s._boundary = timed
    s.rk4(s.t, dt, steps)
    torch.cuda.synchronize()
    del s._boundary
    s.use_graph = True
    return 1000.0 * float(np.mean([a.elapsed_time(b) for a, b in events]))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--P", type=int, default=4)
    ap.add_argument("--N", type=int, default=80)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--elements", default="1,64,256,1024")
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_phased_array.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("phased_array_bench: no CUDA device")
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
                on_face = lambda cen: tile.element_of(cen) >= 0  # noqa: E731
                absorbing = lambda cen: ~((cen[:, 2] < 0.5 * su.h) & (tile.element_of(cen) >= 0))  # noqa: E731
                gc.collect()
                single = problem.linear_solver(su, [0], [0, 1, 2, 3, 4, 5], source_predicate=on_face,
                                               absorbing_predicate=absorbing)
                elems = problem.linear_solver(su, [0], [0, 1, 2, 3, 4, 5], source_elements=tile,
                                              absorbing_predicate=absorbing,
                                              element_delays=np.linspace(0.0, 2e-6, E))
                for s in (single, elems):
                    s.init()
                    s.rk4(0.0, dt, 3)  # capture + warm-up
                ms = {id(single): [], id(elems): []}
                for _ in range(a.repeats):
                    for s in (single, elems):
                        ms[id(s)].append(round(steps_ms(s, dt, a.steps), 4))
                bu = {id(s): round(boundary_us(s, dt, 2), 2) for s in (single, elems)}
                nentries = int(elems._erow[-1].item())
                rec = dict(gpu=name, power_limit=power, P=a.P, N=a.N, dtype=tag, E=E, ndofs=su.global_dofs,
                           boundary_dofs=int(elems._bdofs.numel()), element_entries=nentries,
                           elements_with_facets=int(torch.unique(elems._eelem[:nentries]).numel()), steps=a.steps,
                           ms_per_step=ms[id(elems)], ms_per_step_single=ms[id(single)],
                           boundary_us=bu[id(elems)], boundary_us_single=bu[id(single)],
                           table_bytes=int(elems.gtab.nbytes),
                           finite=bool(torch.isfinite(elems.u).all().item()))
                print(json.dumps(rec), flush=True)
                f.write(json.dumps(rec) + "\n")
                del single, elems
            del su


if __name__ == "__main__":
    main()
