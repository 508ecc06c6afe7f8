#!/usr/bin/env python
"""bench.py - the headline benchmark of the hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], "demo_linear_box"): linear acoustic wave,
explicit RK4, degree-4 hexahedra, 80^3 cells = 33 076 161 dofs per GPU, float64,
source facets on x=0 and absorbing facets on x=L (cuda/demo_linear_box.py:53-122,
256-263).  A *step* is one RK4 time step = 4 fused stages.  With N > 1 the box is
block-partitioned, every GPU keeps an 80^3 block (weak scaling) and the ghost
dofs are exchanged over NCCL each stage.

The JSON line: ``value`` = fused-RK-stage throughput in GDoF/s (global dofs x 4
stages x K / time, K graph-replayed steps, state resident in HBM), the metric
BASELINE.json names ("operator GDoF/s and RK time-steps/s"); ``steps_per_s`` and the
stand-alone operator GDoF/s ride along.  ``e2e`` = the same steps with, per step, the
H2D copy of the step's source amplitudes from pinned memory and the D2H read of a
sampled pressure plane; ``e2e_operator_host_buffers`` = one stiffness action through
the C ABI with x and y in pinned HOST memory.  ``roofline`` = the dominant kernel (the
stiffness kernel; the dual-stiffness stage kernel for the Westervelt workload):
algorithmic bytes (SURVEY.md 8d) / its mean duration inside the RK steps (CUDA events
around each launch), against the measured HBM peak, with the stand-alone back-to-back
figure beside it.  ``stage_roofline`` = the whole fused stage on the bytes it moves.
``affine_geometry`` = the same steps with ``geometry="auto"`` (cells with a constant
Jacobian keep 6 geometric factors; extra, not the headline; ``--geometry auto`` makes it
the measured path and says so in ``config``).  ``cpu_baseline`` is the reference's CPU
path (its own C++ sum-factorisation templates when oracle/_ref is built, else the C
port) timed on this host's cores on a bounded sample of the same workload.
``--workload linear_piston|nonlinear_bowl`` time BASELINE.json's other demo configs.
``--dump-outputs DIR`` writes the state the K timed steps leave behind, so that two builds
run with the same arguments (hence the same inputs) can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# workload constants: cuda/demo_linear_box.py:53-66, 116
P = 4
F0, P0, C0, RHO = 0.5e6, 60000.0, 1500.0, 1000.0
DOMAIN_LENGTH = 0.12
N_PER_GPU = 80  # int(2 * 0.12 / (1500 / 0.5e6)) = 80 cells per direction
CFL = 0.65


def peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cfl_dt(h):
    dt = CFL * h / (C0 * P**2)
    period = 1.0 / F0
    return period / (int(period / dt) + 1)


# --------------------------------------------------------------------------- #
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------- #


class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_id):
        """``gpu_id``: anything ``nvidia-smi --id`` takes - the GPU's UUID (robust under torchrun,
        whatever CUDA_VISIBLE_DEVICES says) or its index."""
        self.index, self.proc, self.lines = gpu_id, None, []

    def start(self, wait_first=8.0):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None
            return
        t0 = time.time()
        while not self.lines and time.time() - t0 < wait_first:  # the first sample can take seconds on a busy 8-GPU box
            time.sleep(0.05)

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        rows = [ln for ts, ln in self.lines if t0 <= ts <= t1 + 0.05] or [ln for _, ln in self.lines]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for nme, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- #
# problem set-up (device-side geometry; host substrate for mesh / dofmap)
# --------------------------------------------------------------------------- #


WORKLOADS = {
    # name: degree, c0, rho, f0, reference cell size h, CFL, BASELINE.json config it stands for
    "linear_box": dict(P=4, c0=1500.0, rho=1000.0, f0=0.5e6, h=0.12 / 80, cfl=0.65, n=80, nonlinear=False,
                       label="demo_linear_box: linear wave, RK4 (BASELINE.json configs[1])"),
    # cuda/demo_linear_piston.py:53-66: degree 5, piston of radius 10 mm on z=0, every other exterior facet absorbing
    "linear_piston": dict(P=5, c0=1500.0, rho=1000.0, f0=0.5e6, h=0.12 / 93, cfl=0.65, n=58, nonlinear=False,
                          label="demo_linear_piston: planar piston + absorbing facets, RK4 (BASELINE.json configs[2])"),
    # cuda/demo_nonlinear_bowl.py:61-75,122: Westervelt, c=1480, f=1.1 MHz, beta=3.5, alpha=0.2 dB, CFL 0.4
    "nonlinear_bowl": dict(P=4, c0=1480.0, rho=1000.0, f0=1.1e6, h=0.08 / 198, cfl=0.4, n=99, nonlinear=True,
                           label="demo_nonlinear_bowl: Westervelt, source disc + all facets absorbing, RK4 "
                                 "(BASELINE.json configs[3])"),
}


def build_problem(rank, world, n_per_gpu, dtype, halo_kind, workload="linear_box", degree=None, geometry="stream",
                  split_cells=True, integrator="rk4", rank_grid=None, renumber_shared=True):
    """The demo's preamble through fenicsx_fus_gpu_b200.problem (device geometry,
    block partition, halo).  Returns the solver and an info dict."""
    from fenicsx_fus_gpu_b200 import problem
    from fenicsx_fus_gpu_b200 import substrate as S

    W = WORKLOADS[workload]
    deg = degree or W["P"]
    grid = tuple(rank_grid) if rank_grid else S.block_grid(world)
    ncells = tuple(n_per_gpu * g for g in grid)
    h = W["h"]  # the demo's cell size; the box grows with the rank grid
    lengths = tuple(h * n for n in ncells)
    used = halo_kind if world > 1 else "none"
    try:
        su = problem.box_setup(deg, ncells, lengths, dtype, rank, world, grid=grid, halo_kind=halo_kind,
                               renumber_shared=renumber_shared)
    except Exception as e:  # peer memory unavailable on this box: NCCL send/recv round instead
        if halo_kind != "p2p" or world == 1:
            raise
        print(f"[bench] peer-memory halo unavailable ({e!r}); using the NCCL halo", file=sys.stderr, flush=True)
        used = "nccl"
        su = problem.box_setup(deg, ncells, lengths, dtype, rank, world, grid=grid, halo_kind="nccl",
                               renumber_shared=renumber_shared)

    def make_solver(geometry="stream"):
        if workload == "linear_box":
            return problem.linear_solver(su, source_facets=[2], absorbing_facets=[3], rho=W["rho"], c0=W["c0"],
                                         f0=W["f0"], p0=P0, geometry=geometry, split_cells=split_cells,
                                         integrator=integrator)
        if workload == "linear_piston":
            piston = problem.disc(0, 1, (0.5 * lengths[0], 0.5 * lengths[1]), 0.01)
            return problem.linear_solver(
                su, source_facets=[0], absorbing_facets=[0, 1, 2, 3, 4, 5], rho=W["rho"], c0=W["c0"], f0=W["f0"],
                p0=P0, source_predicate=piston, geometry=geometry, split_cells=split_cells, integrator=integrator,
                absorbing_predicate=lambda cen: ~(piston(cen) & (cen[:, 2] < 0.5 * h)))
        centre = (0.5 * lengths[1], 0.5 * lengths[2])
        return problem.westervelt_solver(
            su, source_facets=[2], absorbing_facets=[0, 1, 2, 3, 4, 5], rho=W["rho"], c0=W["c0"], f0=W["f0"],
            beta=3.5, alpha_dB=0.2, source_predicate=problem.disc(1, 2, centre, 0.3 * lengths[1]), geometry=geometry,
            split_cells=split_cells)

    solver = make_solver(geometry)
    info = dict(rank_grid=list(grid), make_solver=make_solver, ncells_local=su.mesh.num_cells, ndofs_local=su.ndofs, nlocal=su.nlocal, global_cells=ncells,
                global_dofs=su.global_dofs, grid=grid, h=h, detJ=su.dev["detJ"], tb=su.tables,
                dofmap=su.dev["dofmap"], halo=used, degree=deg,
                dt=problem.cfl_time_step(deg, h, W["c0"], W["f0"], W["cfl"]))
    return solver, info


# --------------------------------------------------------------------------- #
# baseline arms: the reference's own code on this box
# --------------------------------------------------------------------------- #


def time_cpu(steps, warmup, n, degree, dtype, kind=None):
    """The reference's CPU path (baseline/cpu_arm.py): the WHOLE n^3-cell box of the workload,
    split over one process per host core, stepped ``steps`` times with the reference's own
    numba-cpu operators (``kind`` "cpp": its C++ templates; "port": the oracle C port)."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import cpu_arm

    return cpu_arm.run(n=n, P=degree, dtype="float64" if dtype == "f64" else "float32", steps=steps,
                       warmup=warmup, kind=kind)


def reference_cuda_arm(n, degree, dtype, reps=10):
    """The reference's own Numba-CUDA kernels (cuda/operators.py:18-192, shipped unmodified as
    baseline/_ref/cuda/operators.py) on THIS GPU, launched with the reference's launch shapes and
    timed with its protocol (cuda/time_operators.py:204-222, 272-290: one warm-up, 10 launches each
    bracketed by perf_counter_ns + cuda.synchronize), beside this repo's kernels on the same arrays
    with the same protocol.  If Numba cannot JIT for this GPU the error text is the result."""
    import torch

    from fenicsx_fus_gpu_b200 import operators as ops
    from fenicsx_fus_gpu_b200 import problem

    np_t = np.float64 if dtype == "f64" else np.float32
    su = problem.box_setup(degree, n, 0.12 / 80 * n, np_t)
    nc, nd, nn = su.mesh.num_cells, su.ndofs, degree + 1
    G, detJ, dm = su.dev["G"], su.dev["detJ"], su.dev["dofmap"]
    D = torch.from_numpy(su.tables.dphi_1D).cuda()
    c = torch.ones(nc, dtype=G.dtype, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(nd, dtype=G.dtype, device="cuda", generator=gen)
    y = torch.zeros(nd, dtype=G.dtype, device="cuda")
    out = {"workload": f"mass + stiffness action, degree {degree}, {n}^3 cells, {nd} dofs, {dtype}",
           "protocol": "1 warm-up + 10 launches, perf_counter_ns around launch + device synchronise, "
                       "output zero-filled outside the timed region (cuda/time_operators.py:204-222, 272-290)"}

    def timed(launch):
        y.zero_()
        launch()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            y.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter_ns()
            launch()
            torch.cuda.synchronize()
            ts.append((time.perf_counter_ns() - t0) * 1e-9)
        return float(np.mean(ts)), float(np.min(ts))

    K = ops.stiffness_operator(degree, np_t)
    t_k, t_k_min = timed(lambda: K[nc, (nn, nn, nn)](x, c, y, G, dm, D))
    y_ours = y.clone()
    t_m, t_m_min = timed(lambda: ops.mass_operator[1, 128](x, c, y, detJ, dm))
    m_ours = y.clone()
    out["ours"] = {"stiffness_gdofs": nd / t_k / 1e9, "stiffness_ms": t_k * 1e3, "stiffness_ms_min": t_k_min * 1e3,
                   "mass_gdofs": nd / t_m / 1e9, "mass_ms": t_m * 1e3, "mass_ms_min": t_m_min * 1e3}
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref", "cuda"))
        import numba.cuda as ncuda

        if "operators" in sys.modules:
            del sys.modules["operators"]
        import operators as ref_ops  # the reference's cuda/operators.py, unmodified

        ncuda.select_device(torch.cuda.current_device())
        arr = lambda t: ncuda.as_cuda_array(t)  # noqa: E731  zero-copy views of the same device arrays
        xd, yd, cd, Gd, Jd, dmd, Dd = (arr(t) for t in (x, y, c, G, detJ, dm, D))
        stiff = ref_ops.stiffness_operator(degree, np_t)
        t_k, t_k_min = timed(lambda: stiff[nc, (nn, nn, nn)](xd, cd, yd, Gd, dmd, Dd))
        e_k = float((y - y_ours).norm() / y_ours.norm())
        nb = (dm.numel() + 127) // 128
        t_m, t_m_min = timed(lambda: ref_ops.mass_operator[nb, 128](xd, cd, yd, Jd, dmd))
        e_m = float((y - m_ours).norm() / m_ours.norm())
        out["reference_numba_cuda"] = {
            "stiffness_gdofs": nd / t_k / 1e9, "stiffness_ms": t_k * 1e3, "stiffness_ms_min": t_k_min * 1e3,
            "mass_gdofs": nd / t_m / 1e9, "mass_ms": t_m * 1e3, "mass_ms_min": t_m_min * 1e3,
            "launch": f"stiffness[{nc}, ({nn},{nn},{nn})], mass[{nb}, 128]",
            "rel_l2_ours_vs_reference": {"stiffness": e_k, "mass": e_m}}
        out["speedup"] = {"stiffness": out["ours"]["stiffness_gdofs"] / out["reference_numba_cuda"]["stiffness_gdofs"],
                          "mass": out["ours"]["mass_gdofs"] / out["reference_numba_cuda"]["mass_gdofs"]}
    except Exception as e:  # Numba cannot drive this GPU / toolkit: the error text is the record
        out["reference_numba_cuda"] = {"unavailable": f"{type(e).__name__}: {e}"[:600]}
    return out


# --------------------------------------------------------------------------- #
# outputs of the timed path, for comparing two builds
# --------------------------------------------------------------------------- #

DUMP_BYTES = 32 << 20  # every rank's arrays together: within 64 MB with the .npy headers
DUMP_SEED = 20261020


def dump_indices(n, itemsize, narrays, rank=0, world=1):
    """Sorted indices of the first ``n`` entries that one of ``world`` ranks writes for each of its
    ``narrays`` arrays of ``itemsize``-byte floats, so that all ranks together write at most
    DUMP_BYTES.  All ``n`` when they fit the rank's share; else the share split into k equal
    strata of [0, n) with one index drawn in each, seeded by DUMP_SEED and the rank: the same
    indices for every run with the same arguments, at O(k) cost."""
    k = DUMP_BYTES // (world * narrays * itemsize)
    if n <= k:
        return np.arange(n, dtype=np.int64)
    edges = np.arange(k + 1, dtype=np.int64) * n // k
    rng = np.random.default_rng([DUMP_SEED, rank])
    return edges[:-1] + (rng.random(k) * np.diff(edges)).astype(np.int64)


def dump_outputs(out_dir, arrays, rank=0, world=1):
    """Write each tensor of ``arrays`` to ``out_dir/<name>.npy`` (``<name>_rank<r>.npy`` with
    several ranks) in its own float type."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{'' if world == 1 else f'_rank{rank}'}.npy"), t.cpu().numpy())


# --------------------------------------------------------------------------- #
# main
# --------------------------------------------------------------------------- #


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--n-per-gpu", type=int, default=0, help="cells per direction per GPU (default: the workload's)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--workload", default="linear_box", choices=sorted(WORKLOADS),
                    help="which reference demo to time (default: the headline demo_linear_box)")
    ap.add_argument("--degree", type=int, default=0, help="override the workload's polynomial degree (2..7)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-affine", action="store_true", help="skip the extra affine-geometry measurement")
    ap.add_argument("--no-extras", action="store_true", help="only the timed region + roofline (sweeps)")
    ap.add_argument("--geometry", default="stream", choices=["stream", "auto"],
                    help="stream (default, the reference's data flow: G read in full every stage) or auto "
                         "(cells with a constant Jacobian keep 6 factors; the JSON line says so in config)")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU halo: fused put/get kernels over NVLink peer memory, or NCCL send/recv")
    ap.add_argument("--no-split", action="store_true", help="p2p halo without the interior/interface cell split (A/B)")
    ap.add_argument("--split-mode", default="none", choices=["none", "two", "fused"],
                    help="p2p halo: wait, then all cells in one launch (default); interface cells in a second launch; "
                         "or in the same launch behind an in-kernel wait (A/B, see solver.py)")
    ap.add_argument("--integrator", default="rk4", choices=["rk4", "leapfrog"],
                    help="rk4 (the reference's scheme, the headline) or leapfrog (one stiffness action per step)")
    ap.add_argument("--rank-grid", default=None, help="AxBxC rank grid instead of the most cubic one (A/B runs)")
    ap.add_argument("--no-renumber", action="store_true",
                    help="keep the index map's numbering instead of moving the shared owned dofs to a contiguous tail (A/B)")
    ap.add_argument("--no-graph", action="store_true", help="launch the steps eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cpu-kind", default=None, choices=["numba", "cpp", "port"], help="CPU arm implementation")
    ap.add_argument("--sustain-steps", type=int, default=250, help="steps of the extra >= 1 s sustained measurement")
    ap.add_argument("--watchdog", type=int, default=0, help="dump all Python stacks to stderr after this many seconds")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the state they leave (u, v) to DIR/<name>.npy, "
                         "DIR/<name>_rank<r>.npy with several GPUs; on large meshes a seeded sample, all files "
                         "together at most 32 MiB")
    ap.add_argument("-v", "--verbose", action="store_true")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs: the timed path of --impl ours only")
    if a.watchdog > 0:
        import faulthandler

        faulthandler.dump_traceback_later(a.watchdog, exit=True)
    t_start = time.time()

    def log(msg):
        if a.verbose:
            print(f"[bench r{os.environ.get('RANK', '0')} +{time.time() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(3, a.warmup)
    W = WORKLOADS[a.workload]
    deg = a.degree or W["P"]
    n_per_gpu = a.n_per_gpu or W["n"]
    config = {"workload": f"{W['label']}, degree {deg} hexahedra, {n_per_gpu}^3 cells per GPU, {a.dtype}",
              "degree": deg, "cells_per_gpu": n_per_gpu**3, "parallelism": f"block partition x{world}",
              "l2": "working set per GPU (G + dofmap + 9 vectors, GBs) >> 126 MB L2: no flush needed"}
    METRIC = "fused RK4 stage throughput (global dofs x stages / s)"
    NST = 4  # stages (= operator applications) per step
    if a.integrator == "leapfrog":
        if a.workload == "nonlinear_bowl" or a.impl != "ours":
            raise SystemExit("--integrator leapfrog: linear workloads of this repo only (the reference implements RK4)")
        METRIC, NST = "fused leapfrog step throughput (global dofs x steps / s; one operator application per step)", 1

    if a.impl == "reference":
        # the reference's CPU implementation of the path on this box's host cores: the workload's
        # per-GPU box (the whole thing at N = 1), --steps steps after --warmup warm-ups
        if rank != 0:
            return 0
        if W["nonlinear"] or a.workload != "linear_box":
            print(json.dumps({"impl": "reference", "unavailable": "the reference has a CPU loop for demo_linear_box only "
                              "(numba-cpu/demo_linear_box.py); Westervelt / piston have no CPU twin at this size"}), flush=True)
            return 0
        r = time_cpu(a.steps, max(1, a.warmup), n_per_gpu, deg, a.dtype, a.cpu_kind)
        cfg = dict(config)
        cfg["parallelism"] = f"{r['cores']} host processes, cell blocks {'x'.join(map(str, r['grid']))}, no halo exchange"
        cfg["sample"] = r["sample"]
        if world > 1:
            cfg["note"] = (f"N = {world}: the CPU arm runs ONE GPU's share of the weak-scaled workload "
                           f"({n_per_gpu}^3 cells) on this single host; GDoF/s does not depend on the box size")
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "GDoF/s", "n_gpus": a.gpus,
                "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"],
                "steps_per_s": r["steps_per_s"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": a.dtype, "data": "synthetic", "config": cfg,
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "impl",
                                                   "scaling_check", "operators_sha256")},
                "e2e": {"value": r["value"], "unit": "GDoF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return 0

    # stdout carries exactly one JSON line: anything libraries print there meanwhile (NCCL's
    # version banner, ...) is sent to stderr by pointing fd 1 at fd 2 until the line is ready
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this framework has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)

    if a.impl == "reference-cuda":
        # GPU-vs-GPU anchor: the reference's Numba-CUDA kernels on this B200 beside ours
        if rank != 0:
            return 0
        r = reference_cuda_arm(n_per_gpu, deg, a.dtype)
        os.dup2(stdout_fd, 1)
        print(json.dumps({"impl": "reference-cuda", "metric": "operator GDoF/s (stiffness, mass), reference Numba-CUDA "
                          "kernels vs this repo on the same B200", "unit": "GDoF/s", "n_gpus": 1, "dtype": a.dtype,
                          "data": "synthetic", **r}), flush=True)
        return 0

    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from fenicsx_fus_gpu_b200 import _lib
    from fenicsx_fus_gpu_b200 import operators as ops

    dtype = np.float64 if a.dtype == "f64" else np.float32
    s = np.dtype(dtype).itemsize
    lib = _lib.lib()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def maxr(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- N > 1: is the multi-GPU path RIGHT on these GPUs?  One small global box solved on all
    #      ranks (peer-memory halo, interior/interface overlap, graph replay) and on rank 0 alone ----
    parity = None
    if world > 1:
        from fenicsx_fus_gpu_b200.selfcheck import multi_gpu_parity

        keys = ("rel_l2_u", "rel_l2_v", "tol", "ok", "global_cells", "global_dofs", "steps", "halo", "graph",
                "interface_cells", "shared_dofs", "partition")
        for part_kind in ("block", "blob"):
            log(f"multi-GPU parity leg ({part_kind} partition)")
            pr = multi_gpu_parity(P=deg, n_per_rank=max(4, 24 // deg), dtype=dtype, nsteps=8,
                                  workload="westervelt" if W["nonlinear"] else "linear", halo_kind=a.halo,
                                  use_graph=not a.no_graph, split_cells=not a.no_split, partition=part_kind)
            leg = {k: pr[k] for k in keys}
            if part_kind == "block":
                parity = leg
                parity["what"] = ("one global box solved on all ranks (this run's halo, graph replay) vs the same box "
                                  "on rank 0 alone: rel-L2 of the gathered state")
            else:
                leg["what"] = ("the same check on an unstructured-like partition: irregular connected parts, shuffled "
                               "cell / dof / ghost order, pseudo-random ownership of the shared dofs")
                parity["unstructured_like"] = leg
            if not pr["ok"]:
                if rank == 0:
                    os.dup2(stdout_fd, 1)
                    print(json.dumps({"metric": METRIC, "value": None, "n_gpus": world, "multi_gpu_parity": parity,
                                      "error": "multi-GPU parity check failed: not timing a wrong answer"}), flush=True)
                os._exit(3)

    log("building the problem")
    solver, info = build_problem(rank, world, n_per_gpu, dtype, a.halo, a.workload, deg, a.geometry,
                                 split_cells=not a.no_split, integrator=a.integrator,
                                 rank_grid=[int(v) for v in a.rank_grid.split("x")] if a.rank_grid else None,
                                 renumber_shared=not a.no_renumber)
    config["integrator"] = a.integrator
    config["geometry"] = ("G streamed (reference data flow)" if a.geometry == "stream" else
                          f"auto: {solver.nrect} rectilinear + {solver.naff - solver.nrect} affine of {solver.ncells} "
                          "cells per GPU keep 6 geometric factors instead of 6 n^3")
    halo_txt = {"p2p": "NVLink peer memory + per-neighbour epoch flags, no barrier: one kernel gathers the ghost sums, "
                       "closes the shared dofs and puts the next stage input into the neighbours' ghost slots while "
                       f"the close of the non-shared dofs runs (split_mode={a.split_mode})",
                "nccl": "NCCL send/recv", "none": "none (1 GPU)"}[info["halo"]]
    gtxt = "x".join(str(v) for v in ([int(v) for v in a.rank_grid.split("x")] if a.rank_grid else info["rank_grid"]))
    config["parallelism"] = f"block partition x{world} (rank grid {gtxt}), halo: {halo_txt}"
    if world > 1:
        config["local_numbering"] = ("index map's own" if a.no_renumber else
                                     "owned dofs that neighbours ghost moved to a contiguous tail (utils.shared_last_numbering)")
    if world > 1 and info["halo"] == "p2p":
        config["interface_cells_per_gpu"] = int(solver.ninterface)
        config["shared_dofs_per_gpu"] = int(solver.halo.nshared)
    solver.use_graph = not a.no_graph
    solver.split_mode = a.split_mode
    log(f"problem built: {info['ndofs_local']} local dofs, {info['ncells_local']} cells")
    dt = info["dt"]

    # ---- device-resident timing: K graph-replayed RK4 steps ------------------
    uuid = None
    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        pass
    cvd = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
    if a.dump_outputs:
        dump_idx = torch.from_numpy(dump_indices(info["nlocal"], s, 2, rank, world)).cuda()
    clocks = Clocks(uuid or (int(cvd[local_rank]) if local_rank < len(cvd) else local_rank))
    clocks.start()
    solver.init()
    solver.rk4(0.0, dt, warmup)  # warm-up (captures the graph)
    torch.cuda.synchronize()
    log(f"warm-up done (graph={'yes' if solver._graph is not None else 'no: ' + str(solver.graph_error)})")
    lib.fus_reset_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    barrier()
    e0.record()
    solver.rk4(solver.t, dt, a.steps)
    e1.record()
    barrier()
    elapsed = maxr(e0.elapsed_time(e1) * 1e-3)
    gdofs_global = info["global_dofs"]
    value = gdofs_global * NST * a.steps / elapsed / 1e9
    log(f"timed region done: {elapsed * 1e3 / a.steps:.3f} ms/step")
    # the state the timed steps leave, gathered on the device before the next steps overwrite it;
    # copied to the host and written once the clock sampling below has stopped
    dumped = {"u": solver.u[dump_idx], "v": solver.v[dump_idx]} if a.dump_outputs else None

    # ---- sustained: the same steps for >= 1 s (the contract's K is short); the clocks are sampled
    #      from the start of the timed region to the end of this one (all of it the same workload) ----
    sustained = None
    if a.sustain_steps > 0 and not a.no_extras:
        ns = max(a.sustain_steps, a.steps)
        barrier()
        e0.record()
        solver.rk4(solver.t, dt, ns)
        e1.record()
        barrier()
        el_s = maxr(e0.elapsed_time(e1) * 1e-3)
        sustained = {"steps": ns, "seconds": el_s, "ms_per_step": el_s / ns * 1e3,
                     "value": gdofs_global * NST * ns / el_s / 1e9, "unit": "GDoF/s"}
        log(f"sustained: {sustained['ms_per_step']:.3f} ms/step over {el_s:.2f} s")
    w1 = time.time()
    clk = clocks.stop(w0, w1)
    clk["window"] = "timed region + sustained run (same steps)"
    if dumped is not None:
        dump_outputs(a.dump_outputs, dumped, rank, world)
    if world > 1:  # every rank's GPU, not only rank 0's
        allc = [None] * world
        dist.all_gather_object(allc, clk)
        clk = dict(clk)
        clk["per_rank_sm_mhz"] = [c.get("sm_mhz") for c in allc]
        clk["reasons"] = sorted({r for c in allc for r in c.get("reasons", [])})
        clk["samples"] = int(sum(c.get("samples", 0) for c in allc))
    if getattr(solver.halo, "p2p", False):
        solver.halo.status()  # a timed-out wait means the numbers are meaningless: raise

    # kernels per step: counted once in eager mode (a graph replay bypasses the C entry points)
    lib.fus_reset_launch_count()
    solver.use_graph = False
    solver.rk4(solver.t, dt, 1)
    torch.cuda.synchronize()
    per_step = int(lib.fus_launch_count())
    # the dominant kernel IN SITU: the same steps launched eagerly with a CUDA-event pair around
    # every stage-kernel launch (per stage: one, or interior + interface with the peer-memory halo)
    solver.probe = []
    nprobe = min(a.steps, 10)
    solver.rk4(solver.t, dt, nprobe)
    torch.cuda.synchronize()
    t_in_step = float(np.sum([e_a.elapsed_time(e_b) for e_a, e_b in solver.probe])) * 1e-3 / (NST * nprobe)
    n_probed = len(solver.probe)
    solver.probe = None
    solver.use_graph = not a.no_graph

    # ---- end to end: per step, H2D of the step's source amplitudes from pinned host,
    #      the step, D2H of the sampled pressure plane (the demo's 100x100 probe grid) -------
    nsample = min(10000, info["nlocal"])
    sample_idx = torch.linspace(0, info["nlocal"] - 1, nsample, device="cuda").to(torch.int64)
    sample_dev = torch.empty(nsample, dtype=solver.T, device="cuda")
    sample_host = torch.empty(nsample, dtype=solver.T).pin_memory()
    tab_host = torch.from_numpy(solver.source_table(solver.t, dt, a.steps + warmup)).pin_memory()
    solver.gtab = torch.zeros((1, 8), dtype=solver.T, device="cuda")
    solver.step_dev.zero_()
    if solver.use_graph:
        solver._capture(dt)  # graph bound to the 1-row device table
    log("e2e graph ready")
    row = solver.gtab

    def e2e_step(k):
        row.copy_(tab_host[k:k + 1], non_blocking=True)  # H2D: this step's inputs
        solver.step_dev.zero_()
        solver._replay_step(dt)
        check = _lib.fn("fus_pack_fwd", dtype)(solver.u.data_ptr(), sample_dev.data_ptr(), sample_idx.data_ptr(),
                                               nsample, torch.cuda.current_stream().cuda_stream)
        assert check == 0
        sample_host.copy_(sample_dev, non_blocking=True)  # D2H: the step's result
        torch.cuda.current_stream().synchronize()
        return float(sample_host[0])

    solver.begin_steps()
    for k in range(warmup):
        e2e_step(k)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for k in range(a.steps):
        e2e_step(warmup + k)
    e1.record()
    solver.end_steps()
    barrier()
    e2e_elapsed = maxr(max(e0.elapsed_time(e1) * 1e-3, 0.0))
    e2e_wall = maxr(time.perf_counter() - t0)
    e2e_value = gdofs_global * NST * a.steps / max(e2e_elapsed, e2e_wall) / 1e9
    h2d = 8 * s
    d2h = nsample * s

    log("e2e done")
    # ---- the dominant kernel alone, under CUDA events on the launching stream (roofline):
    #      3 warm-ups, then `reps` back-to-back launches between one event pair (mean) and
    #      `reps` individually bracketed launches (min), SURVEY.md 8(d) protocol ----
    nc, nd = info["ncells_local"], info["ndofs_local"]
    n = deg + 1
    nd3 = n**3
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(nd, dtype=solver.T, device="cuda", generator=gen)
    y = torch.zeros(nd, dtype=solver.T, device="cuda")
    D = torch.from_numpy(info["tb"].dphi_1D).cuda()
    tname = "double" if a.dtype == "f64" else "float"
    if a.geometry == "auto":
        # the solver's own stage-kernel launches (rectilinear / affine / streamed ranges) on its own vectors
        solver._set_tables()
        launch = solver._stage_kernel if W["nonlinear"] else solver._stiffness
        geo = "2" if solver.nrect == nc else ("1" if solver.naff == nc else "mixed")
        kname = f"stiffness_kernel<{tname},{n},{1 if W['nonlinear'] else 0},1,GEO={geo}> (geometry=auto)"
        nstream = nc - solver.naff
        per_dof = 3 if W["nonlinear"] else 2
        bytes_stiff = nstream * (nd3 * 4 + 6 * nd3 * s + 2 * s) + solver.naff * (nd3 * 4 + 8 * s) + per_dof * s * nd
    elif W["nonlinear"]:
        # the Westervelt stage kernel: both stiffness terms in one pass over G (the cell-mass pair is
        # pointwise in the close kernel), launched as the solver launches it, on its own vectors
        solver._set_tables()
        launch = solver._stage_kernel
        kname = f"stiffness_kernel<{tname},{n},1,1,0> (fus_stiffness2_{a.dtype}: K(c3; un) + K(c4; vn))"
        # per cell: dofmap + G + 2 coefficients; per dof: read un, vn, write b
        bytes_stiff = nc * (nd3 * 4 + 6 * nd3 * s + 2 * s) + 3 * s * nd
    else:
        K = ops.stiffness_operator(deg, dtype)

        def launch():
            K[nc, (n, n, n)](x, solver.cell_coeff2, y, solver.G, solver.dofmap, D)
        kname = f"stiffness_kernel<{tname},{n},0,1> (fus_stiffness_{a.dtype})"
        bytes_stiff = nc * (nd3 * 4 + 6 * nd3 * s + s) + 2 * s * nd  # SURVEY.md 8(d): B_K per cell + 2s per dof
    reps = max(20, a.steps)
    for _ in range(3):
        launch()
    barrier()
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    t_stiff = e0.elapsed_time(e1) * 1e-3 / reps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for ea, eb in evs:
        y.zero_()
        ea.record()
        launch()
        eb.record()
    torch.cuda.synchronize()
    t_stiff_min = float(np.min([ea.elapsed_time(eb) for ea, eb in evs])) * 1e-3
    peak, peak_kind = peaks()
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "stiffness_traffic.json")))
        if (n_per_gpu == tr.get("n_per_gpu") and a.dtype == tr.get("dtype") and a.workload == "linear_box"
                and deg == 4 and world == 1 and a.geometry == "stream"):
            traffic = tr["dram_bytes_per_launch"]
    except Exception:
        pass
    # achieved = algorithmic bytes / the kernel's average duration inside the RK steps (CUDA events
    # around each of its launches); the stand-alone figure (the same kernel launched back to
    # back, which runs into the power cap sooner) rides along
    roofline = {"kernel": kname, "bound": "hbm", "achieved": bytes_stiff / t_in_step / 1e9, "peak": peak,
                "unit": "GB/s", "frac": bytes_stiff / t_in_step / 1e9 / peak, "traffic": traffic,
                "traffic_source": None if traffic is None else "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum "
                                                               "of this kernel (profiles/stiffness_traffic.json)",
                "peak_kind": peak_kind, "algorithmic_bytes_per_launch": bytes_stiff, "launch_ms": t_in_step * 1e3,
                "launches_timed": n_probed, "timing": "CUDA events around every launch of the kernel inside the RK steps"
,
                "standalone": {"launch_ms": t_stiff * 1e3, "launch_ms_min": t_stiff_min * 1e3, "launches_timed": reps,
                               "achieved": bytes_stiff / t_stiff / 1e9, "frac": bytes_stiff / t_stiff / 1e9 / peak,
                               "timing": "back-to-back launches between one event pair"}}
    # the mass operator (cells) for the "operators" block
    evm = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    c1 = torch.ones(nc, dtype=solver.T, device="cuda")
    for ea, eb in evm:
        y.zero_()
        ea.record()
        ops.mass_operator[1, 128](x, c1, y, info["detJ"], info["dofmap"])
        eb.record()
    torch.cuda.synchronize()
    t_mass = float(np.mean([ea.elapsed_time(eb) for ea, eb in evm])) * 1e-3
    bytes_mass = nc * (nd3 * (4 + s) + s) + 2 * s * nd
    stage_bytes = solver.stage_bytes()
    stage_t = elapsed / (NST * a.steps)

    # ---- the operator through the C ABI with HOST buffers (fus_stiffness_host_*): x from pinned
    #      host memory, y back to pinned host memory, both copies inside the call ----
    op_host = None
    if not W["nonlinear"] and solver.G is not None and a.geometry == "stream" and not a.no_extras:
        xh = torch.randn(nd, dtype=solver.T).pin_memory()
        yh = torch.zeros(nd, dtype=solver.T).pin_memory()
        fh = _lib.fn("fus_stiffness_host", dtype)
        st = torch.cuda.current_stream().cuda_stream
        op_host = {}
        for label, flags in (("accumulate", 0), ("y_zero", _lib.FUS_HOST_Y_ZERO)):
            def host_call():
                rc = fh(xh.data_ptr(), yh.data_ptr(), nd, x.data_ptr(), y.data_ptr(), solver.cell_coeff2.data_ptr(),
                        solver.G.data_ptr(), solver.dofmap.data_ptr(), D.data_ptr(), nc, deg, flags, st)
                assert rc == 0
            host_call()
            barrier()
            t0h = time.perf_counter()
            nh = 5
            for _ in range(nh):
                host_call()  # synchronous on return
            th = maxr((time.perf_counter() - t0h) / nh)
            op_host[label] = {"value": gdofs_global / th / 1e9, "unit": "GDoF/s", "ms_per_call": th * 1e3,
                              "h2d_bytes_per_call": (2 if flags == 0 else 1) * nd * s, "d2h_bytes_per_call": nd * s}
        op_host["what"] = ("fus_stiffness_host: y_host (+)= K x_host through the C ABI with pinned HOST buffers, copies "
                           "inside the call; 'y_zero' = FUS_HOST_Y_ZERO (y is not uploaded, cleared on the device)")
        del xh, yh

    # ---- the same steps with geometry="auto" (extra, not the headline): cells with a constant
    #      Jacobian keep 6 geometric factors instead of 6 n^3 (results equal to rounding) ----
    affine = None
    if not a.no_affine and not a.no_extras and a.geometry == "stream" and (world == 1 or info["halo"] == "nccl"):  # (the peer-memory arena holds one solver's vectors)
        del x, y
        sol2 = info["make_solver"]("auto")
        sol2.use_graph = not a.no_graph
        sol2.init()
        sol2.rk4(0.0, dt, warmup)
        barrier()
        e0.record()
        sol2.rk4(sol2.t, dt, a.steps)
        e1.record()
        barrier()
        el2 = maxr(e0.elapsed_time(e1) * 1e-3)
        affine = {"value": gdofs_global * NST * a.steps / el2 / 1e9, "unit": "GDoF/s", "ms_per_step": el2 / a.steps * 1e3,
                  "steps_per_s": a.steps / el2, "affine_cells_per_gpu": sol2.naff, "cells_per_gpu": sol2.ncells,
                  "algorithmic_bytes_per_stage": sol2.stage_bytes(),
                  "note": "solver(geometry='auto'): G = wq x Gc on cells with a constant Jacobian (all cells of "
                          "this box); not the headline because unstructured meshes stream G"}
        if world > 1:
            sol2._graph = None

    line = {
        "metric": METRIC, "value": value, "unit": "GDoF/s",
        "workload": a.workload, "n_gpus": world, "steps": a.steps, "warmup": warmup, "ms_per_step": elapsed / a.steps * 1e3,
        "steps_per_s": a.steps / elapsed, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic", "config": {**config, "global_dofs": gdofs_global,
                                                          "global_cells": list(info["global_cells"])},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "GDoF/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps_per_s": a.steps / max(e2e_elapsed, e2e_wall)},
        "gpu_launches": per_step * a.steps,
        "roofline": roofline,
        "stage_roofline": {"bound": "hbm", "achieved": stage_bytes / stage_t / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": stage_bytes / stage_t / 1e9 / peak,
                           "algorithmic_bytes_per_stage": stage_bytes, "stage_ms": stage_t * 1e3,
                           "bytes_model": ("stage kernel bytes + 10.25 vector passes per stage (what the fused "
                                           "ping-pong stages move: 9 + 12 + 12 + 8 per step)" if NST == 4 else
                                           "stiffness bytes + 7 vector passes per leapfrog step"),
                           "survey_8d_model": None if NST != 4 else {
                                               "algorithmic_bytes_per_stage": solver.stage_bytes_survey(),
                                               "frac": solver.stage_bytes_survey() / stage_t / 1e9 / peak,
                                               "note": "SURVEY.md 8(d): 6s + stiffness + 8s per dof, more than "
                                                       "this implementation moves"}},
        "sustained": sustained,
        "multi_gpu_parity": parity,
        "e2e_operator_host_buffers": op_host,
        "affine_geometry": affine,
        "operators": {("westervelt_stage_kernel_gdofs" if W["nonlinear"] else "stiffness_gdofs"): info["ndofs_local"] / t_stiff / 1e9, "mass_gdofs": info["ndofs_local"] / t_mass / 1e9,
                      "mass_roofline_frac": bytes_mass / t_mass / 1e9 / peak, "mass_ms": t_mass * 1e3,
                      "per_gpu_dofs": info["ndofs_local"]},
    }
    if rank == 0:
        line["cpu_baseline"] = None
        if world == 1 and not a.no_cpu and not a.no_extras and a.workload == "linear_box":
            # the reference's numba-cpu path on this host's cores: the same box, 3 steps (bounded sample)
            try:
                r = time_cpu(3, 1, n_per_gpu, deg, a.dtype, a.cpu_kind)
                line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "impl", "ms_per_step",
                                                          "scaling_check", "operators_sha256")}
                if r["impl"] == "numba":  # second, labelled figure: the reference's C++ templates in the same harness
                    try:
                        r2 = time_cpu(2, 1, n_per_gpu, deg, a.dtype, "cpp")
                        if r2["impl"] == "cpp":
                            line["cpu_baseline"]["cpp_templates"] = {k: r2[k] for k in ("value", "unit", "cores", "ms_per_step", "sample")}
                    except Exception as e:
                        line["cpu_baseline"]["cpp_templates"] = {"error": repr(e)[:300]}
            except Exception as e:
                line["cpu_baseline"] = {"error": repr(e)[:500]}
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down: ncclCommDestroy blocks while captured graphs still hold NCCL
        # kernels, so drop the graphs first and do not wait on communicator
        # destruction (the process is about to exit anyway).
        dist.barrier()
        torch.cuda.synchronize()
        solver._graph = None
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
