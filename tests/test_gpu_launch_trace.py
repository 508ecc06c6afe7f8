"""Launch trace of the solvers against ``golden/launch_trace.json``.

A recording stand-in for the ctypes library handle logs every C-ABI call a solver makes, per
(emulated) rank: the symbol and its arguments, integers as they are, floats exactly
(``float.hex``) and pointers - the entries of the pointer arrays of the halo calls included -
as ids in order of first appearance.  Two parts are compared:

* the steps (2 eager ``rk4`` steps, then one ``step_eager`` for the RK4 solvers): identical,
  pointer ids included;
* the set-up (``box_setup`` through ``init``): identical symbols and non-pointer arguments
  (temporaries freed and reused by the allocator may change which addresses repeat).

The cases cover the integrators, float types, streamed and mixed (rectilinear / affine / streamed)
geometry, no halo, the pack/send/unpack halo and the peer-memory halo with its split modes on two
ranks emulated on one GPU.  ``golden/make_launch_trace.py`` writes the golden file (gzip-compressed JSON).
"""

import ctypes as C
import gzip
import json
import os
import threading

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "launch_trace.json.gz")
P, NCELLS, LENGTHS = 3, (6, 3, 3), (0.006, 0.003, 0.003)
_SKIP = {"fus_last_error", "fus_halo_destroy"}  # error reporting; teardown runs whenever the GC does


def _cases():
    out = {}

    def add(work, geometry="stream", halo="none", dtype="f64", split_mode="none", split_cells=True, renumber=True):
        name = "-".join([work, dtype, geometry, halo] + ([split_mode] if split_mode != "none" else [])
                        + ([] if split_cells else ["nosplit"]) + ([] if renumber else ["mask"]))
        out[name] = dict(work=work, geometry=geometry, halo=halo, dtype=dtype, split_mode=split_mode,
                         split_cells=split_cells, renumber=renumber)

    for work in ("linear", "leapfrog", "westervelt", "westervelt_cells"):
        for geometry, halo in (("stream", "none"), ("auto", "none"), ("stream", "nccl"), ("stream", "p2p"),
                               ("auto", "p2p")):
            add(work, geometry, halo)
    add("linear", dtype="f32")
    add("linear", "auto", "p2p", dtype="f32")
    for geometry in ("stream", "auto"):
        for mode in ("two", "fused"):
            add("linear", geometry, "p2p", split_mode=mode)
    add("linear", halo="p2p", split_cells=False)
    add("linear", halo="p2p", renumber=False)
    add("linear", halo="p2p", split_mode="two", renumber=False)
    add("leapfrog", halo="p2p", split_mode="fused")
    add("leapfrog", halo="p2p", renumber=False)
    add("westervelt", halo="p2p", split_mode="two")
    add("westervelt_cells", "auto", "p2p", split_mode="fused")
    add("westervelt_cells", halo="p2p", split_cells=False)
    add("westervelt", halo="p2p", dtype="f32", split_mode="fused", renumber=False)
    return out


CASES = _cases()


class _Recorder:
    """Stands in for the library handle: forwards every call and logs it for the calling thread
    (one thread per emulated rank)."""

    def __init__(self, lib):
        self._real = lib
        self._tls = threading.local()

    def take(self, more=True):
        """The log so far; a fresh log with fresh pointer ids follows if ``more``."""
        log = getattr(self._tls, "log", None)
        self._tls.log, self._tls.ids = ([], {}) if more else (None, None)
        return log

    def _pid(self, p):
        p = p.value if isinstance(p, C.c_void_p) else p
        if not p:
            return None
        return "p%d" % self._tls.ids.setdefault(int(p), len(self._tls.ids))

    def _encode(self, args, argtypes):
        out = []
        for i, a in enumerate(args):
            if isinstance(a, C.Array):  # pointer array, followed by its entry count
                out.append([self._pid(a[j]) for j in range(int(args[i + 1]))])
            elif (i < len(argtypes) and argtypes[i] is C.c_void_p) or isinstance(a, C.c_void_p):
                out.append(self._pid(a))
            elif isinstance(a, (float, np.floating)):
                out.append(float(a).hex())
            elif isinstance(a, (int, np.integer)):
                out.append(int(a))
            else:
                out.append(type(a).__name__)
        return out

    def __getattr__(self, name):
        f = getattr(self._real, name)

        def call(*args):
            log = getattr(self._tls, "log", None)
            if log is not None and name not in _SKIP:
                log.append([name] + self._encode(args, getattr(f, "argtypes", None) or ()))
            return f(*args)

        return call


def _warp(su):
    """Mix the three geometry kinds along x: vertices with x < 0.3 Lx jittered (streamed cells), y
    sheared by the part beyond 0.6 Lx (affine cells), rectilinear cells in between."""
    import torch

    from fenicsx_fus_gpu_b200 import precompute as pre

    x = su.mesh.x_g.astype(np.float64)
    X, Y, Z = (x / su.h).T
    lo = X < 0.3 * NCELLS[0]
    x[lo] += 0.1 * su.h * np.stack([np.sin(7 * Y + 3 * Z), np.sin(5 * X + 2 * Z), np.sin(3 * X + 4 * Y)], 1)[lo]
    x[:, 1] += 0.3 * np.maximum(x[:, 0] - 0.6 * LENGTHS[0], 0.0)
    su.mesh.x_g = np.ascontiguousarray(x, dtype=su.mesh.x_g.dtype)
    su.dev["x_g"] = torch.from_numpy(su.mesh.x_g).cuda()
    pre.compute_geometry(su.dev["G"], su.dev["detJ"], (su.dev["x_dofs"], su.dev["x_g"]), su.mesh.num_cells,
                         su.dev["dphi"], su.dev["wts"])


def _run_rank(case, rec, rank, world, transport=None, sdata=None):
    import torch

    import problems
    from fenicsx_fus_gpu_b200 import problem
    from fenicsx_fus_gpu_b200 import substrate as S
    from fenicsx_fus_gpu_b200.scatterer import P2PHaloExchange, local_fabric

    dt = np.float64 if case["dtype"] == "f64" else np.float32
    rec.take()
    fabric = None
    if case["halo"] == "p2p":
        fabric = local_fabric(transport.cluster, rank, P2PHaloExchange.arena_bytes(S.num_dofs(NCELLS, P), dt))
    su = problem.box_setup(P, NCELLS, LENGTHS, dt, rank, world, comm=transport, scatter_data=sdata,
                           halo_kind=case["halo"], fabric=fabric, renumber_shared=case["renumber"])
    _warp(su)
    kw = dict(geometry=case["geometry"], use_graph=False, split_cells=case["split_cells"])
    work = case["work"]
    if work in ("linear", "leapfrog"):
        s = problem.linear_solver(su, [2], [3, 5], integrator="leapfrog" if work == "leapfrog" else "rk4", **kw)
        step = problems.cfl_dt(P, su.h, 1500.0, 0.5e6, cfl=0.3)
    else:
        s = problem.westervelt_solver(su, [2], [0, 1, 3, 4, 5], alpha_dB=20.0, p0=1.0e6,
                                      mass_form="cells" if work == "westervelt_cells" else "pointwise", **kw)
        step = problems.cfl_dt(P, su.h, 1480.0, 1.1e6, cfl=0.3)
    s.split_mode = case["split_mode"]
    s.init()
    setup = rec.take()
    s.rk4(0.0, step, 2)
    if work != "leapfrog":
        s.step_eager(step)
    torch.cuda.synchronize()
    steps = rec.take(more=False)
    meta = dict(stage_bytes=s.stage_bytes(), naff=s.naff, nrect=s.nrect, ninterface=s.ninterface,
                nsegs=len(s._segs))
    return dict(meta=meta, setup=setup, steps=steps)


def trace(name):
    """{"ranks": [{"meta", "setup", "steps"} per rank]} of case ``name``."""
    from fenicsx_fus_gpu_b200 import _lib
    from fenicsx_fus_gpu_b200 import substrate as S
    from fenicsx_fus_gpu_b200 import utils
    from fenicsx_fus_gpu_b200.scatterer import LocalCluster

    case = CASES[name]
    real = _lib.lib()
    rec = _lib._lib = _Recorder(real)  # before any halo or solver exists: the halo keeps the handle it sees
    try:
        if case["halo"] == "none":
            return dict(ranks=[_run_rank(case, rec, 0, 1)])
        dt = np.float64 if case["dtype"] == "f64" else np.float32
        parts = S.partition_box(NCELLS, P, 2, lengths=LENGTHS, dtype=dt)
        sdata = utils.compute_scatterer_data_all([p.index_map for p in parts])
        return dict(ranks=LocalCluster(2).run(lambda r, tr: _run_rank(case, rec, r, 2, tr, sdata[r])))
    finally:
        _lib._lib = real


def _strip_pointers(log):
    return [[("p" if isinstance(a, str) and a.startswith("p") else
              [None if e is None else "p" for e in a] if isinstance(a, list) else a) for a in call] for call in log]


def _first_diff(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        if x != y:
            return f"call {i}: {x} != golden {y}"
    return f"length {len(a)} != golden {len(b)}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_launch_trace_matches_golden(name):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    with gzip.open(GOLDEN, "rt") as f:
        gold = json.load(f)[name]["ranks"]
    got = trace(name)["ranks"]
    assert len(got) == len(gold)
    for r, (g, e) in enumerate(zip(got, gold)):
        assert g["meta"] == e["meta"], (r, g["meta"], e["meta"])
        assert g["steps"] == e["steps"], (r, _first_diff(g["steps"], e["steps"]))
        gs, es = _strip_pointers(g["setup"]), _strip_pointers(e["setup"])
        assert gs == es, (r, _first_diff(gs, es))
