"""The dual-operand and Westervelt cell kernels, the mass kernels, the boundary-term kernel and
the RK / leapfrog stage kernels, each against a plain float64 reference of the same operation.

The whole-run solver tests compare rel-L2 norms after many steps.  The second stiffness operand
and the Westervelt mass pair are small there, so an error in them, or in a few cells or dofs,
can stay under those tolerances.  Here every output entry i is checked on its own:

    |out_i - ref_i| <= k * (u_T + u_64) * Y_i

``ref`` is computed in float64 from exactly the values the kernel sees (inputs stored in T and
widened, the T copy of the derivative table, affine factors expanded from their T values).
``Y`` bounds the rounding: ``|K|(|x|)`` for the cell kernels, or a first-order error majorant
for the elementwise kernels (``Tracked`` below).  ``u_T`` is the unit roundoff of the kernel's
type and ``u_64`` that of the reference.  A per-entry bound does not depend on the atomic
summation order, and cancellation cannot make it flaky.  Every cell-kernel test also checks
that the bound is sharp enough: references with one term dropped or one factor wrong must
violate it somewhere.
"""

import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U64 = 2.0**-53
UNIT = {np.dtype(np.float64): 2.0**-53, np.dtype(np.float32): 2.0**-24}
PACK = {np.dtype(np.float64): 2, np.dtype(np.float32): 4}  # elements per 16-byte vector access
BAD_ARGUMENT = 100002
TYPES = [np.float64, np.float32]

# worst |err| / (u_T * Y) seen per kernel family, printed at the end of the module (run with -s)
MARGINS = {}


def _note(family, dt, ratio, k):
    key = (family, np.dtype(dt).name)
    old = MARGINS.get(key, (0.0, k))
    MARGINS[key] = (max(old[0], ratio), k)


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    for (family, dt), (ratio, k) in sorted(MARGINS.items()):
        print(f"\nmargin {family} {dt}: max |err|/(u_T*Y) = {ratio:.3g} (k = {k})")


# --------------------------------------------------------------------------- #
# float64 references
# --------------------------------------------------------------------------- #
def cells_per_batch():
    """{(dtype, n): B} from the Cfg table of csrc/stiffness_kernel.cuh."""
    path = os.path.join(ROOT, "fenicsx_fus_gpu_b200", "csrc", "stiffness_kernel.cuh")
    with open(path) as f:
        rows = re.findall(r"^FUS_CFG\((double|float), (\d+), (\d+), \d+, \d+\)", f.read(), re.M)
    return {(np.dtype(np.float64 if t == "double" else np.float32), int(n)): int(b) for t, n, b in rows}


def box_dofmap(ncells, P, seed):
    """Tensor-product dofmap of the first ``ncells`` cells of a box with 4 x 5 cells per x-slab
    (dofs shared by up to 8 cells), dof numbers randomly permuted.  Returns (dofmap, ndofs)."""
    n, ny, nz = P + 1, 5, 4
    nx = -(-ncells // (ny * nz))
    my, mz = ny * P + 1, nz * P + 1
    c = np.arange(nx * ny * nz)[:ncells]
    cx, cy, cz = c // (ny * nz), (c // nz) % ny, c % nz
    i, j, k = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    g = (((cx[:, None] * P + i.ravel()) * my + cy[:, None] * P + j.ravel()) * mz + cz[:, None] * P + k.ravel())
    used, dm = np.unique(g, return_inverse=True)
    perm = np.random.default_rng(seed).permutation(used.size)
    return np.ascontiguousarray(perm[dm.reshape(g.shape)], dtype=np.int32), used.size


def stiffness_ref(D, G, c, x, dofmap, nd):
    """sum_cells K(c; x) in float64, sum-factorised: gradient along each axis with D, then
    c * G * grad, then D^T along each axis, then scatter-add.  D[q, i] = l_i'(x_q); G (nc, n^3, 6)
    as [G00 G01 G02 G11 G12 G22].  With every argument replaced by its absolute value this is the
    majorant |K|(|x|)."""
    n = D.shape[0]
    u = x[dofmap].reshape(-1, n, n, n)
    gx = np.einsum("ql,cljk->cqjk", D, u)
    gy = np.einsum("ql,cilk->ciqk", D, u)
    gz = np.einsum("ql,cijl->cijq", D, u)
    g = G.reshape(-1, n, n, n, 6) * c[:, None, None, None, None]
    f0 = g[..., 0] * gx + g[..., 1] * gy + g[..., 2] * gz
    f1 = g[..., 1] * gx + g[..., 3] * gy + g[..., 4] * gz
    f2 = g[..., 2] * gx + g[..., 4] * gy + g[..., 5] * gz
    yc = (np.einsum("qi,cqjk->cijk", D, f0) + np.einsum("qj,ciqk->cijk", D, f1)
          + np.einsum("qk,cijq->cijk", D, f2))
    return np.bincount(dofmap.ravel(), weights=yc.ravel(), minlength=nd)


def mass_ref(x, c, detJ, dofmap, nd):
    """sum_entities M(c; x): y[dm[e, i]] += c[e] * detJ[e, i] * x[dm[e, i]], float64."""
    return np.bincount(dofmap.ravel(), weights=(x[dofmap] * detJ * c[:, None]).ravel(), minlength=nd)


def abs_all(*a):
    return [np.abs(v) for v in a]


def check_bound(out, ref, Y, k, dt, family):
    """Assert |out - ref| <= k (u_T + u_64) Y entrywise; record the worst |err| / (u_T Y)."""
    out = np.asarray(out, np.float64)
    err = np.abs(out - ref)
    bound = k * (UNIT[np.dtype(dt)] + U64) * Y
    bad = ~(err <= bound)
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise AssertionError(f"{family}: {int(bad.sum())} entries out of bound, first {i}: out {out[i]!r} "
                             f"ref {ref[i]!r} err {err[i]:.3g} bound {bound[i]:.3g}")
    pos = Y > 0
    ratio = float((err[pos] / (UNIT[np.dtype(dt)] * Y[pos])).max()) if pos.any() else 0.0
    _note(family, dt, ratio, k)


def violates(out, ref, Y, k, dt):
    err = np.abs(np.asarray(out, np.float64) - ref)
    return bool(np.any(err > k * (UNIT[np.dtype(dt)] + U64) * Y))


class Tracked:
    """A float64 value with a first-order rounding majorant M: evaluated in a type with unit
    roundoff u, the same expression is within ~u * M of ``v`` (each operation adds the
    magnitude of its result; errors propagate through + and * and / to first order).  Inputs
    are exact (M = 0).  The elementwise kernels make at most a few roundings along any chain,
    so k = 4 covers them with room for fused multiply-adds and second-order terms."""

    __slots__ = ("v", "m")

    def __init__(self, v, m=None):
        self.v = np.asarray(v, np.float64)
        self.m = np.zeros_like(self.v) if m is None else m

    @staticmethod
    def of(a):
        return a if isinstance(a, Tracked) else Tracked(a)

    def __add__(self, o):
        o = Tracked.of(o)
        r = self.v + o.v
        return Tracked(r, self.m + o.m + np.abs(r))

    def __mul__(self, o):
        o = Tracked.of(o)
        r = self.v * o.v
        return Tracked(r, np.abs(self.v) * o.m + np.abs(o.v) * self.m + np.abs(r))

    def __truediv__(self, o):
        o = Tracked.of(o)
        r = self.v / o.v
        return Tracked(r, self.m / np.abs(o.v) + np.abs(self.v) * o.m / o.v**2 + np.abs(r))


K_ELEM = 4


def open_ref(x, adt, first):
    """fus_rk_open: [first: u0 = u; v0 = v]; un = u0 + adt ku; ku = v0 + adt kv; b = 0.
    ``x`` maps names to float64 arrays; returns {name: Tracked} of the written vectors."""
    u0 = Tracked(x["u"]) if first else Tracked(x["u0"])
    v0 = Tracked(x["v"]) if first else Tracked(x["v0"])
    out = {"un": Tracked(x["ku"]) * adt + u0, "ku": Tracked(x["kv"]) * adt + v0, "b": Tracked(0 * x["b"])}
    if first:
        out.update(u0=u0, v0=v0)
    return out


def close_ref(x, form, bdt, adt, mode, kv_stored=True):
    """fus_rk_close (form "lin"), _westervelt ("west"), _westervelt_pw ("pw") and
    fus_leapfrog_close ("leap", mode 4) as include/fus_b200.h states them."""
    t = {k: Tracked(v) for k, v in x.items()}
    if form == "leap":
        v = t["b"] / t["m"] * bdt + t["v"]
        return {"v": v, "u": v * adt + t["u"], "b": Tracked(0 * x["b"])}
    if mode == 3:  # the stage input is the base state: un = u0, vn = v0
        ku, u, v, xin = t["v0"], t["u0"], t["v0"], t["u0"]
    else:
        ku, u, v, xin = t["ku"], t["u"], t["v"], t.get("un")
    num, den = t["b"], None
    if form == "lin":
        den = t["m"]
    elif form == "west":
        den = t["m"] + t["m0"]
    else:
        den = xin * t["m2"] + t["m0"]
        num = ku * ku * t["m5"] + t["b"]
    kv = num / den
    out = {"u": ku * bdt + u, "v": kv * bdt + v}
    if kv_stored:
        out["kv"] = kv
    if form == "west":
        out["m"] = Tracked(0 * x["m"])
    zero = Tracked(0 * x["b"])
    if mode in (1, 3):
        out.update(un=ku * adt + t["u0"], ku=kv * adt + t["v0"], b=zero)
    elif mode == 2:
        out.update(u0=out["u"], v0=out["v"], un=out["u"], ku=out["v"], b=zero)
    elif mode == 4:
        out["b"] = zero
    return out


def boundary_ref(b, vn, dof, src, src2, absb, g, dg):
    """b[dof[i]] += g src[i] + dg src2[i] + vn[dof[i]] absb[i] (dof unique); missing terms None."""
    acc = Tracked(np.zeros(dof.size))
    if src is not None:
        acc = acc + Tracked(src) * g
    if src2 is not None:
        acc = acc + Tracked(src2) * dg
    if absb is not None:
        acc = acc + Tracked(vn[dof]) * Tracked(absb)
    r = Tracked(b.copy())
    s = Tracked(b[dof]) + acc
    r.v[dof], r.m[dof] = s.v, s.m
    return r


# --------------------------------------------------------------------------- #
# CPU checks of the references
# --------------------------------------------------------------------------- #
def test_cells_per_batch_table_parses():
    B = cells_per_batch()
    assert set(B) == {(np.dtype(t), n) for t in TYPES for n in range(3, 9)}
    assert all(b >= 1 for b in B.values())


@pytest.mark.parametrize("P", range(2, 8))
def test_stiffness_and_mass_references_match_oracle(P):
    import problems
    from oracle import oracle as orc

    d = problems.linear_problem(P, (3, 2, 2), (1.0, 0.8, 0.9), np.float64, perturb=0.15, seed=P)
    rng = np.random.default_rng(P)
    nd, nc = d.ndofs, d.dofmap.shape[0]
    x = rng.standard_normal(nd)
    c = rng.uniform(0.5, 2.0, nc) * rng.choice([-1.0, 1.0], nc)
    D = np.asarray(d.tb.dphi_1D, np.float64)
    y_orc = np.zeros(nd)
    orc.stiffness_operator(P, x, c, y_orc, d.G, d.dofmap, D)
    y = stiffness_ref(D, d.G, c, x, d.dofmap, nd)
    Y = stiffness_ref(*abs_all(D, d.G, c, x), d.dofmap, nd)
    assert np.all(Y >= np.abs(y))
    assert np.linalg.norm(y - y_orc) <= 1e-13 * np.linalg.norm(y_orc)
    assert np.all(np.abs(y - y_orc) <= (4 * (P + 1) + 20) * 2 * U64 * Y)
    m_orc = np.zeros(nd)
    orc.mass_operator(x, c, m_orc, d.detJ, d.dofmap)
    m = mass_ref(x, c, d.detJ, d.dofmap, nd)
    assert np.linalg.norm(m - m_orc) <= 1e-14 * np.linalg.norm(m_orc)
    assert np.all(mass_ref(*abs_all(x, c, d.detJ), d.dofmap, nd) >= np.abs(m))


def test_stage_references_are_classical_rk4():
    """The open / close references chained as a solver chains the kernels (open + 1/1/1/2, and
    the ping-pong 3/1/1/4 with buffer swaps) integrate u' = v, m v' = b(u, v) exactly as the
    textbook RK4 does, for a linear b."""
    rng = np.random.default_rng(1)
    n, dt, nsteps = 50, 0.05, 4
    A, Bc, m = rng.uniform(-2, -1, n), rng.uniform(-0.5, 0.5, n), rng.uniform(1, 2, n)
    bfun = lambda un, vn: A * un + Bc * vn  # noqa: E731
    a_rk, b_rk = (0.0, 0.5, 0.5, 1.0), (1 / 6, 1 / 3, 1 / 3, 1 / 6)
    u, v = rng.standard_normal(n), rng.standard_normal(n)
    uc, vc = u.copy(), v.copy()
    for _ in range(nsteps):  # textbook
        k1 = (vc, bfun(uc, vc) / m)
        k2 = (vc + dt / 2 * k1[1], bfun(uc + dt / 2 * k1[0], vc + dt / 2 * k1[1]) / m)
        k3 = (vc + dt / 2 * k2[1], bfun(uc + dt / 2 * k2[0], vc + dt / 2 * k2[1]) / m)
        k4 = (vc + dt * k3[1], bfun(uc + dt * k3[0], vc + dt * k3[1]) / m)
        uc = uc + dt / 6 * (k1[0] + 2 * k2[0] + 2 * k3[0] + k4[0])
        vc = vc + dt / 6 * (k1[1] + 2 * k2[1] + 2 * k3[1] + k4[1])

    def apply(x, upd):
        x.update({k: t.v for k, t in upd.items()})

    z = np.zeros(n)
    x = dict(u=u.copy(), v=v.copy(), u0=z.copy(), v0=z.copy(), ku=z.copy(), kv=z.copy(), un=z.copy(), b=z.copy(), m=m)
    for _ in range(nsteps):
        apply(x, open_ref(x, 0.0, True))
        for s in range(4):
            x["b"] = bfun(x["un"], x["ku"])
            apply(x, close_ref(x, "lin", b_rk[s] * dt, a_rk[s + 1] * dt if s < 3 else 0.0, 1 if s < 3 else 2))
    assert np.allclose(x["u"], uc, rtol=1e-13, atol=0) and np.allclose(x["v"], vc, rtol=1e-13, atol=0)
    base, acc = [u.copy(), v.copy()], [z.copy(), z.copy()]
    y = dict(ku=z.copy(), un=z.copy(), b=z.copy(), m=m)
    for _ in range(nsteps):
        for s in range(4):
            y.update(u=acc[0], v=acc[1], u0=base[0], v0=base[1])
            y["b"] = bfun(base[0], base[1]) if s == 0 else bfun(y["un"], y["ku"])
            apply(y, close_ref(y, "lin", b_rk[s] * dt, a_rk[s + 1] * dt if s < 3 else 0.0, (3, 1, 1, 4)[s],
                               kv_stored=False))
            acc = [y["u"], y["v"]]
        base, acc = acc, base
    assert np.array_equal(base[0], x["u"]) and np.array_equal(base[1], x["v"])


def test_tracked_majorant_bounds_float32_evaluation():
    """The elementwise majorant bounds what float32 arithmetic actually makes of the close."""
    rng = np.random.default_rng(3)
    n = 100000
    x = {k: rng.standard_normal(n).astype(np.float32).astype(np.float64) for k in ("u", "v", "ku", "b", "u0", "v0")}
    x["m0"] = rng.uniform(2, 4, n).astype(np.float32).astype(np.float64)
    x["m2"] = rng.uniform(-0.5, 0.5, n).astype(np.float32).astype(np.float64)
    x["m5"] = rng.uniform(-1, 1, n).astype(np.float32).astype(np.float64)
    x["un"] = x["u0"]
    bdt = float(np.float32(0.3))
    f = {k: v.astype(np.float32) for k, v in x.items()}
    m = f["un"] * f["m2"] + f["m0"]
    kv = (f["ku"] * f["ku"] * f["m5"] + f["b"]) / m
    v32 = np.float32(bdt) * kv + f["v"]
    r = close_ref(x, "pw", bdt, 0.0, 0)
    assert np.all(np.abs(v32 - r["v"].v) <= K_ELEM * 2.0**-24 * r["v"].m)
    assert not np.all(np.abs(v32 - r["v"].v) <= 0.01 * 2.0**-24 * r["v"].m)  # and is not vacuous


# --------------------------------------------------------------------------- #
# GPU plumbing
# --------------------------------------------------------------------------- #
def _torch_cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _lib():
    from fenicsx_fus_gpu_b200 import _lib as L

    return L


class Dev:
    """A device copy of a host array inside a buffer with guard elements before and after, so
    that the pointer handed to a kernel can sit ``shift`` elements off a 16-byte boundary."""

    GUARD = 16

    def __init__(self, torch, a, shift=0, seed=0):
        a = np.ascontiguousarray(a)
        self.n, self.dtype, self.lead = a.size, a.dtype, self.GUARD + shift
        rng = np.random.default_rng(seed + 7)
        self.before = rng.standard_normal(self.lead).astype(a.dtype) if a.dtype.kind == "f" else np.zeros(self.lead, a.dtype)
        self.after = rng.standard_normal(self.GUARD).astype(a.dtype) if a.dtype.kind == "f" else np.zeros(self.GUARD, a.dtype)
        self.buf = torch.from_numpy(np.concatenate([self.before, a.ravel(), self.after])).cuda()
        self.ptr = self.buf.data_ptr() + self.lead * a.dtype.itemsize

    def get(self):
        h = self.buf.cpu().numpy()
        bits = lambda z: z.view(np.uint8)  # noqa: E731
        assert np.array_equal(bits(h[:self.lead]), bits(self.before)), "guard before the vector was written"
        assert np.array_equal(bits(h[self.lead + self.n:]), bits(self.after)), "guard after the vector was written"
        return h[self.lead:self.lead + self.n]


def _bits_equal(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _t(dt, v):
    """A scalar as the kernel receives it (rounded to T), widened to float64."""
    return float(np.dtype(dt).type(v))


# --------------------------------------------------------------------------- #
# GPU: cell kernels
# --------------------------------------------------------------------------- #
def _k_cell(n):
    """Roundings on the longest dependency chain of one output entry of a cell kernel:
    2 (ca xa + cb xb) + n (gradient) + 1 (affine: coeff * wq) + 3 (the G product) + 1 (coeff)
    + n + 1 (D^T contraction, joined by the Westervelt b term) + 2 (sum of the three directions)
    + 9 (the initial value plus up to 8 cells per dof, added atomically in any order)
    + 1 (the rectilinear kernel's K1 = D^T w D and weight products are rounded to T) = 2n + 20."""
    return 2 * n + 20


def _cell_case(P, dt, form, geo, nc, off, seed, gshift=0):
    """Host inputs of one launch over cells [off, off + nc) of arrays holding off + nc + 1 cells,
    plus the float64 reference and its majorant."""
    from fenicsx_fus_gpu_b200 import operators as ops
    from fenicsx_fus_gpu_b200 import substrate as S

    n = P + 1
    Nd = n**3
    rng = np.random.default_rng(seed)
    tot = off + nc + 1
    dm, nd = box_dofmap(tot, P, seed)
    tb = S.element_tables(P, "basix", dt)
    D = np.asarray(tb.dphi_1D, dt)
    sgn = lambda k: rng.uniform(0.5, 2.0, k) * rng.choice([-1.0, 1.0], k)  # noqa: E731
    h = dict(xa=rng.standard_normal(nd), xb=rng.standard_normal(nd), ca=sgn(tot), cb=sgn(tot), c2=sgn(tot),
             c5=sgn(tot), y=rng.standard_normal(nd), m=rng.standard_normal(nd))
    if geo == "streamed":
        h["G"] = rng.standard_normal((tot, Nd, 6))
        h["detJ"] = rng.uniform(0.5, 2.0, (tot, Nd))
    else:
        Gc = rng.standard_normal((tot, 6))
        if geo == "rect":
            Gc[:, [1, 2, 4]] = 0.0
        h["Gc"], h["detJc"] = Gc, rng.uniform(0.5, 2.0, tot)
    h = {k: np.ascontiguousarray(v, dt) for k, v in h.items()}
    h["dofmap"] = dm
    h["D"] = D
    sl = slice(off, off + nc)
    r = {k: np.asarray(v, np.float64) for k, v in h.items() if k != "dofmap"}
    if geo == "streamed":
        G, detJ = r["G"][sl], r["detJ"][sl]
    else:
        if geo == "rect":
            k1, w1 = ops.rect_tables(D, np.asarray(tb.wts, dt), dt)
            h["k1"], h["w1"] = k1, w1
            w = np.asarray(w1, np.float64)
            wq = (w[:, None, None] * w[None, :, None] * w[None, None, :]).ravel()
        else:
            h["wq"] = np.ascontiguousarray(tb.wts, dt)
            wq = np.asarray(h["wq"], np.float64)
        G = wq[None, :, None] * r["Gc"][sl][:, None, :]
        detJ = wq[None, :] * r["detJc"][sl][:, None]
    return h, r, dict(G=G, detJ=detJ, D=r["D"], dm=dm[sl], nd=nd, sl=sl, Nd=Nd, gshift=gshift)


def _cell_refs(r, g, form, mutate=None):
    """(ref, majorant) of y (stiffness2) or (b, m) (Westervelt) for the cells of ``g``."""
    sl, D, G, detJ, dm, nd = g["sl"], g["D"], g["G"], g["detJ"], g["dm"], g["nd"]
    ca, cb, c2, c5 = r["ca"][sl], r["cb"][sl], r["c2"][sl], r["c5"][sl]
    if mutate == "cb":
        cb = 0 * cb
    if mutate == "c5":
        c5 = 0 * c5
    if mutate == "c2":
        c2 = 0 * c2
    if mutate == "swapG":
        G = G[..., [0, 2, 1, 3, 4, 5]]
    if mutate == "last":
        dm, G, detJ, ca, cb, c2, c5 = dm[:-1], G[:-1], detJ[:-1], ca[:-1], cb[:-1], c2[:-1], c5[:-1]
    y = r["y"] + stiffness_ref(D, G, ca, r["xa"], dm, nd) + stiffness_ref(D, G, cb, r["xb"], dm, nd)
    Y = (np.abs(r["y"]) + stiffness_ref(*abs_all(D, G, ca, r["xa"]), dm, nd)
         + stiffness_ref(*abs_all(D, G, cb, r["xb"]), dm, nd))
    if form == "stiffness2":
        return (y, Y), None
    y = y + mass_ref(r["xb"] ** 2, c5, detJ, dm, nd)
    Y = Y + mass_ref(r["xb"] ** 2, np.abs(c5), detJ, dm, nd)
    m = r["m"] + mass_ref(r["xa"], c2, detJ, dm, nd)
    M = np.abs(r["m"]) + mass_ref(*abs_all(r["xa"], c2, detJ), dm, nd)
    return (y, Y), (m, M)


def _cell_launch(torch, P, dt, form, geo, h, g, flags=0, null_detjc=False):
    """Launch one cell kernel on cells g['sl']; returns (rc, y, m) with y, m the device buffers."""
    L = _lib()
    S_ = np.dtype(dt).itemsize
    off, Nd = g["sl"].start, g["Nd"]
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    keep = []

    def cell_ptr(a, per_cell):  # pointer to row ``off`` of a per-cell array
        t = a if isinstance(a, torch.Tensor) else dv(a)
        keep.append(t)
        return t.data_ptr() + off * per_cell * t.element_size()

    y, m = Dev(torch, h["y"], seed=1), Dev(torch, h["m"], seed=2)
    xa, xb = dv(h["xa"]), dv(h["xb"])
    keep += [xa, xb]
    args_c = [cell_ptr(h[k], 1) for k in ("ca", "cb", "c2", "c5")]
    dmp = cell_ptr(h["dofmap"], Nd)
    D = h["D"]
    st = torch.cuda.current_stream().cuda_stream
    if geo == "rect":
        L.check(L.fn("fus_set_rect_tables", dt)(P, h["k1"].ctypes.data, h["w1"].ctypes.data, st))
    if geo == "streamed":
        # G placed so that the launched pointer (row ``off``) sits gshift bytes past a 16-byte boundary
        per = 16 // S_
        pad = ((g["gshift"] // S_) - off * Nd * 6) % per
        flat = np.concatenate([np.zeros(pad, dt), h["G"].ravel(), np.zeros(per, dt)])
        Gt = dv(flat)
        keep.append(Gt)
        Gp = Gt.data_ptr() + (pad + off * Nd * 6) * S_
        assert Gp % 16 == g["gshift"]
        dJ = cell_ptr(h["detJ"], Nd)
    else:
        Gp, dJ = cell_ptr(h["Gc"], 6), cell_ptr(h["detJc"], 1)
        if null_detjc:
            dJ = None
    ca, cb, c2, c5 = args_c
    nc = g["sl"].stop - off
    tail = [dmp, D.ctypes.data, nc, P, flags, st]
    if form == "stiffness2":
        name = {"streamed": "fus_stiffness2", "affine": "fus_stiffness2_affine", "rect": "fus_stiffness2_rect"}[geo]
        args = [xa.data_ptr(), ca, xb.data_ptr(), cb, y.ptr, Gp]
    else:
        name = {"streamed": "fus_stiffness_westervelt", "affine": "fus_stiffness_westervelt_affine",
                "rect": "fus_stiffness_westervelt_rect"}[geo]
        args = [xa.data_ptr(), ca, xb.data_ptr(), cb, c2, c5, m.ptr, y.ptr, Gp, dJ]
    if geo == "affine":
        wq = dv(h["wq"])
        keep.append(wq)
        args.append(wq.data_ptr())
    rc = L.fn(name, dt)(*args, *tail)
    torch.cuda.synchronize()
    return rc, y, m


def _run_cell_case(torch, P, dt, form, geo, nc, off, seed, gshift=0, mutations=None):
    h, r, g = _cell_case(P, dt, form, geo, nc, off, seed, gshift)
    rc, y, m = _cell_launch(torch, P, dt, form, geo, h, g)
    assert rc == 0, _lib().lib().fus_last_error()
    k = _k_cell(P + 1)
    (yr, Y), mm = _cell_refs(r, g, form)
    yo = y.get()
    fam = f"{form}_{geo}"
    check_bound(yo, yr, Y, k, dt, fam)
    mo = m.get()
    if mm is None:
        assert _bits_equal(mo, h["m"])  # the dual form has no m
    else:
        check_bound(mo, mm[0], mm[1], k, dt, fam + "_m")
    if mutations is None:
        mutations = ["cb", "last"] + (["swapG"] if geo != "rect" else []) + (["c5", "c2"] if form != "stiffness2" else [])
    for mu in mutations:
        (ym, _), mmu = _cell_refs(r, g, form, mu)
        if mu == "c2":
            assert violates(mo, mmu[0], mm[1], k, dt), f"{fam}: m is within the bound of a reference without c2"
        else:
            assert violates(yo, ym, Y, k, dt), f"{fam}: y is within the bound of a reference with mutation {mu}"


@pytest.mark.gpu
@pytest.mark.parametrize("geo", ["streamed", "affine", "rect"])
@pytest.mark.parametrize("form", ["stiffness2", "westervelt"])
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("P", range(2, 8))
def test_cell_kernel_vs_float64_reference(P, dt, form, geo):
    """Cell counts 1, B-1, B, B+1 (B cells per batch) launched on a sub-range of the arrays;
    the streamed forms also with G one element off 16 bytes (no bulk copies) and, in float32,
    8 bytes off (bulk copies with a shifted batch)."""
    torch = _torch_cuda()
    B = cells_per_batch()[(np.dtype(dt), P + 1)]
    shifts = [0] if geo != "streamed" else ([0, 8] if np.dtype(dt).itemsize == 8 else [0, 4, 8])
    for i, nc in enumerate(sorted({1, max(B - 1, 1), B, B + 1})):
        for gshift in shifts:
            _run_cell_case(torch, P, dt, form, geo, nc, off=3, seed=100 * P + 10 * i + gshift, gshift=gshift)


@pytest.mark.gpu
@pytest.mark.parametrize("geo", ["streamed", "affine", "rect"])
@pytest.mark.parametrize("form", ["stiffness2", "westervelt"])
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("P", [2, 4])
def test_cell_kernel_many_batches_per_cta(P, dt, form, geo):
    """Enough cells that every persistent CTA runs at least three batches (the prefetch registers
    rotate once per batch): at most 16 CTAs of 128 threads fit on an SM."""
    torch = _torch_cuda()
    B = cells_per_batch()[(np.dtype(dt), P + 1)]
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    nc = nsm * 16 * B * 3 + 1
    _run_cell_case(torch, P, dt, form, geo, nc, off=0, seed=P, mutations=["last"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_cell_kernel_argument_checks(dt):
    """FUS_NO_ATOMICS with a Westervelt form and a null detJc are refused before any launch."""
    torch = _torch_cuda()
    L = _lib()
    for geo in ("streamed", "affine", "rect"):
        h, r, g = _cell_case(3, dt, "westervelt", geo, 4, 0, 1)
        before = L.lib().fus_launch_count()
        rc, y, m = _cell_launch(torch, 3, dt, "westervelt", geo, h, g, flags=L.FUS_NO_ATOMICS)
        assert rc == BAD_ARGUMENT
        if geo != "streamed":
            rc, y, m = _cell_launch(torch, 3, dt, "westervelt", geo, h, g, null_detjc=True)
            assert rc == BAD_ARGUMENT
        assert L.lib().fus_launch_count() == before
        assert _bits_equal(y.get(), h["y"]) and _bits_equal(m.get(), h["m"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("P", range(2, 8))
def test_mass_kernels_vs_float64_reference(P, dt):
    """fus_mass on cells (ncols = n^3) and facets (ncols = n^2) and fus_westervelt_mass on cells,
    into nonzero y / m / b, through row-offset pointers.  k = 3 roundings per contribution + the
    number of contributions to the dof (atomics in any order) + 1."""
    torch = _torch_cuda()
    L = _lib()
    n = P + 1
    rng = np.random.default_rng(P)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    st = torch.cuda.current_stream().cuda_stream
    S_ = np.dtype(dt).itemsize
    for ncols, nent in ((n**3, 37), (n**2, 301)):
        if ncols == n**3:
            dm, nd = box_dofmap(nent + 2, P, P)
        else:
            nd = 4 * nent
            dm = rng.integers(0, nd, (nent + 2, ncols)).astype(np.int32)
        off = 2
        x, w = rng.standard_normal(nd).astype(dt), rng.standard_normal(nd).astype(dt)
        c = (rng.uniform(0.5, 2, nent + 2) * rng.choice([-1, 1], nent + 2)).astype(dt)
        c5 = (rng.uniform(0.5, 2, nent + 2) * rng.choice([-1, 1], nent + 2)).astype(dt)
        detJ = rng.uniform(0.5, 2, (nent + 2, ncols)).astype(dt)
        y0, b0 = rng.standard_normal(nd).astype(dt), rng.standard_normal(nd).astype(dt)
        xd, wd, cd, c5d, dJd, dmd = dv(x), dv(w), dv(c), dv(c5), dv(detJ), dv(dm)
        y, m, b = Dev(torch, y0, seed=1), Dev(torch, y0, seed=2), Dev(torch, b0, seed=3)
        L.check(L.fn("fus_mass", dt)(xd.data_ptr(), cd.data_ptr() + off * S_, y.ptr, dJd.data_ptr() + off * ncols * S_,
                                     dmd.data_ptr() + off * ncols * 4, nent, ncols, st))
        if ncols == n**3:
            L.check(L.fn("fus_westervelt_mass", dt)(xd.data_ptr(), wd.data_ptr(), cd.data_ptr() + off * S_,
                                                    c5d.data_ptr() + off * S_, m.ptr, b.ptr,
                                                    dJd.data_ptr() + off * ncols * S_, dmd.data_ptr() + off * ncols * 4,
                                                    nent, ncols, st))
        torch.cuda.synchronize()
        sl = slice(off, off + nent)
        f = lambda a: np.asarray(a, np.float64)  # noqa: E731
        dms, dJs = dm[sl], f(detJ[sl])
        k = 5 + int(np.bincount(dms.ravel(), minlength=nd).max())
        yo = y.get()
        yr = f(y0) + mass_ref(f(x), f(c[sl]), dJs, dms, nd)
        Y = np.abs(f(y0)) + mass_ref(*abs_all(f(x), f(c[sl]), dJs), dms, nd)
        check_bound(yo, yr, Y, k, dt, "mass")
        assert violates(yo, f(y0) + mass_ref(f(x), f(c[sl][:-1]), dJs[:-1], dms[:-1], nd), Y, k, dt)
        if ncols == n**3:
            mo, bo = m.get(), b.get()
            check_bound(mo, yr, Y, k, dt, "westervelt_mass")
            br = f(b0) + mass_ref(f(w) ** 2, f(c5[sl]), dJs, dms, nd)
            Bm = np.abs(f(b0)) + mass_ref(f(w) ** 2, np.abs(f(c5[sl])), dJs, dms, nd)
            check_bound(bo, br, Bm, k + 1, dt, "westervelt_mass")
            assert violates(bo, f(b0), Bm, k + 1, dt)
        else:
            assert _bits_equal(m.get(), y0) and _bits_equal(b.get(), b0)


# --------------------------------------------------------------------------- #
# GPU: stage kernels
# --------------------------------------------------------------------------- #
def _lengths(dt):
    W = PACK[np.dtype(dt)]
    # 2^22 + 3: n / W is above the grid cap of 8 blocks of 256 threads per SM in both types
    return sorted({0, 1, W - 1, W, W + 1, 1023, 2**22 + 3})


def _mask(n, seed):
    """Random skip mask of whole aligned groups of 4 dofs; the group holding the last dof is set."""
    rng = np.random.default_rng(seed)
    groups = rng.random((n + 3) // 4) < 0.4
    if groups.size:
        groups[-1] = True
    bits = np.repeat(groups, 4)[:n]
    return bits, np.packbits(bits.astype(np.uint8), bitorder="little")


STAGE_VECS = {
    "open": ["u", "v", "u0", "v0", "ku", "kv", "un", "b"],
    "lin": ["u", "v", "u0", "v0", "ku", "kv", "un", "b", "m"],
    "west": ["u", "v", "u0", "v0", "ku", "kv", "un", "b", "m", "m0"],
    "pw": ["u", "v", "u0", "v0", "ku", "kv", "un", "b", "m0", "m2", "m5"],
    "leap": ["u", "v", "b", "m"],
}


def _stage_inputs(form, n, dt, seed, mode=None):
    rng = np.random.default_rng(seed)
    x = {k: rng.standard_normal(n, dtype=dt) for k in STAGE_VECS[form]}
    if form in ("lin", "leap"):
        x["m"] = rng.uniform(0.5, 2.0, n).astype(dt)
    if form == "west":  # m: the state-dependent part, m0 the lumped mass
        x["m"] = rng.uniform(-0.5, 0.5, n).astype(dt)
        x["m0"] = rng.uniform(2.0, 4.0, n).astype(dt)
    if form == "pw":
        x["m0"] = rng.uniform(2.0, 4.0, n).astype(dt)
        x["m2"] = rng.uniform(-0.5, 0.5, n).astype(dt)
        x["m5"] = rng.uniform(-1.0, 1.0, n).astype(dt)
        x["un"] = np.clip(x["un"], -2, 2)
        x["u0"] = np.clip(x["u0"], -2, 2)
    if mode == 3:  # not read: a read would leave NaN behind
        for k in ("u", "v", "ku", "un"):
            x[k][:] = np.nan
    elif form in ("lin", "west"):
        x["un"][:] = np.nan  # written, never read
    return x


def _stage_call(torch, form, dt, x, mode, n, shift, mask, kv_null, first=1, step=None,
                adt=0.37, bdt=0.21):
    """Run one open / close launch on guarded copies of ``x``; returns (rc, {name: Dev})."""
    L = _lib()
    d = {k: Dev(torch, v, shift=shift, seed=i) for i, (k, v) in enumerate(x.items())}
    p = lambda k: d[k].ptr if k in d else None  # noqa: E731
    st = torch.cuda.current_stream().cuda_stream
    mk = None
    if mask is not None:
        mt = torch.from_numpy(mask).cuda()
        d["_mask"] = mt
        mk = mt.data_ptr()
    sp = step.data_ptr() if step is not None else None
    kv = None if kv_null else p("kv")
    if form == "open":
        rc = L.fn("fus_rk_open", dt)(p("u"), p("v"), p("u0"), p("v0"), p("ku"), p("kv"), p("un"), p("b"), adt, first, n, st)
    elif form == "lin":
        rc = L.fn("fus_rk_close", dt)(p("u"), p("v"), p("u0"), p("v0"), p("ku"), kv, p("un"), p("b"), p("m"), bdt, adt,
                                      mode, n, sp, mk, st)
    elif form == "west":
        rc = L.fn("fus_rk_close_westervelt", dt)(p("u"), p("v"), p("u0"), p("v0"), p("ku"), kv, p("un"), p("b"), p("m"),
                                                 p("m0"), bdt, adt, mode, n, sp, mk, st)
    elif form == "pw":
        rc = L.fn("fus_rk_close_westervelt_pw", dt)(p("u"), p("v"), p("u0"), p("v0"), p("ku"), kv, p("un"), p("b"),
                                                    p("m0"), p("m2"), p("m5"), bdt, adt, mode, n, sp, mk, st)
    else:
        rc = L.fn("fus_leapfrog_close", dt)(p("u"), p("v"), p("b"), p("m"), bdt, adt, n, sp, mk, st)
    torch.cuda.synchronize()
    return rc, d


def _check_stage(form, dt, x, d, mode, bits, kv_null, first, adt, bdt):
    f = {k: np.asarray(v, np.float64) for k, v in x.items()}
    if form == "open":
        ref = open_ref(f, _t(dt, adt), first)
    else:
        ref = close_ref(f, form, _t(dt, bdt), _t(dt, adt), mode if form != "leap" else 4, kv_stored=not kv_null)
    out = {k: v.get() for k, v in d.items() if not k.startswith("_")}
    keep = bits if bits is not None else np.zeros(next(iter(x.values())).size, bool)
    fam = "open" if form == "open" else f"close_{form}"
    for k, o in out.items():
        assert _bits_equal(o[keep], x[k][keep]), f"{fam}: {k} changed at a masked dof"
        if k not in ref:
            assert _bits_equal(o, x[k]), f"{fam} mode {mode}: {k} written"
            continue
        sel = ~keep
        check_bound(o[sel], ref[k].v[sel], ref[k].m[sel], K_ELEM, dt, fam)
    # copies are copies, zeros are zeros
    free = ~keep
    if form == "open" and first:
        assert _bits_equal(out["u0"], x["u"]) and _bits_equal(out["v0"], x["v"])
    if form != "leap" and mode == 2:
        for a, b_ in (("u0", "u"), ("v0", "v"), ("un", "u"), ("ku", "v")):
            assert _bits_equal(out[a][free], out[b_][free])
    if "b" in ref:
        assert np.all(out["b"][free] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("form,mode", [("open", 0), ("open", 1)] + [(f, m) for f in ("lin", "west", "pw") for m in range(5)]
                         + [("leap", 4)])
def test_stage_kernel_vs_float64_reference(form, mode, dt):
    """Every length of ``_lengths`` on the vector path (16-byte aligned pointers) and the scalar
    path (one element off), without and with a skip mask; guards around every vector, masked dofs
    and unwritten vectors bit-identical; kv == NULL in the chained modes when masked; step_dev
    moves by one per launch exactly in modes 2 and 4 (for n == 0 too).  ``mode`` is ``first`` for
    the open kernel."""
    torch = _torch_cuda()
    lengths = _lengths(dt)
    for n in lengths:
        for shift in (0, 1):
            for masked in (False, True):
                if masked and form == "open":
                    continue
                if n == lengths[-1] and masked != (shift == 1) and form != "open":
                    continue  # the longest vector: unmasked on the vector path, masked on the scalar path
                bits, mask = _mask(n, n + shift) if masked else (None, None)
                x = _stage_inputs(form, n, dt, seed=n + 17 * shift + mode, mode=None if form == "open" else mode)
                kv_null = masked and form != "open" and form != "leap" and mode != 0
                step = torch.tensor([5], dtype=torch.int64, device="cuda")
                adt, bdt = 0.37, 0.21
                rc, d = _stage_call(torch, form, dt, x, mode, n, shift, mask, kv_null, first=mode, step=step,
                                    adt=adt, bdt=bdt)
                assert rc == 0, _lib().lib().fus_last_error()
                _check_stage(form, dt, x, d, mode, bits, kv_null, mode, adt, bdt)
                counts = form == "leap" or (form != "open" and mode in (2, 4))
                assert int(step.item()) == (6 if counts else 5), f"{form} mode {mode} n {n}: step_dev {int(step.item())}"


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_empty_close_still_counts_the_step(dt):
    """n == 0 with a step counter in modes 2 / 4 (a rank whose owned dofs are all shared, closed
    by fus_rk_close_shared) advances step_dev, which selects the source row of the next step."""
    torch = _torch_cuda()
    x = {k: np.zeros(0, dt) for vecs in STAGE_VECS.values() for k in vecs}
    for form, modes in (("lin", range(5)), ("west", range(5)), ("pw", range(5)), ("leap", [4])):
        for mode in modes:
            step = torch.zeros(1, dtype=torch.int64, device="cuda")
            xs = {k: x[k] for k in STAGE_VECS[form]}
            for _ in range(3):
                rc, _d = _stage_call(torch, form, dt, xs, mode, 0, 0, None, False, step=step)
                assert rc == 0
            want = 3 if mode in (2, 4) else 0
            assert int(step.item()) == want, f"{form} mode {mode}: step_dev {int(step.item())} after 3 launches"


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_stage_kernel_argument_checks(dt):
    """next_mode 5, mode 0 without kv and a null pointwise mass are refused before any launch."""
    torch = _torch_cuda()
    L = _lib()
    n = 64
    before = L.lib().fus_launch_count()
    for form in ("lin", "west", "pw"):
        x = _stage_inputs(form, n, dt, 1)
        rc, d = _stage_call(torch, form, dt, x, 5, n, 0, None, False)
        assert rc == BAD_ARGUMENT
        rc, d = _stage_call(torch, form, dt, x, 0, n, 0, None, True)
        assert rc == BAD_ARGUMENT
        for k, v in d.items():
            assert _bits_equal(v.get(), x[k])
    x = _stage_inputs("pw", n, dt, 2)
    for missing in ("m0", "m2", "m5"):
        for nn in (0, n):
            xs = {k: v for k, v in x.items() if k != missing}
            step = torch.zeros(1, dtype=torch.int64, device="cuda")
            rc, d = _stage_call(torch, "pw", dt, xs, 2, nn, 0, None, False, step=step)
            assert rc == BAD_ARGUMENT and int(step.item()) == 0
    assert L.lib().fus_launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_ping_pong_steps_equal_open_and_chained_closes(dt):
    """The ping-pong sequence 3/1/1/4 with base / accumulator swaps makes the same arithmetic bit
    for bit as open(first, a_0 = 0) followed by 1/1/1/2, for every close form."""
    torch = _torch_cuda()
    L = _lib()
    n, nsteps, dtime = 4099, 3, 0.013
    a_rk, b_rk = (0.0, 0.5, 0.5, 1.0), (1 / 6, 1 / 3, 1 / 3, 1 / 6)
    st = torch.cuda.current_stream().cuda_stream
    tt = torch.float64 if np.dtype(dt) == np.float64 else torch.float32
    rng = np.random.default_rng(5)
    for form in ("lin", "west", "pw"):
        h = lambda lo, hi: torch.from_numpy(rng.uniform(lo, hi, n).astype(dt)).cuda()  # noqa: E731
        u_init, v_init = h(-1, 1), h(-1, 1)
        m, m0, m2, m5 = h(0.5, 2), h(2, 4), h(-0.3, 0.3), h(-1, 1)
        mass = {"lin": [m], "west": [None, m0], "pw": [m0, m2, m5]}[form]
        wm = torch.zeros(n, dtype=tt, device="cuda")

        def bfun(b, un, vn):
            b.copy_(-0.7 * un + 0.3 * vn + 0.1 * un * vn)
            if form == "west":  # the cell form accumulates a state-dependent mass beside b
                wm.copy_(0.2 * un)

        def close(u, v, u0, v0, ku, kv, un, b, bdt, adt, mode):
            ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
            masses = [ptr(wm) if t is None else ptr(t) for t in mass]
            name = {"lin": "fus_rk_close", "west": "fus_rk_close_westervelt", "pw": "fus_rk_close_westervelt_pw"}[form]
            L.check(L.fn(name, dt)(ptr(u), ptr(v), ptr(u0), ptr(v0), ptr(ku), ptr(kv), ptr(un), ptr(b), *masses,
                                   bdt, adt, mode, n, None, None, st), name)

        z = lambda: torch.zeros(n, dtype=tt, device="cuda")  # noqa: E731
        # open + 1/1/1/2
        u, v, u0, v0, ku, kv, un, b = u_init.clone(), v_init.clone(), z(), z(), z(), z(), z(), z()
        for _ in range(nsteps):
            L.check(L.fn("fus_rk_open", dt)(u.data_ptr(), v.data_ptr(), u0.data_ptr(), v0.data_ptr(), ku.data_ptr(),
                                            kv.data_ptr(), un.data_ptr(), b.data_ptr(), 0.0, 1, n, st))
            for s in range(4):
                bfun(b, un, ku)
                close(u, v, u0, v0, ku, kv, un, b, b_rk[s] * dtime, a_rk[s + 1] * dtime if s < 3 else 0.0,
                      1 if s < 3 else 2)
        # ping-pong: the first stage's input is the base state itself
        base, acc = [u_init.clone(), v_init.clone()], [z(), z()]
        ku2, un2, b2 = z(), z(), z()
        for _ in range(nsteps):
            for s in range(4):
                bfun(b2, *(base if s == 0 else (un2, ku2)))
                close(acc[0], acc[1], base[0], base[1], ku2, None, un2, b2, b_rk[s] * dtime,
                      a_rk[s + 1] * dtime if s < 3 else 0.0, (3, 1, 1, 4)[s])
            base, acc = acc, base
        torch.cuda.synchronize()
        assert torch.equal(base[0], u) and torch.equal(base[1], v), form
        assert not torch.equal(u, u_init)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", TYPES, ids=["f64", "f32"])
def test_boundary_terms_vs_float64_reference(dt):
    """Every null / non-null combination of src, src2, absb; scalar amplitudes and table rows
    selected by step_dev (NULL: row 0) with non-trivial gstride / goff; n = 0; b off the dof list
    bit-identical."""
    torch = _torch_cuda()
    L = _lib()
    rng = np.random.default_rng(9)
    st = torch.cuda.current_stream().cuda_stream
    nd = 5000
    b0, vn = rng.standard_normal(nd).astype(dt), rng.standard_normal(nd).astype(dt)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    vnd = dv(vn)
    tab = rng.standard_normal(7 * 11 + 4).astype(dt)
    tabd = dv(tab)
    g, dg = 0.83, -1.27
    for nb in (0, 1, 1023, 3001):
        dof = np.sort(rng.choice(nd, nb, replace=False)).astype(np.int32)
        rng.shuffle(dof)
        dofd = dv(dof)
        terms = {k: rng.standard_normal(nb).astype(dt) for k in ("src", "src2", "absb")}
        termd = {k: dv(v) for k, v in terms.items()}
        for combo in range(8):
            use = {k: bool(combo >> i & 1) for i, k in enumerate(("src", "src2", "absb"))}
            tp = {k: (termd[k].data_ptr() if use[k] else None) for k in termd}
            for amp in ("scalar", "row", "row0"):
                cases = [(None, 8, 0)] if amp == "scalar" else ([(s, 11, o) for s in (0, 3, 6) for o in (1, 4)]
                                                                  if amp == "row" else [(None, 11, 5)])
                for s, gstride, goff in cases:
                    b = Dev(torch, b0, seed=combo)
                    step = torch.tensor([s], dtype=torch.int64, device="cuda") if s is not None else None
                    rc = L.fn("fus_boundary_terms", dt)(
                        b.ptr, vnd.data_ptr(), dofd.data_ptr(), tp["src"], tp["src2"], tp["absb"], g, dg,
                        tabd.data_ptr() if amp != "scalar" else None, step.data_ptr() if step is not None else None,
                        gstride, goff, nb, st)
                    assert rc == 0
                    torch.cuda.synchronize()
                    if amp == "scalar":
                        ga, dga = _t(dt, g), _t(dt, dg)
                    else:
                        row = s if s is not None else 0
                        ga, dga = float(tab[row * gstride + goff]), float(tab[row * gstride + goff + 1])
                    f = lambda a: np.asarray(a, np.float64)  # noqa: E731
                    ref = boundary_ref(f(b0), f(vn), dof, *(f(terms[k]) if use[k] else None for k in terms), ga, dga)
                    out = b.get()
                    off = np.ones(nd, bool)
                    off[dof] = False
                    assert _bits_equal(out[off], b0[off])
                    check_bound(out, ref.v, ref.m, K_ELEM, dt, "boundary_terms")
                    if nb and use["src"] and amp == "row":
                        wrong = boundary_ref(f(b0), f(vn), dof, *(f(terms[k]) if use[k] else None for k in terms),
                                             float(tab[goff]), float(tab[goff + 1]))
                        assert s == 0 or violates(out, wrong.v, ref.m, K_ELEM, dt), "table row ignores step_dev"
