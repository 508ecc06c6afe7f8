// Shared by stiffness.cu (G streamed through the TMA ring) and stiffness_affine.cu
// (affine cells, G = wq x Gc): the kernel template, its layouts and launch helpers.
// Each translation unit gets its own copy of the __constant__ derivative tables.
#pragma once

#include "halo_internal.cuh"

namespace {

__constant__ double c_D64[6][64];
__constant__ float c_D32[6][64];
// rectilinear cells (GEO == 2): 1-D stiffness matrix K1 = D^T diag(w1) D and the 1-D weights
__constant__ double c_K64[6][64];
__constant__ float c_K32[6][64];
__constant__ double c_W64[6][8];
__constant__ float c_W32[6][8];
// trilinear cells (GEO == 3): the 1-D quadrature points, in dof order (and the 1-D weights above)
__constant__ double c_X64[6][8];
__constant__ float c_X32[6][8];

template <typename T, int P>
struct DTable;
template <int P>
struct DTable<double, P> {
  static __device__ __forceinline__ double at(int i) { return c_D64[P - 2][i]; }
};
template <int P>
struct DTable<float, P> {
  static __device__ __forceinline__ float at(int i) { return c_D32[P - 2][i]; }
};
template <typename T, int P>
struct KTable;
template <int P>
struct KTable<double, P> {
  static __device__ __forceinline__ double at(int i) { return c_K64[P - 2][i]; }
  static __device__ __forceinline__ double w(int i) { return c_W64[P - 2][i]; }
  static __device__ __forceinline__ double x(int i) { return c_X64[P - 2][i]; }
};
template <int P>
struct KTable<float, P> {
  static __device__ __forceinline__ float at(int i) { return c_K32[P - 2][i]; }
  static __device__ __forceinline__ float w(int i) { return c_W32[P - 2][i]; }
  static __device__ __forceinline__ float x(int i) { return c_X32[P - 2][i]; }
};

// cells per CTA batch / threads per CTA / min CTAs per SM, per (n, sizeof T)
template <typename T, int n>
struct Cfg;
#define FUS_CFG(TYPE, N, BCELLS, THREADS_, MINB_)       \
  template <>                                           \
  struct Cfg<TYPE, N> {                                 \
    static constexpr int B = BCELLS;                    \
    static constexpr int THREADS = THREADS_;            \
    static constexpr int MINB = MINB_;                  \
  };
// (measured on B200, tools/sweep.py: 256-thread CTAs only pay where n^2 packs badly into 128)
FUS_CFG(double, 3, 14, 128, 4)
FUS_CFG(double, 4, 8, 128, 3)
FUS_CFG(double, 5, 5, 128, 3)
FUS_CFG(double, 6, 3, 128, 3)
FUS_CFG(double, 7, 5, 256, 1)
FUS_CFG(double, 8, 1, 64, 3)
FUS_CFG(float, 3, 14, 128, 6)
FUS_CFG(float, 4, 8, 128, 6)
FUS_CFG(float, 5, 5, 128, 5)
FUS_CFG(float, 6, 7, 256, 2)
FUS_CFG(float, 7, 2, 128, 4)
FUS_CFG(float, 8, 2, 128, 3)
#undef FUS_CFG

constexpr int kStages = 2;

constexpr int ceil_cong(int lo, int r, int M) {  // smallest v >= lo with v = r (mod M)
  return lo + (((r - lo) % M) + M) % M;
}

template <typename T, int n>
struct Layout {
  static constexpr int S = (int)sizeof(T);
  static constexpr int B = Cfg<T, n>::B;
  static constexpr int N2 = n * n;
  static constexpr int Nd = n * n * n;
  // tile strides in elements (see header comment); M lanes share a wavefront
  static constexpr int M = S == 8 ? 16 : 32;
  static constexpr int SPY = ceil_cong(N2, n % M, M);
  static constexpr int SCY = n * SPY;
  static constexpr int SPZ = ceil_cong(N2, 1, M);
  static constexpr int SCZ = ceil_cong(n * SPZ, N2 % M, M);
  // G staging: per-cell record block of CB bytes at stride GC bytes
  static constexpr int CB = Nd * 6 * S;
  static constexpr int GC = ceil_cong(CB + 16, (N2 * 6 * S) % 128, 128);
  static constexpr int STAGE = ((B * GC + 32 + 127) / 128) * 128;
  static constexpr int BAR = 128;
  static constexpr int TILE_Y = ((B * SCY * S + 127) / 128) * 128;
  static constexpr int TILE_Z = ((B * SCZ * S + 127) / 128) * 128;
  static constexpr int SMEM = BAR + kStages * STAGE + TILE_Y + TILE_Z;
  static constexpr int SMEM_AFF = BAR + TILE_Y + TILE_Z;  // affine cells: no G staging ring
  // trilinear cells: 36 tangent coefficients per cell, two batches (this one, the next)
  static constexpr int TCREC = 36;
  static constexpr int TCBUF = ((B * TCREC * S + 127) / 128) * 128;
  static constexpr int SMEM_TRI = SMEM_AFF + 2 * TCBUF;
};

template <typename T>
struct StiffArgs {
  const T* xa;
  const T* ca;
  const T* xb;  // dual mode only
  const T* cb;
  T* y;
  const T* G;
  const int32_t* dofmap;
  // Westervelt mode only
  const T* detJ;
  const T* cm;
  const T* cy;
  T* m;
  // affine-cell mode only: G[c,q,:] = wq[q] * Gc[c,:], detJ[c,q] = wq[q] * detJc[c]
  const T* Gc;
  const T* wq;
  const T* detJc;
  // trilinear-cell mode only: Tc[c, d, m, :] (36 values per cell), the tangent of reference
  // direction d as a bilinear function of the other two coordinates (u, v):
  //   t_d = Tc[d,0] + u Tc[d,1] + v Tc[d,2] + u v Tc[d,3]
  const T* Tc;
  long long ncells;
  int bulk_ok;  // G base aligned for the 2-element vector loads of the AoS records
  // multi-GPU (WAIT instantiations): cells [wait_from, ncells) of this launch touch ghost dofs.
  // Before a CTA gathers for its first such batch it waits until every owner of this rank's ghosts
  // has raised its FWD epoch (their halo put has landed): the forward exchange overlaps the
  // interior cells of the SAME launch, no second launch, no second pipeline fill and drain.
  const unsigned long long* wait_row;  // this rank's FWD flag row
  const int* wait_src;                 // owner ranks
  int wait_nsrc;
  unsigned long long* wait_ctr;        // the handle's counters (FUS_CTR_FWD_WAITED is read, never written here)
  long long wait_from;
};

// Gathers of x in a WAIT instantiation.  While a CTA works on interior cells it reads owned dofs
// only and uses the read-only path (__ldg, LDG.CONSTANT - measured 3 % faster for this gather than
// plain loads).  The neighbours write the ghost entries of x while the kernel runs, so once the
// CTA has passed the halo wait every gather goes to L2 (__ldcg): a line cached in L1 before the
// put landed (an interior cell gathering the owned dofs next to the first ghost entry) can never
// be served.  Interface cells are a few per cent of the cells.
template <typename T>
struct G6 {
  T g0, g1, g2, g3, g4, g5;
};

// 6 geometric factors of one quadrature point from shared memory
__device__ __forceinline__ G6<double> load_g6(const double* p) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  const double2 c = *reinterpret_cast<const double2*>(p + 4);
  return {a.x, a.y, b.x, b.y, c.x, c.y};
}
__device__ __forceinline__ G6<float> load_g6(const float* p) {
  const float2 a = *reinterpret_cast<const float2*>(p);
  const float2 b = *reinterpret_cast<const float2*>(p + 2);
  const float2 c = *reinterpret_cast<const float2*>(p + 4);
  return {a.x, a.y, b.x, b.y, c.x, c.y};
}

// MODE 0: y += K(ca; xa).  MODE 1: y += K(ca; xa) + K(cb; xb) with one read of G.
// MODE 2: MODE 1 plus the Westervelt cell-mass pair on the same gathered pencils:
//         m += M(cm; xa),  y += M(cy; xb^2)   (cuda/demo_nonlinear_bowl.py:609-612, 626-628)
// GEO 0: G streamed through the TMA ring.
// GEO 1 (affine): every cell of the launch has a constant Jacobian, so its 6*n^3 geometric
//   factors are wq[q] * Gc[cell, 0..5]: nothing is streamed but the dofmap, the shared-memory
//   ring and the TMA copies disappear, and the n quadrature weights a thread needs live in
//   registers.
// GEO 2 (rectilinear): affine AND Gc diagonal (axis-aligned box cells) with tensor-product
//   weights: the three directions decouple, y = cc * sum_d g_dd (w x w) (x) K1_d u with the
//   constant 1-D stiffness matrix K1 = D^T diag(w1) D - one n x n product per pencil and
//   direction, the y / z pencils are transformed in place (8 tile passes instead of 16, two
//   barriers instead of five).
// GEO 3 (trilinear): nothing is streamed but the dofmap and 36 coefficients per cell; the geometric
//   factors are RECOMPUTED at every quadrature point from the cell's trilinear map.  Along the x
//   pencil a thread owns, the tangent t_0 is constant and t_1, t_2 are affine in the pencil
//   coordinate, so a point costs 6 FMAs for the tangents, three cross products c_a (the rows of
//   adj J), det = t_0 . c_0, one division, and the product
//       f_a = (w / |det|) c_a . (g_0 c_0 + g_1 c_1 + g_2 c_2)         ( = sum_b G_ab g_b )
//   without ever forming G: ~60 flops per point against 6 streamed values.
//   MODE 2 takes w |det| of the same point for the cell-mass pair: cm xa and cy xb^2 are kept per
//   point from the gather until the transform loop, where m and the x-pencil sum receive them.
template <typename T, int n, int MODE, bool ATOMIC, int GEO, bool WAIT>
__global__ void __launch_bounds__(Cfg<T, n>::THREADS, Cfg<T, n>::MINB)
    stiffness_kernel(const StiffArgs<T> a) {
  constexpr bool TRI = GEO == 3;
  constexpr bool AFF = GEO == 1 || GEO == 2;
  constexpr bool NOSTREAM = GEO >= 1;  // no G ring (AFF or TRI)
  constexpr bool RECT = GEO == 2;
  constexpr bool DUAL = MODE >= 1;
  constexpr bool WEST = MODE == 2;
  using L = Layout<T, n>;
  using D = DTable<T, n - 1>;
  constexpr int B = L::B;
  constexpr int Nd = L::Nd;
  constexpr int N2 = L::N2;
  constexpr int THREADS = Cfg<T, n>::THREADS;
  static_assert(B * N2 <= THREADS, "one thread per (cell, j, k)");
  static_assert(B <= 32, "one lane of warp 0 per bulk copy");

  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  constexpr int RING = NOSTREAM ? 0 : kStages * L::STAGE;
  unsigned char* stages = smem + L::BAR;
  T* UY = reinterpret_cast<T*>(smem + L::BAR + RING);
  T* UZ = reinterpret_cast<T*>(smem + L::BAR + RING + L::TILE_Y);
  unsigned char* const tcb = smem + L::BAR + L::TILE_Y + L::TILE_Z;  // TRI: two coefficient buffers
  (void)tcb;

  const int tid = threadIdx.x;
  const int cs = tid / N2;  // cell slot within the batch
  const int t2 = tid - cs * N2;
  const int ra = t2 / n;  // the two pencil coordinates this thread plays
  const int rb = t2 - ra * n;
  const bool lane_ok = cs < B;

  // tile bases for the three ownerships
  T* const uy1 = UY + cs * L::SCY + t2;                  // + i*SPY : (j,k) = (ra,rb)
  T* const uz1 = UZ + cs * L::SCZ + t2;                  // + i*SPZ
  T* const uy2 = UY + cs * L::SCY + ra * L::SPY + rb;    // + j*n   : (i,k) = (ra,rb)
  T* const uz3 = UZ + cs * L::SCZ + rb * L::SPZ + ra * n;  // + k    : (i,j) = (rb,ra)

  const long long nb = (a.ncells + B - 1) / B;
  const long long stride = gridDim.x;

  if constexpr (!NOSTREAM) {
    if (tid == 0) {
#pragma unroll
      for (int s = 0; s < kStages; ++s) mbar_init(&full[s], 1);
      fence_mbar_init();
    }
    __syncthreads();
  }
  T wreg[AFF ? n : 1];  // affine mode: this thread's quadrature weights w[i, j, k], i = 0..n-1
  (void)wreg;
  if constexpr (RECT) {
    using KT = KTable<T, n - 1>;
#pragma unroll
    for (int i = 0; i < n; ++i) wreg[i] = KT::w(i) * (KT::w(ra) * KT::w(rb));
  } else if constexpr (AFF) {
#pragma unroll
    for (int i = 0; i < n; ++i) wreg[i] = lane_ok ? __ldg(a.wq + i * N2 + t2) : T(0);
  }

  // A batch goes through the TMA unit unless it is the last one of the array
  // (ragged, and the 16-byte rounding may read a few bytes past the end).
  auto bulk_eligible = [&](long long b) { return a.bulk_ok && b < nb - 1; };
  auto batch_shift = [&](long long b) {
    return (unsigned)((reinterpret_cast<unsigned long long>(a.G) + (unsigned long long)b * B * L::CB) & 15ull);
  };

  // Called by all 32 lanes of warp 0: lane c issues the copy of cell c (B <= 14),
  // so the B bulk copies of a batch go out in parallel instead of one after another.
  auto issue = [&](long long b, int s) {
    fence_proxy_async_smem();  // generic reads of this stage (previous use) before the refill
    const unsigned long long g0 =
        reinterpret_cast<unsigned long long>(a.G) + (unsigned long long)b * B * L::CB;
    const unsigned shift = (unsigned)(g0 & 15ull);
    unsigned char* st = stages + s * L::STAGE;
    const int c = tid;
    const unsigned long long src = g0 + (unsigned long long)c * L::CB;
    const unsigned long long sa = src & ~15ull, se = (src + L::CB + 15ull) & ~15ull;
    const unsigned bytes = c < B ? (unsigned)(se - sa) : 0u;
    const unsigned total = __reduce_add_sync(0xffffffffu, bytes);
    if (c == 0) mbar_arrive_expect_tx(&full[s], total);
    __syncwarp();
    if (c < B)
      bulk_g2s_hint(st + shift + c * L::GC - (unsigned)(src & 15ull), reinterpret_cast<const void*>(sa),
                    bytes, &full[s], l2_policy_evict_first());
  };

  // ---- register prefetch of the dofmap / x pencil of a batch ----------------
  auto load_dofs = [&](long long b, int (&dof)[n]) {
    const long long cell = b * B + cs;
    if (lane_ok && b < nb && cell < a.ncells) {
      const int32_t* dm = a.dofmap + cell * (long long)Nd + t2;
#pragma unroll
      for (int i = 0; i < n; ++i) dof[i] = __ldg(dm + i * N2);
    } else {
#pragma unroll
      for (int i = 0; i < n; ++i) dof[i] = -1;
    }
  };
  bool waited = false;  // WAIT: this CTA has passed the halo wait (CTA-uniform)
  (void)waited;
  auto load_x = [&](const int (&dof)[n], T (&xa)[n], T (&xb)[n]) {
#pragma unroll
    for (int i = 0; i < n; ++i) {
      xa[i] = T(0);
      if constexpr (DUAL) xb[i] = T(0);
      if (dof[i] >= 0) {
        xa[i] = __ldg(a.xa + dof[i]);
        if constexpr (DUAL) xb[i] = __ldg(a.xb + dof[i]);
      }
    }
  };
  auto load_x_l2 = [&](const int (&dof)[n], T (&xa)[n], T (&xb)[n]) {
#pragma unroll
    for (int i = 0; i < n; ++i) {
      xa[i] = T(0);
      if constexpr (DUAL) xb[i] = T(0);
      if (dof[i] >= 0) {
        xa[i] = __ldcg(a.xa + dof[i]);
        if constexpr (DUAL) xb[i] = __ldcg(a.xb + dof[i]);
      }
    }
  };
  // WAIT: called (by every thread of the CTA) before the x gather of batch `bx`
  unsigned long long expect = 0;
  long long b_wait = 0;
  (void)expect;
  (void)b_wait;
  if constexpr (WAIT) {
    expect = a.wait_ctr[FUS_CTR_FWD_WAITED] + 1ULL;
    b_wait = a.wait_from / B;  // first batch holding an interface cell
  }
  auto halo_wait = [&](long long bx) {
    if constexpr (WAIT) {
      if (!waited && bx >= b_wait) {
        fus_wait_flags(a.wait_row, a.wait_src, a.wait_nsrc, expect, a.wait_ctr);
        waited = true;
      }
    }
  };

  auto load_detj = [&](long long b, T (&dj)[n]) {
    const long long cell = b * B + cs;
    if (lane_ok && b < nb && cell < a.ncells) {
      const T* p = a.detJ + cell * (long long)Nd + t2;
#pragma unroll
      for (int i = 0; i < n; ++i) dj[i] = __ldg(p + i * N2);
    } else {
#pragma unroll
      for (int i = 0; i < n; ++i) dj[i] = T(0);
    }
  };

  // Register pipeline, two batches deep so that no load depends on another load
  // issued in the same batch (the compiler is free to hoist these read-only
  // loads to the top of the loop body):
  //   dof  : this batch (scatter)          xv : this batch's x pencil
  //   dofn : next batch (x gather below)   xvn: next batch's x pencil (in flight)
  //   dofm : the batch after (in flight)
  int dof[n], dofn[n], dofm[n];
  T xv[n], xw[n], xvn[n], xwn[n];  // xw*: second vector in dual mode
  (void)xw;
  (void)xwn;
  T dj[WEST ? n : 1], djn[WEST ? n : 1], bex[WEST ? n : 1];  // Westervelt: detJ pencil, extra b term
  T mx[WEST && TRI ? n : 1];  // Westervelt, trilinear: cm xa until w |det| is known
  (void)dj;
  (void)djn;
  (void)bex;
  (void)mx;

  // Rectilinear mode uses the per-cell scalars right at the top of a batch (the other modes
  // first need them two barriers later), so they ride the register pipeline one batch ahead:
  // [0..2] Gc diagonal, then coeff | (ca, cb) | (ca, cb, cm, cy, detJc).
  constexpr int NCS = RECT ? 3 + (DUAL ? (WEST ? 5 : 2) : 1) : 1;
  T csc[NCS], cscn[NCS];
  (void)csc;
  (void)cscn;
  auto load_cell_scalars = [&](long long b, T* c) {
    if constexpr (RECT) {
      const long long cell = b * B + cs;
      const bool ok = lane_ok && b < nb && cell < a.ncells;
#pragma unroll
      for (int q = 0; q < NCS; ++q) c[q] = T(0);
      if (ok) {
        c[0] = __ldg(a.Gc + cell * 6);
        c[1] = __ldg(a.Gc + cell * 6 + 3);
        c[2] = __ldg(a.Gc + cell * 6 + 5);
        c[3] = __ldg(a.ca + cell);
        if constexpr (DUAL) c[4] = __ldg(a.cb + cell);
        if constexpr (WEST) {
          c[5] = __ldg(a.cm + cell);
          c[6] = __ldg(a.cy + cell);
          c[7] = __ldg(a.detJc + cell);
        }
      }
    }
  };

  // TRI: the coefficient records of a batch (B * 36 values, contiguous in Tc) are fetched one
  // batch ahead by the first threads of the CTA, held in registers through the batch and stored
  // into the other shared buffer at its end
  constexpr int NTC = TRI ? (B * L::TCREC + THREADS - 1) / THREADS : 1;
  T tcn[NTC];
  (void)tcn;
  auto load_tc = [&](long long b) {
    if constexpr (TRI) {
      const long long cell0 = b * B;
      const long long lim = b < nb ? ((a.ncells - cell0) < (long long)B ? (a.ncells - cell0) : (long long)B) * L::TCREC : 0;
#pragma unroll
      for (int q = 0; q < NTC; ++q) {
        const int idx = tid + q * THREADS;
        tcn[q] = idx < lim ? __ldg(a.Tc + cell0 * L::TCREC + idx) : T(0);
      }
    }
  };
  auto store_tc = [&](int buf) {
    if constexpr (TRI) {
      T* dst = reinterpret_cast<T*>(tcb + buf * L::TCBUF);
#pragma unroll
      for (int q = 0; q < NTC; ++q) {
        const int idx = tid + q * THREADS;
        if (idx < B * L::TCREC) dst[idx] = tcn[q];
      }
    }
  };

  // prologue: first batch of this CTA
  load_cell_scalars(blockIdx.x, csc);
  if constexpr (TRI) {
    load_tc(blockIdx.x);
    store_tc(0);  // visible after the first barrier of the loop
  }
  if constexpr (!NOSTREAM) {
    if (tid < 32 && (long long)blockIdx.x < nb && bulk_eligible(blockIdx.x)) issue(blockIdx.x, 0);
  }
  load_dofs(blockIdx.x, dof);
  load_dofs(blockIdx.x + stride, dofn);
  halo_wait(blockIdx.x);
  if (WAIT && waited) {
    load_x_l2(dof, xv, xw);
  } else {
    load_x(dof, xv, xw);
  }
  if constexpr (WEST && !NOSTREAM) load_detj(blockIdx.x, reinterpret_cast<T(&)[n]>(dj));

  int it = 0;
  for (long long b = blockIdx.x; b < nb; b += stride, ++it) {
    const int s = it & 1;
    const long long bn = b + stride;
    // TMA prefetch of the next batch into the other stage (consumed last iteration)
    if constexpr (!NOSTREAM) {
      if (tid < 32 && bn < nb && bulk_eligible(bn)) issue(bn, s ^ 1);
    }
    load_tc(bn);

    unsigned char* st = stages + s * L::STAGE;
    const long long cell0 = b * B;
    const int ncur = (int)((a.ncells - cell0) < (long long)B ? (a.ncells - cell0) : (long long)B);
    const bool active = lane_ok && cs < ncur;
    const bool bulk = !NOSTREAM && bulk_eligible(b);
    const T* Gs = reinterpret_cast<const T*>(st + (bulk ? batch_shift(b) : 0u));
    G6<T> gc = {T(0), T(0), T(0), T(0), T(0), T(0)};  // affine mode: the cell's 6 factors (used after two barriers)
    T djc = T(0);
    (void)gc;
    (void)djc;
    if constexpr (RECT) {
      gc.g0 = csc[0];
      gc.g3 = csc[1];
      gc.g5 = csc[2];
      if constexpr (WEST) djc = csc[7];
    } else if constexpr (AFF) {
      if (active) {
        const T* p = a.Gc + (cell0 + cs) * 6;
        gc = {__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3), __ldg(p + 4), __ldg(p + 5)};
        if constexpr (WEST) djc = __ldg(a.detJc + cell0 + cs);
      }
    } else if constexpr (TRI) {
      // nothing per cell here: the coefficient records are in shared memory
    } else if (!bulk) {
      // tail batch / unaligned base: cooperative loads through the generic proxy
      const T* gsrc = a.G + cell0 * (long long)(Nd * 6);
      T* gdst = reinterpret_cast<T*>(st);
      for (int idx = tid; idx < ncur * Nd * 6; idx += THREADS) {
        const int c = idx / (Nd * 6);
        gdst[c * (L::GC / L::S) + (idx - c * Nd * 6)] = gsrc[idx];
      }
    }

    // in flight during this whole batch: the dofmap entries of the batch after
    // next and the x pencil of the next batch (its entries arrived a batch ago)
    load_dofs(bn + stride, dofm);
    if (bn < nb) halo_wait(bn);
    if (WAIT && waited) {
      load_x_l2(dofn, xvn, xwn);
    } else {
      load_x(dofn, xvn, xwn);
    }
    if constexpr (WEST && !NOSTREAM) load_detj(bn, reinterpret_cast<T(&)[n]>(djn));
    load_cell_scalars(bn, cscn);

    // ---- x pencil (registers) -> tiles; x-direction gradient ----------------
    T gx[n];
    T cc = T(1);
    if (active) {
      if constexpr (DUAL) {
        const T ca = RECT ? csc[3] : a.ca[cell0 + cs], cb = RECT ? csc[NCS > 4 ? 4 : 0] : a.cb[cell0 + cs];
        if constexpr (WEST) {
          const T cm = RECT ? csc[NCS > 5 ? 5 : 0] : a.cm[cell0 + cs];
          const T cy = RECT ? csc[NCS > 6 ? 6 : 0] : a.cy[cell0 + cs];
#pragma unroll
          for (int i = 0; i < n; ++i) {
            if constexpr (TRI) {
              mx[i] = xv[i] * cm;                // times w |det| in the transform loop
              bex[i] = (xw[i] * xw[i]) * cy;
            } else {
              T dji;
              if constexpr (AFF) {
                dji = wreg[i] * djc;
              } else {
                dji = dj[i];
              }
              atomicAdd(a.m + dof[i], xv[i] * dji * cm);   // m += cm detJ un
              bex[i] = (xw[i] * xw[i]) * dji * cy;          // b += cy detJ vn^2 (joins the scatter)
            }
          }
        }
#pragma unroll
        for (int i = 0; i < n; ++i) xv[i] = ca * xv[i] + cb * xw[i];
      } else {
        cc = RECT ? csc[NCS > 3 ? 3 : 0] : a.ca[cell0 + cs];
      }
#pragma unroll
      for (int i = 0; i < n; ++i) {
        uy1[i * L::SPY] = xv[i];
        uz1[i * L::SPZ] = xv[i];
      }
      if constexpr (!RECT) {
#pragma unroll
        for (int i = 0; i < n; ++i) {
          T acc = T(0);
#pragma unroll
          for (int l = 0; l < n; ++l) acc += D::at(i * n + l) * xv[l];
          gx[i] = acc;
        }
      }
    }
    T ry[n];
    if constexpr (RECT) {
      using KT = KTable<T, n - 1>;
      const T wab = KT::w(ra) * KT::w(rb);  // the same product in all three ownerships
      if (active) {
        const T sx = cc * gc.g0 * wab;
#pragma unroll
        for (int i = 0; i < n; ++i) {
          T acc = T(0);
#pragma unroll
          for (int l = 0; l < n; ++l) acc += KT::at(i * n + l) * xv[l];
          if constexpr (WEST) {
            ry[i] = bex[i] + sx * acc;
          } else {
            ry[i] = sx * acc;
          }
        }
      }
      __syncthreads();
      if (active) {  // y pencils (i,k) = (ra,rb) and z pencils (i,j) = (rb,ra), in place
        const T sy = cc * gc.g3 * wab, sz = cc * gc.g5 * wab;
        T u[n];
#pragma unroll
        for (int l = 0; l < n; ++l) u[l] = uy2[l * n];
#pragma unroll
        for (int j = 0; j < n; ++j) {
          T acc = T(0);
#pragma unroll
          for (int l = 0; l < n; ++l) acc += KT::at(j * n + l) * u[l];
          uy2[j * n] = sy * acc;
        }
#pragma unroll
        for (int l = 0; l < n; ++l) u[l] = uz3[l];
#pragma unroll
        for (int k = 0; k < n; ++k) {
          T acc = T(0);
#pragma unroll
          for (int l = 0; l < n; ++l) acc += KT::at(k * n + l) * u[l];
          uz3[k] = sz * acc;
        }
      }
      __syncthreads();
    } else {
    __syncthreads();

    // ---- y pencils (i,k) = (ra,rb); z pencils (i,j) = (rb,ra) ---------------
    T gy[n], gz[n];
    if (active) {
      T u[n];
#pragma unroll
      for (int l = 0; l < n; ++l) u[l] = uy2[l * n];
#pragma unroll
      for (int j = 0; j < n; ++j) {
        T acc = T(0);
#pragma unroll
        for (int l = 0; l < n; ++l) acc += D::at(j * n + l) * u[l];
        gy[j] = acc;
      }
#pragma unroll
      for (int l = 0; l < n; ++l) u[l] = uz3[l];
#pragma unroll
      for (int k = 0; k < n; ++k) {
        T acc = T(0);
#pragma unroll
        for (int l = 0; l < n; ++l) acc += D::at(k * n + l) * u[l];
        gz[k] = acc;
      }
    }
    __syncthreads();  // every pencil has been read: overwrite u with the gradients
    if (active) {
#pragma unroll
      for (int j = 0; j < n; ++j) uy2[j * n] = gy[j];
#pragma unroll
      for (int k = 0; k < n; ++k) uz3[k] = gz[k];
    }
    if (bulk) mbar_wait(&full[s], (uint32_t)((it >> 1) & 1));
    __syncthreads();

    // ---- geometric transform at (i, j, k), (j,k) = (ra,rb); x-direction D^T --
    if (active) {
      const T* Gc = Gs + cs * (L::GC / L::S) + t2 * 6;
#pragma unroll
      for (int l = 0; l < n; ++l) {
        if constexpr (WEST && !TRI) {
          ry[l] = bex[l];
        } else {
          ry[l] = T(0);
        }
      }
      // TRI: the tangents along this thread's pencil (eta, zeta fixed; xi = X[i] varies):
      //   t_0 constant,  t_1 = a1 + xi b1,  t_2 = a2 + xi b2
      T t0[3], a1[3], b1[3], a2[3], b2[3];
      T wab = T(0);
      (void)t0;
      (void)a1;
      (void)b1;
      (void)a2;
      (void)b2;
      (void)wab;
      if constexpr (TRI) {
        using KT = KTable<T, n - 1>;
        const T* tc = reinterpret_cast<const T*>(tcb + (it & 1) * L::TCBUF) + cs * L::TCREC;
        const T eta = KT::x(ra), zeta = KT::x(rb);
        const T ez = eta * zeta;
        wab = cc * (KT::w(ra) * KT::w(rb));
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          t0[c] = tc[c] + eta * tc[3 + c] + zeta * tc[6 + c] + ez * tc[9 + c];
          a1[c] = tc[12 + c] + zeta * tc[18 + c];
          b1[c] = tc[15 + c] + zeta * tc[21 + c];
          a2[c] = tc[24 + c] + eta * tc[30 + c];
          b2[c] = tc[27 + c] + eta * tc[33 + c];
        }
      }
#pragma unroll
      for (int i = 0; i < n; ++i) {
        const T wy = uy1[i * L::SPY];
        const T wz = uz1[i * L::SPZ];
        T f0, f1, f2;
        if constexpr (TRI) {
          using KT = KTable<T, n - 1>;
          const T xi = KT::x(i);
          const T p0 = a1[0] + xi * b1[0], p1 = a1[1] + xi * b1[1], p2 = a1[2] + xi * b1[2];  // t_1
          const T q0 = a2[0] + xi * b2[0], q1 = a2[1] + xi * b2[1], q2 = a2[2] + xi * b2[2];  // t_2
          // rows of adj J: c0 = t1 x t2, c1 = t2 x t0, c2 = t0 x t1
          const T c00 = p1 * q2 - p2 * q1, c01 = p2 * q0 - p0 * q2, c02 = p0 * q1 - p1 * q0;
          const T c10 = q1 * t0[2] - q2 * t0[1], c11 = q2 * t0[0] - q0 * t0[2], c12 = q0 * t0[1] - q1 * t0[0];
          const T c20 = t0[1] * p2 - t0[2] * p1, c21 = t0[2] * p0 - t0[0] * p2, c22 = t0[0] * p1 - t0[1] * p0;
          const T det = t0[0] * c00 + t0[1] * c01 + t0[2] * c02;
          const T sc = (wab * KT::w(i)) / fabs(det);
          const T v0 = gx[i] * c00 + wy * c10 + wz * c20;
          const T v1 = gx[i] * c01 + wy * c11 + wz * c21;
          const T v2 = gx[i] * c02 + wy * c12 + wz * c22;
          f0 = sc * (c00 * v0 + c01 * v1 + c02 * v2);
          f1 = sc * (c10 * v0 + c11 * v1 + c12 * v2);
          f2 = sc * (c20 * v0 + c21 * v1 + c22 * v2);
          if constexpr (WEST) {
            const T wdet = (wab * KT::w(i)) * fabs(det);  // detJ of the streamed form at this point
            atomicAdd(a.m + dof[i], mx[i] * wdet);        // m += cm detJ un
            ry[i] += bex[i] * wdet;                       // b += cy detJ vn^2
          }
        } else {
          G6<T> g;
          T sc;
          if constexpr (AFF) {
            g = gc;
            sc = cc * wreg[i];
          } else {
            g = load_g6(Gc + i * (N2 * 6));
            sc = cc;
          }
          f0 = sc * (g.g0 * gx[i] + g.g1 * wy + g.g2 * wz);
          f1 = sc * (g.g1 * gx[i] + g.g3 * wy + g.g4 * wz);
          f2 = sc * (g.g2 * gx[i] + g.g4 * wy + g.g5 * wz);
        }
#pragma unroll
        for (int l = 0; l < n; ++l) ry[l] += D::at(i * n + l) * f0;
        uy1[i * L::SPY] = f1;
        uz1[i * L::SPZ] = f2;
      }
    }
    __syncthreads();

    // ---- D^T along y and z, in place (each thread rewrites its own pencil) --
    if (active) {
      T f[n];
#pragma unroll
      for (int l = 0; l < n; ++l) f[l] = uy2[l * n];
#pragma unroll
      for (int j = 0; j < n; ++j) {
        T acc = T(0);
#pragma unroll
        for (int l = 0; l < n; ++l) acc += D::at(l * n + j) * f[l];
        uy2[j * n] = acc;
      }
#pragma unroll
      for (int l = 0; l < n; ++l) f[l] = uz3[l];
#pragma unroll
      for (int k = 0; k < n; ++k) {
        T acc = T(0);
#pragma unroll
        for (int l = 0; l < n; ++l) acc += D::at(l * n + k) * f[l];
        uz3[k] = acc;
      }
    }
    __syncthreads();
    }  // !RECT

    // ---- sum the three directions and scatter-add the x pencil --------------
    if (active) {
#pragma unroll
      for (int i = 0; i < n; ++i) {
        const T val = ry[i] + uy1[i * L::SPY] + uz1[i * L::SPZ];
        if constexpr (ATOMIC) {
          atomicAdd(a.y + dof[i], val);
        } else {
          a.y[dof[i]] += val;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < n; ++i) {
      dof[i] = dofn[i];
      dofn[i] = dofm[i];
      xv[i] = xvn[i];
      if constexpr (DUAL) xw[i] = xwn[i];
      if constexpr (WEST && !NOSTREAM) dj[i] = djn[i];
    }
    store_tc((it + 1) & 1);  // next batch's coefficients (nobody reads that buffer any more)
    if constexpr (RECT) {
#pragma unroll
      for (int q = 0; q < NCS; ++q) csc[q] = cscn[q];
    }
    __syncthreads();  // tiles and stage s are free again
  }
}

template <typename T, int n, int MODE, bool ATOMIC, int GEO, bool WAIT>
int launch_one(const StiffArgs<T>& a, cudaStream_t stream) {
  using L = Layout<T, n>;
  constexpr int SMEM = GEO == 3 ? L::SMEM_TRI : (GEO ? L::SMEM_AFF : L::SMEM);
  auto kern = stiffness_kernel<T, n, MODE, ATOMIC, GEO, WAIT>;
  // per instantiation AND per device: the shared-memory opt-in is a per-device attribute
  static int blocks_per_sm[64] = {0};
  int dev = 0;
  FUS_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "stiffness: device index >= 64");
  if (blocks_per_sm[dev] == 0) {
    FUS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    int occ = 0;
    FUS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, Cfg<T, n>::THREADS, SMEM));
    blocks_per_sm[dev] = occ > 0 ? occ : 1;
  }
  const long long nb = (a.ncells + L::B - 1) / L::B;
  long long grid = (long long)fus_num_sms() * blocks_per_sm[dev];
  if (grid > nb) grid = nb;
  kern<<<(unsigned)grid, Cfg<T, n>::THREADS, SMEM, stream>>>(a);
  FUS_LAUNCH_CHECK("stiffness_kernel");
  return 0;
}

template <typename T, int n, int MODE, bool ATOMIC, int GEO>
int launch_cfg(StiffArgs<T> a, cudaStream_t stream) {
  // a halo wait armed by fus_stiffness_arm_halo_wait applies to this launch (and is consumed)
  const FusHaloDev* hd = nullptr;
  long long from = 0;
  a.wait_row = nullptr;
  a.wait_src = nullptr;
  a.wait_nsrc = 0;
  a.wait_ctr = nullptr;
  a.wait_from = a.ncells;
  if (fus_take_armed_wait(&hd, &from)) {
    if constexpr (ATOMIC) {
      if (hd->n_owner_ranks > 0 && from < a.ncells) {
        a.wait_row = hd->pad + (long long)FUS_ROW_FWD * hd->world;
        a.wait_src = hd->owner_ranks;
        a.wait_nsrc = hd->n_owner_ranks;
        a.wait_ctr = hd->ctr;
        a.wait_from = from < 0 ? 0 : from;
        return launch_one<T, n, MODE, ATOMIC, GEO, true>(a, stream);
      }
    } else {
      return fus_set_error(FUS_ERR_BAD_ARGUMENT, "stiffness: a halo wait cannot be combined with FUS_NO_ATOMICS");
    }
  }
  return launch_one<T, n, MODE, ATOMIC, GEO, false>(a, stream);
}

template <typename T, int MODE, int GEO>
int launch(const StiffArgs<T>& a, int P, int flags, cudaStream_t stream) {
  const bool atomic = !(flags & FUS_NO_ATOMICS);
#define FUS_CASE(N)                                                       \
  case N - 1:                                                             \
    return atomic ? launch_cfg<T, N, MODE, true, GEO>(a, stream)          \
                  : launch_cfg<T, N, MODE == 2 ? 1 : MODE, false, GEO>(a, stream);
  switch (P) {
    FUS_CASE(3)
    FUS_CASE(4)
    FUS_CASE(5)
    FUS_CASE(6)
    FUS_CASE(7)
    FUS_CASE(8)
  }
#undef FUS_CASE
  return fus_set_error(FUS_ERR_BAD_DEGREE, "stiffness: degree must be 2..7");
}

template <typename T>
int set_dphi(int P, const T* dphi, cudaStream_t stream) {
  if (P < 2 || P > 7) return fus_set_error(FUS_ERR_BAD_DEGREE, "set_dphi: degree must be 2..7");
  if (dphi == nullptr) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "set_dphi: null table");
  const size_t bytes = sizeof(T) * (P + 1) * (P + 1);
  const size_t off = sizeof(T) * 64 * (P - 2);
  if constexpr (sizeof(T) == 8) {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_D64, dphi, bytes, off, cudaMemcpyDefault, stream));
  } else {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_D32, dphi, bytes, off, cudaMemcpyDefault, stream));
  }
  return 0;
}

}  // namespace
