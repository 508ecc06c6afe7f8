// Fused RK4 stage kernels, sm_100a.
//
// The reference runs one RK stage as 13 separate vector launches plus two
// facet mass launches (/root/reference/cuda/demo_linear_box.py:491-563;
// CPU twin numba-cpu/demo_linear_box.py:425-459; C++ cpp/common/Linear.hpp:
// 237-344), every one a full pass over 2-3 vectors.  Here a stage is
//     [open]  ->  stiffness (+ boundary terms)  ->  close (chained with the
//                                                    next stage's open)
// so the vector work of a stage is ONE pass: 7 reads + 5 writes per dof.
//
// Stage algebra (a, b = Butcher coefficients; ku holds vn, "f0: ku = vn"):
//   open : un = u0 + a dt ku ; vn = v0 + a dt kv ; ku <- vn ; b <- 0
//   close: kv = b / m ; u += b_i dt ku ; v += b_i dt kv
// Ping-pong steps (next_mode 3 / 1 / 1 / 4): the first stage of a step takes its input
// straight from the base state (a_0 = 0: un = u0, vn = v0) and starts the accumulators from
// it, the last one leaves the new state in the accumulators, and the caller swaps base and
// accumulator buffers between steps: 9 + 12 + 12 + 8 vector passes per step instead of 4 x 12,
// same arithmetic bit for bit.
// Pure HBM streams, 16-byte vector accesses, grid-stride over a few waves.

#include <initializer_list>

#include "halo_internal.cuh"

namespace {

constexpr int kThreads = 256;

template <typename T>
struct Vec;
template <>
struct Vec<double> {
  using type = double2;
  static constexpr int W = 2;
};
template <>
struct Vec<float> {
  using type = float4;
  static constexpr int W = 4;
};

template <typename T, int W>
struct Pack {
  T v[W];
};

template <typename T, bool VEC>
__device__ __forceinline__ Pack<T, Vec<T>::W> ld(const T* p, long long k) {
  Pack<T, Vec<T>::W> r;
  if constexpr (VEC) {
    *reinterpret_cast<typename Vec<T>::type*>(r.v) =
        reinterpret_cast<const typename Vec<T>::type*>(p)[k];
  } else {
    r.v[0] = p[k];
  }
  return r;
}
template <typename T, bool VEC>
__device__ __forceinline__ void st(T* p, long long k, const Pack<T, Vec<T>::W>& r) {
  if constexpr (VEC) {
    reinterpret_cast<typename Vec<T>::type*>(p)[k] =
        *reinterpret_cast<const typename Vec<T>::type*>(r.v);
  } else {
    p[k] = r.v[0];
  }
}

template <typename T>
struct OpenArgs {
  const T* u;
  const T* v;
  T* u0;
  T* v0;
  T* ku;
  const T* kv;
  T* un;
  T* b;
  T adt;
  int first;
  long long n;
};

template <typename T, bool VEC>
__device__ __forceinline__ void open_body(const OpenArgs<T>& a, long long k) {
  constexpr int W = VEC ? Vec<T>::W : 1;
  using P = Pack<T, Vec<T>::W>;
  P u0, v0, ku, kv, un, vn, z;
  if (a.first) {
    u0 = ld<T, VEC>(a.u, k);
    v0 = ld<T, VEC>(a.v, k);
    st<T, VEC>(a.u0, k, u0);
    st<T, VEC>(a.v0, k, v0);
  } else {
    u0 = ld<T, VEC>(a.u0, k);
    v0 = ld<T, VEC>(a.v0, k);
  }
  ku = ld<T, VEC>(a.ku, k);
  kv = ld<T, VEC>(a.kv, k);
#pragma unroll
  for (int w = 0; w < W; ++w) {
    un.v[w] = a.adt * ku.v[w] + u0.v[w];
    vn.v[w] = a.adt * kv.v[w] + v0.v[w];
    z.v[w] = T(0);
  }
  st<T, VEC>(a.un, k, un);
  st<T, VEC>(a.ku, k, vn);
  st<T, VEC>(a.b, k, z);
}

template <typename T, bool VEC>
__global__ void __launch_bounds__(kThreads, 4) rk_open_kernel(const OpenArgs<T> a) {
  constexpr int W = VEC ? Vec<T>::W : 1;
  const long long stride = (long long)gridDim.x * kThreads;
  const long long i0 = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long nv = a.n / W;
  for (long long k = i0; k < nv; k += stride) open_body<T, VEC>(a, k);
  if constexpr (VEC) {
    const long long k = nv * W + i0;
    if (k < a.n) open_body<T, false>(a, k);
  }
}

template <typename T>
struct CloseArgs {
  T* u;
  T* v;
  T* u0;
  T* v0;
  T* ku;
  T* kv;  // may be null when chained (next_mode != 0)
  T* un;
  T* b;
  T* m;         // Westervelt: state-dependent part, zeroed here; linear: the lumped mass (read only)
  const T* m0;  // Westervelt only
  const T* m2;  // pointwise Westervelt (WEST == 2): lumped M(c2; 1) and M(c5; 1)
  const T* m5;
  T bdt;
  T adt_next;
  int next_mode;
  long long n;
  long long* step;  // device step counter, incremented at a step boundary (may be null)
  // multi-GPU: bit d set <=> dof d is shared with a neighbour and is closed by
  // rk_close_shared_kernel once the reverse halo has landed (null: close everything)
  const unsigned char* skip;
};

// WEST 0: linear (kv = b / m).  WEST 1: m += m0, kv = b / m, m = 0 (the cell-mass pair was
// accumulated into m and b by the stage kernel).  WEST 2: the lumped mass is diagonal, so the
// cell-mass pair of cuda/demo_nonlinear_bowl.py:609-612, 626-628 is pointwise:
//   M(c2; un) = un * M(c2; 1) = un * m2,   M(c5; vn^2) = vn^2 * m5
// and kv = (b + vn^2 m5) / (m0 + un m2) with un, vn the stage input (un still holds it here).
// WEST 3: not an RK stage but a whole LEAPFROG step of the second-order system (u at whole steps,
// v at half steps; the reference implements RK4 only, the north star also names leapfrog):
//   v += bdt * b / m ; u += adt_next * v ; b = 0
// with m = m_lumped - (dt/2) absb, which makes the absorbing term a (v+ + v-)/2 time-centred
// (second order, unconditionally damping) at no extra cost.  4 reads + 3 writes per dof.
template <typename T, bool VEC, int WEST>
__device__ __forceinline__ void close_body(const CloseArgs<T>& a, long long k) {
  constexpr int W = VEC ? Vec<T>::W : 1;
  using P = Pack<T, Vec<T>::W>;
  if constexpr (WEST == 3) {
    const P b = ld<T, VEC>(a.b, k), m = ld<T, VEC>(a.m, k);
    P u = ld<T, VEC>(a.u, k), v = ld<T, VEC>(a.v, k), z;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      v.v[w] = a.bdt * (b.v[w] / m.v[w]) + v.v[w];
      u.v[w] = a.adt_next * v.v[w] + u.v[w];
      z.v[w] = T(0);
    }
    st<T, VEC>(a.u, k, u);
    st<T, VEC>(a.v, k, v);
    st<T, VEC>(a.b, k, z);
    return;
  }
  P b = ld<T, VEC>(a.b, k);
  P m;
  if constexpr (WEST == 2) {
    m = ld<T, VEC>(a.m0, k);
  } else {
    m = ld<T, VEC>(a.m, k);
  }
  P ku, u, v, u0, v0;
  if (a.next_mode == 3) {
    // first stage of a ping-pong step: the accumulators start from the base state (u0, v0),
    // which is also the stage input (un = u0, vn = ku = v0): nothing else is read
    u0 = ld<T, VEC>(a.u0, k);
    v0 = ld<T, VEC>(a.v0, k);
    ku = v0;
    u = u0;
    v = v0;
  } else {
    ku = ld<T, VEC>(a.ku, k);
    u = ld<T, VEC>(a.u, k);
    v = ld<T, VEC>(a.v, k);
  }
  P kv, z;
  if constexpr (WEST == 1) {
    P m0 = ld<T, VEC>(a.m0, k);
#pragma unroll
    for (int w = 0; w < W; ++w) m.v[w] = m.v[w] + m0.v[w];  // axpy(1.0, m0, m)
  }
  if constexpr (WEST == 2) {
    const P m2 = ld<T, VEC>(a.m2, k);
    const P m5 = ld<T, VEC>(a.m5, k);
    P xin;  // the stage input un: the base state itself in the first stage of a ping-pong step
    if (a.next_mode == 3) {
      xin = u0;
    } else {
      xin = ld<T, VEC>(a.un, k);
    }
#pragma unroll
    for (int w = 0; w < W; ++w) {
      m.v[w] = xin.v[w] * m2.v[w] + m.v[w];                 // m = m0 + M(c2; un)
      b.v[w] = (ku.v[w] * ku.v[w]) * m5.v[w] + b.v[w];      // b += M(c5; vn^2)
    }
  }
#pragma unroll
  for (int w = 0; w < W; ++w) {
    kv.v[w] = b.v[w] / m.v[w];
    u.v[w] = a.bdt * ku.v[w] + u.v[w];
    v.v[w] = a.bdt * kv.v[w] + v.v[w];
    z.v[w] = T(0);
  }
  st<T, VEC>(a.u, k, u);
  st<T, VEC>(a.v, k, v);
  if (a.kv != nullptr) st<T, VEC>(a.kv, k, kv);
  if constexpr (WEST == 1) st<T, VEC>(a.m, k, z);
  if (a.next_mode == 1 || a.next_mode == 3) {
    if (a.next_mode == 1) {
      u0 = ld<T, VEC>(a.u0, k);
      v0 = ld<T, VEC>(a.v0, k);
    }
    P un, vn;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      un.v[w] = a.adt_next * ku.v[w] + u0.v[w];
      vn.v[w] = a.adt_next * kv.v[w] + v0.v[w];
    }
    st<T, VEC>(a.un, k, un);
    st<T, VEC>(a.ku, k, vn);
    st<T, VEC>(a.b, k, z);
  } else if (a.next_mode == 2) {
    st<T, VEC>(a.u0, k, u);
    st<T, VEC>(a.v0, k, v);
    st<T, VEC>(a.un, k, u);
    st<T, VEC>(a.ku, k, v);
    st<T, VEC>(a.b, k, z);
  } else if (a.next_mode == 4) {
    st<T, VEC>(a.b, k, z);  // last stage of a ping-pong step: the accumulators ARE the new state
  }
}

template <typename T, bool VEC, int WEST>
__global__ void __launch_bounds__(kThreads, 3) rk_close_kernel(const CloseArgs<T> a) {
  constexpr int W = VEC ? Vec<T>::W : 1;
  const long long stride = (long long)gridDim.x * kThreads;
  const long long i0 = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long nv = a.n / W;
  if (a.skip == nullptr) {
    for (long long k = i0; k < nv; k += stride) close_body<T, VEC, WEST>(a, k);
    if constexpr (VEC) {
      const long long k = nv * W + i0;
      if (k < a.n) close_body<T, false, WEST>(a, k);
    }
  } else {
    // The mask marks whole aligned groups of 4 dofs (fus_halo_create), so a pack (W = 2 or 4
    // dofs, W divides 4) is either closed here or left entirely to rk_close_shared_kernel.  The
    // mask byte of the NEXT iteration is fetched before this iteration's loads are issued, so
    // the test never sits in front of the vector loads.
    long long k = i0;
    unsigned cur = k < nv ? (unsigned)a.skip[(k * W) >> 3] : 0u;
    for (; k < nv; k += stride) {
      const long long kn = k + stride;
      const unsigned nxt = kn < nv ? (unsigned)a.skip[(kn * W) >> 3] : 0u;
      if (((cur >> (unsigned)((k * W) & 7)) & 1u) == 0u) close_body<T, VEC, WEST>(a, k);
      cur = nxt;
    }
    if constexpr (VEC) {
      const long long kt = nv * W + i0;
      if (kt < a.n && !(((unsigned)a.skip[kt >> 3] >> (unsigned)(kt & 7)) & 1u)) close_body<T, false, WEST>(a, kt);
    }
  }
  if (a.step != nullptr && (a.next_mode == 2 || a.next_mode == 4) && i0 == 0) *a.step += 1;
}

// Multi-GPU: the stage closing on the unique owned dofs that are ghosts on a neighbour
// (their b is complete only after the reverse halo), fused with the forward halo of the
// NEXT stage: the fresh stage input (un, vn = ku; or the new state u, v after the last
// stage) goes straight from registers into the neighbours' ghost slots, then the FWD epoch.
// Runs BESIDE rk_close_kernel, which keeps 3 blocks of 256 threads x 80 registers resident per SM
// (61k of the 64k registers).  Blocks of 64 threads fit into what is left, so this kernel starts at
// once instead of waiting for close blocks to retire, and never displaces one: with 256-thread
// blocks the close of the ranks that own shared faces took 530 us instead of 485 on 8 GPUs
// (profiles/r02_multigpu_timeline.md).  Its threads mostly wait on remote loads; a small grid is enough.
constexpr int kSharedThreads = 64;

template <typename T, int WEST>
__global__ void __launch_bounds__(kSharedThreads) rk_close_shared_kernel(const CloseArgs<T> a, const FusHaloDev h, int put,
                                                                         int gather) {
  const long long stride = (long long)gridDim.x * kSharedThreads;
  T* const xa = a.next_mode == 4 ? a.u : a.un;
  T* const xb = a.next_mode == 4 ? a.v : a.ku;
  for (long long i = (long long)blockIdx.x * kSharedThreads + threadIdx.x; i < h.nu; i += stride) {
    const long long k = h.uniq[i];
    const long long j0 = h.uoff[i], j1 = h.uoff[i + 1];
    if (gather && j1 > j0) {
      // reverse halo, fused: add the neighbours' ghost partial sums of this dof (loaded straight
      // from their vectors) and clear them there for the next stage; the local assembly of b[k]
      // finished before this kernel, and nobody else touches dof k now
      T sb = T(0), sm = T(0);
      for (long long j = j0; j < j1; ++j) {
        const long long dl = h.seg_delta[h.useg[j]];
        const long long rp = h.upos[j];
        T* rb = reinterpret_cast<T*>(reinterpret_cast<char*>(a.b) + dl) + rp;
        sb += *reinterpret_cast<volatile const T*>(rb);
        *rb = T(0);
        if constexpr (WEST == 1) {
          T* rm = reinterpret_cast<T*>(reinterpret_cast<char*>(a.m) + dl) + rp;
          sm += *reinterpret_cast<volatile const T*>(rm);
          *rm = T(0);
        }
      }
      a.b[k] += sb;
      if constexpr (WEST == 1) a.m[k] += sm;
    }
    close_body<T, false, WEST>(a, k);
    if (put) {
      const T va = xa[k], vb = xb[k];
      for (long long j = j0; j < j1; ++j) {
        const long long dl = h.seg_delta[h.useg[j]];
        const long long rp = h.upos[j];
        reinterpret_cast<T*>(reinterpret_cast<char*>(xa) + dl)[rp] = va;
        reinterpret_cast<T*>(reinterpret_cast<char*>(xb) + dl)[rp] = vb;
      }
    }
  }
  if (put) {
    if (fus_last_block(&h.ctr[FUS_CTR_TICKET_CLOSE]))
      fus_signal(&h.ctr[FUS_CTR_TICKET_CLOSE], &h.ctr[FUS_CTR_FWD_SENT], h.fwd_targets, h.n_ghost_ranks);
  }
}

// The end of a multi-GPU stage's boundary launch: the last block raises the REV epoch on every owner
// of my ghosts (= fus_halo_signal_reverse, without a launch of its own on the critical path).
__device__ __forceinline__ void boundary_signal(const FusHaloDev& h, int consume_fwd) {
  if (fus_last_block(&h.ctr[FUS_CTR_TICKET_BOUNDARY])) {
    // the stiffness launches of this stage have consumed one FWD epoch (their in-kernel wait
    // reads the counter, this kernel - the next one on the stream - advances it)
    if (threadIdx.x == 0 && consume_fwd) h.ctr[FUS_CTR_FWD_WAITED] += 1ULL;
    fus_signal(&h.ctr[FUS_CTR_TICKET_BOUNDARY], &h.ctr[FUS_CTR_REV_SENT], h.rev_targets, h.n_owner_ranks);
  }
}

// b[dof[i]] += g*src[i] + dg*src2[i] + vn[dof[i]]*absb[i]; the dof list is unique.
// SIGNAL (multi-GPU): this is the last kernel of a stage that writes ghost partial sums, so its
// last block raises the REV epoch on every owner of my ghosts (= fus_halo_signal_reverse, without
// a launch of its own on the critical path).
template <typename T, bool SIGNAL>
__global__ void __launch_bounds__(kThreads)
    boundary_kernel(T* b, const T* __restrict__ vn, const int32_t* __restrict__ dof,
                    const T* __restrict__ src, const T* __restrict__ src2,
                    const T* __restrict__ absb, T g, T dg, const T* __restrict__ gtab,
                    const long long* __restrict__ step, int gstride, int goff, long long n, const FusHaloDev h,
                    int consume_fwd) {
  if (gtab != nullptr) {
    const long long s = step != nullptr ? *step : 0;
    g = gtab[s * gstride + goff];
    dg = gtab[s * gstride + goff + 1];
  }
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const int d = dof[i];
    T acc = T(0);
    if (src != nullptr) acc += g * src[i];
    if (src2 != nullptr) acc += dg * src2[i];
    if (absb != nullptr) acc += vn[d] * absb[i];
    b[d] += acc;
  }
  if constexpr (SIGNAL) boundary_signal(h, consume_fwd);
}

// Phased-array source: every source dof carries one (element, weight) entry per array element whose
// facets contain it (CSR rows over the same compact dof list; a dof that only absorbs has an empty
// row), and the element's own stage amplitudes come from the table
//   G = etab + step*8E + stage*2E,  DG = G + E          (layout (rows, 4 stages, 2, E))
//   b[dof[i]] += sum_{k in row i} (w[k] G[elem[k]] + w2[k] DG[elem[k]]) + vn[dof[i]] absb[i]
// One thread per dof, the sum in row order: deterministic, no atomics.  The 2E stage values are read
// through the read-only path: E <= a few thousand values shared by every thread stay in L1 / L2.
template <typename T, bool SIGNAL>
__global__ void __launch_bounds__(kThreads)
    boundary_elements_kernel(T* b, const T* __restrict__ vn, const int32_t* __restrict__ dof,
                             const int32_t* __restrict__ row, const int32_t* __restrict__ elem,
                             const T* __restrict__ w, const T* __restrict__ w2, const T* __restrict__ absb,
                             const T* __restrict__ etab, const long long* __restrict__ step, int E, int stage,
                             long long n, const FusHaloDev h, int consume_fwd) {
  const long long s = step != nullptr ? *step : 0;
  const T* __restrict__ G = etab + s * 8LL * E + 2LL * stage * E;
  const T* __restrict__ DG = G + E;
  const long long stride = (long long)gridDim.x * kThreads;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const int d = dof[i];
    const int k1 = row[i + 1];
    T acc = T(0);
    for (int k = row[i]; k < k1; ++k) {
      const int e = elem[k];
      acc += w[k] * __ldg(G + e);
      if (w2 != nullptr) acc += w2[k] * __ldg(DG + e);
    }
    if (absb != nullptr) acc += vn[d] * absb[i];
    b[d] += acc;
  }
  if constexpr (SIGNAL) boundary_signal(h, consume_fwd);
}

inline unsigned grid_for(long long n) {
  long long blocks = (n + kThreads - 1) / kThreads;
  const long long cap = (long long)fus_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

inline bool aligned16(std::initializer_list<const void*> ps) {
  uintptr_t bits = 0;
  for (const void* p : ps) bits |= reinterpret_cast<uintptr_t>(p);
  return (bits & 15u) == 0;
}

template <typename T>
int open_entry(const T* u, const T* v, T* u0, T* v0, T* ku, const T* kv, T* un, T* b, T adt,
               int first, int64_t n, void* stream) {
  if (n < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_open: n < 0");
  if (n == 0) return 0;
  OpenArgs<T> a{u, v, u0, v0, ku, kv, un, b, adt, first, n};
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  if (aligned16({u, v, u0, v0, ku, kv, un, b})) {
    rk_open_kernel<T, true><<<grid_for(n / Vec<T>::W + 1), kThreads, 0, st_>>>(a);
  } else {
    rk_open_kernel<T, false><<<grid_for(n), kThreads, 0, st_>>>(a);
  }
  FUS_LAUNCH_CHECK("rk_open_kernel");
  return 0;
}

template <typename T, int WEST>
int close_entry(T* u, T* v, T* u0, T* v0, T* ku, T* kv, T* un, T* b, T* m, const T* m0, T bdt,
                T adt_next, int next_mode, int64_t n, int64_t* step, const uint8_t* skip, void* stream,
                const T* m2 = nullptr, const T* m5 = nullptr) {
  if (n < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close: n < 0");
  if (next_mode < 0 || next_mode > 4) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close: next_mode");
  if (next_mode == 0 && kv == nullptr)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close: kv must be stored when not chained");
  if (WEST == 2 && (m0 == nullptr || m2 == nullptr || m5 == nullptr))
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_westervelt_pw: null m0 / m2 / m5");
  if (WEST == 3 && (u == nullptr || v == nullptr || b == nullptr || m == nullptr))
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "leapfrog_close: null vector");
  const bool counts_step = step != nullptr && (next_mode == 2 || next_mode == 4);
  if (n == 0 && !counts_step) return 0;
  CloseArgs<T> a{u, v, u0, v0, ku, kv, un, b, m, m0, m2, m5, bdt, adt_next, next_mode, n,
                 reinterpret_cast<long long*>(step), skip};
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  if (n == 0) {
    // an empty range still ends the step (a rank whose owned dofs are all closed by
    // fus_rk_close_shared_*): one block touches no dof and advances the counter
    rk_close_kernel<T, false, WEST><<<1, kThreads, 0, st_>>>(a);
  } else if (aligned16({u, v, u0, v0, ku, kv, un, b, m, m0, m2, m5})) {
    rk_close_kernel<T, true, WEST><<<grid_for(n / Vec<T>::W + 1), kThreads, 0, st_>>>(a);
  } else {
    rk_close_kernel<T, false, WEST><<<grid_for(n), kThreads, 0, st_>>>(a);
  }
  FUS_LAUNCH_CHECK("rk_close_kernel");
  return 0;
}

// variant 0: linear, 1: Westervelt "cells" form, 2: Westervelt pointwise form
template <typename T>
int close_shared_entry(fus_halo* halo, int variant, int put_next, int gather, T* u, T* v, T* u0, T* v0, T* ku, T* un, T* b,
                       T* m, const T* m0, const T* m2, const T* m5, T bdt, T adt_next, int next_mode,
                       void* stream) {
  if (halo == nullptr) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_shared: null halo handle");
  if (variant < 0 || variant > 3) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_shared: variant");
  if (next_mode < 1 || next_mode > 4) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_shared: next_mode 1..4");
  if (((variant == 1 || variant == 2) && m0 == nullptr) || (variant == 2 && (m2 == nullptr || m5 == nullptr)) ||
      ((variant <= 1 || variant == 3) && m == nullptr))
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_shared: null mass vector");
  if (variant == 3 && next_mode != 4)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "rk_close_shared: the leapfrog variant takes next_mode 4");
  const FusHaloDev& h = *fus_halo_dev_of(halo);
  if (h.nu == 0) return 0;  // nothing shared: nobody ghosts my dofs, nobody waits for my signal
  CloseArgs<T> a{u, v, u0, v0, ku, nullptr, un, b, m, m0, m2, m5, bdt, adt_next, next_mode, h.size_local,
                 nullptr, nullptr};
  long long blocks = (h.nu + kSharedThreads - 1) / kSharedThreads;
  const long long cap = (long long)fus_num_sms() * 2;
  if (blocks > cap) blocks = cap;
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  const int put = put_next ? 1 : 0, gat = gather ? 1 : 0;
  if (variant == 0) {
    rk_close_shared_kernel<T, 0><<<(unsigned)blocks, kSharedThreads, 0, st_>>>(a, h, put, gat);
  } else if (variant == 1) {
    rk_close_shared_kernel<T, 1><<<(unsigned)blocks, kSharedThreads, 0, st_>>>(a, h, put, gat);
  } else if (variant == 3) {
    rk_close_shared_kernel<T, 3><<<(unsigned)blocks, kSharedThreads, 0, st_>>>(a, h, put, gat);
  } else {
    rk_close_shared_kernel<T, 2><<<(unsigned)blocks, kSharedThreads, 0, st_>>>(a, h, put, gat);
  }
  FUS_LAUNCH_CHECK("rk_close_shared_kernel");
  return 0;
}

template <typename T>
int boundary_entry(T* b, const T* vn, const int32_t* dof, const T* src, const T* src2,
                   const T* absb, T g, T dg, const T* gtab, const int64_t* step, int gstride,
                   int goff, int64_t n, void* stream, fus_halo* halo = nullptr, int consume_fwd = 0) {
  if (n < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms: n < 0");
  const bool signal = halo != nullptr && fus_halo_dev_of(halo)->n_owner_ranks > 0;
  if (n == 0 && !signal) return 0;
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  const long long* stp = reinterpret_cast<const long long*>(step);
  if (signal) {
    boundary_kernel<T, true><<<grid_for(n), kThreads, 0, st_>>>(b, vn, dof, src, src2, absb, g, dg, gtab, stp,
                                                                gstride, goff, n, *fus_halo_dev_of(halo), consume_fwd);
  } else {
    boundary_kernel<T, false><<<grid_for(n), kThreads, 0, st_>>>(b, vn, dof, src, src2, absb, g, dg, gtab, stp,
                                                                 gstride, goff, n, FusHaloDev{}, 0);
  }
  FUS_LAUNCH_CHECK("boundary_kernel");
  return 0;
}

template <typename T>
int boundary_elements_entry(T* b, const T* vn, const int32_t* dof, const int32_t* row, const int32_t* elem,
                            const T* w, const T* w2, const T* absb, const T* etab, const int64_t* step, int E,
                            int stage, int64_t n, void* stream, fus_halo* halo = nullptr, int consume_fwd = 0) {
  if (n < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements: n < 0");
  if (E < 1) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements: num_elements < 1");
  if (stage < 0 || stage > 3) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements: stage 0..3");
  if (n > 0 && (b == nullptr || dof == nullptr || etab == nullptr || row == nullptr || elem == nullptr || w == nullptr))
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements: null b / dof / etab / row / elem / w");
  if (n > 0 && absb != nullptr && vn == nullptr)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements: null vn with absb");
  const bool signal = halo != nullptr && fus_halo_dev_of(halo)->n_owner_ranks > 0;
  if (n == 0 && !signal) return 0;
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  const long long* stp = reinterpret_cast<const long long*>(step);
  if (signal) {
    boundary_elements_kernel<T, true><<<grid_for(n), kThreads, 0, st_>>>(
        b, vn, dof, row, elem, w, w2, absb, etab, stp, E, stage, n, *fus_halo_dev_of(halo), consume_fwd);
  } else {
    boundary_elements_kernel<T, false><<<grid_for(n), kThreads, 0, st_>>>(
        b, vn, dof, row, elem, w, w2, absb, etab, stp, E, stage, n, FusHaloDev{}, 0);
  }
  FUS_LAUNCH_CHECK("boundary_elements_kernel");
  return 0;
}

}  // namespace

extern "C" {

#define FUS_RK_API(SFX, T)                                                                       \
  int fus_rk_open_##SFX(const T* u, const T* v, T* u0, T* v0, T* ku, const T* kv, T* un, T* b,   \
                        T adt, int first, int64_t n, void* s) {                                  \
    return open_entry<T>(u, v, u0, v0, ku, kv, un, b, adt, first, n, s);                         \
  }                                                                                              \
  int fus_rk_close_##SFX(T* u, T* v, T* u0, T* v0, T* ku, T* kv, T* un, T* b, const T* m, T bdt, \
                         T adt_next, int next_mode, int64_t n, int64_t* step_dev,                \
                         const uint8_t* skip_mask, void* s) {                                    \
    return close_entry<T, 0>(u, v, u0, v0, ku, kv, un, b, const_cast<T*>(m), nullptr, bdt,       \
                             adt_next, next_mode, n, step_dev, skip_mask, s);                    \
  }                                                                                              \
  int fus_rk_close_shared_##SFX(fus_halo_t* halo, int variant, int put_next, int gather, T* u,   \
                                T* v, T* u0, T* v0, T* ku, T* un, T* b, T* m, const T* m0,       \
                                const T* m2, const T* m5, T bdt, T adt_next, int next_mode,      \
                                void* s) {                                                       \
    return close_shared_entry<T>(halo, variant, put_next, gather, u, v, u0, v0, ku, un, b, m,    \
                                 m0, m2, m5, bdt, adt_next, next_mode, s);                       \
  }                                                                                              \
  int fus_rk_close_westervelt_##SFX(T* u, T* v, T* u0, T* v0, T* ku, T* kv, T* un, T* b, T* m,   \
                                    const T* m0, T bdt, T adt_next, int next_mode, int64_t n,    \
                                    int64_t* step_dev, const uint8_t* skip_mask, void* s) {      \
    return close_entry<T, 1>(u, v, u0, v0, ku, kv, un, b, m, m0, bdt, adt_next, next_mode, n,    \
                             step_dev, skip_mask, s);                                            \
  }                                                                                              \
  int fus_rk_close_westervelt_pw_##SFX(T* u, T* v, T* u0, T* v0, T* ku, T* kv, T* un, T* b,      \
                                       const T* m0, const T* m2, const T* m5, T bdt, T adt_next, \
                                       int next_mode, int64_t n, int64_t* step_dev,              \
                                       const uint8_t* skip_mask, void* s) {                      \
    return close_entry<T, 2>(u, v, u0, v0, ku, kv, un, b, nullptr, m0, bdt, adt_next, next_mode, \
                             n, step_dev, skip_mask, s, m2, m5);                                 \
  }                                                                                              \
  int fus_leapfrog_close_##SFX(T* u, T* v, T* b, const T* m, T dt_v, T dt_u, int64_t n,          \
                               int64_t* step_dev, const uint8_t* skip_mask, void* s) {           \
    return close_entry<T, 3>(u, v, nullptr, nullptr, nullptr, nullptr, nullptr, b,               \
                             const_cast<T*>(m), nullptr, dt_v, dt_u, 4, n, step_dev, skip_mask,  \
                             s);                                                                 \
  }                                                                                              \
  int fus_boundary_terms_##SFX(T* b, const T* vn, const int32_t* dof, const T* src,              \
                               const T* src2, const T* absb, T g, T dg, const T* gtab,           \
                               const int64_t* step_dev, int gstride, int goff, int64_t n,        \
                               void* s) {                                                        \
    return boundary_entry<T>(b, vn, dof, src, src2, absb, g, dg, gtab, step_dev, gstride, goff,  \
                             n, s);                                                              \
  }                                                                                              \
  int fus_boundary_terms_signal_##SFX(fus_halo_t* halo, T* b, const T* vn, const int32_t* dof,   \
                                      const T* src, const T* src2, const T* absb, T g, T dg,     \
                                      const T* gtab, const int64_t* step_dev, int gstride,       \
                                      int goff, int64_t n, int consume_forward, void* s) {       \
    if (halo == nullptr)                                                                         \
      return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_signal: null halo handle");     \
    return boundary_entry<T>(b, vn, dof, src, src2, absb, g, dg, gtab, step_dev, gstride, goff,  \
                             n, s, halo, consume_forward);                                       \
  }                                                                                              \
  int fus_boundary_terms_elements_##SFX(T* b, const T* vn, const int32_t* dof, const int32_t* row,  \
                                        const int32_t* elem, const T* w, const T* w2,            \
                                        const T* absb, const T* etab, const int64_t* step_dev,   \
                                        int num_elements, int stage, int64_t n, void* s) {       \
    return boundary_elements_entry<T>(b, vn, dof, row, elem, w, w2, absb, etab, step_dev,        \
                                      num_elements, stage, n, s);                                \
  }                                                                                              \
  int fus_boundary_terms_elements_signal_##SFX(                                                  \
      fus_halo_t* halo, T* b, const T* vn, const int32_t* dof, const int32_t* row,               \
      const int32_t* elem, const T* w, const T* w2, const T* absb, const T* etab,                \
      const int64_t* step_dev, int num_elements, int stage, int64_t n, int consume_forward,      \
      void* s) {                                                                                 \
    if (halo == nullptr)                                                                         \
      return fus_set_error(FUS_ERR_BAD_ARGUMENT, "boundary_terms_elements_signal: null halo handle"); \
    return boundary_elements_entry<T>(b, vn, dof, row, elem, w, w2, absb, etab, step_dev,        \
                                      num_elements, stage, n, s, halo, consume_forward);         \
  }

FUS_RK_API(f64, double)
FUS_RK_API(f32, float)
#undef FUS_RK_API

}  // extern "C"
