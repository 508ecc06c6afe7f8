// Stiffness action on TRILINEAR hexahedra with the geometry recomputed in the kernel, degree 2..7,
// sm_100a - the on-the-fly-geometry mode SURVEY.md 8(d)/(f-1) names.
//
// The reference precomputes G = w |det J| J^-1 J^-T at every quadrature point
// (/root/reference/cuda/precompute.py:115-163) from the cell's 8 vertices and streams the 6 n^3
// values per cell through every operator application (cuda/operators.py:154-164).  The geometry
// map is trilinear, so the tangent of reference direction d is bilinear in the other two
// coordinates: 4 vectors per direction, 36 numbers per cell (fus_trilinear_coeffs_*) from which
// the GEO = 3 instantiation of stiffness_kernel.cuh rebuilds the factors point by point.
// HBM bytes per cell: Nd*4 (dofmap) + 37 s instead of Nd*4 + (6 Nd + 1) s; ~60 more flops per
// point.  Same result as the streamed kernel to rounding (tests/test_gpu_vertex.py).  The Westervelt
// cell form and the lumped mass take w |det J| from the same coefficients, so a solver on trilinear
// cells never allocates a per-point table (tests/test_gpu_vertex_solver.py).

#include "stiffness_kernel.cuh"

namespace {

constexpr int kCoeffThreads = 128;

// Tc[c, d, m, k] = sum_v M[d, m, v] x_g[x_dofs[c, v], k]
template <typename T>
__global__ void __launch_bounds__(kCoeffThreads)
    trilinear_coeffs_kernel(T* __restrict__ Tc, const int32_t* __restrict__ x_dofs,
                            const T* __restrict__ x_g, const T* __restrict__ M, long long ncells) {
  __shared__ T sM[96];
  if (threadIdx.x < 96) sM[threadIdx.x] = M[threadIdx.x];
  __syncthreads();
  const long long stride = (long long)gridDim.x * kCoeffThreads;
  for (long long c = (long long)blockIdx.x * kCoeffThreads + threadIdx.x; c < ncells; c += stride) {
    T coord[8][3];
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const long long d = x_dofs[c * 8 + v];
#pragma unroll
      for (int k = 0; k < 3; ++k) coord[v][k] = x_g[d * 3 + k];
    }
#pragma unroll
    for (int dm = 0; dm < 12; ++dm) {
      T s0 = T(0), s1 = T(0), s2 = T(0);
#pragma unroll
      for (int v = 0; v < 8; ++v) {
        const T w = sM[dm * 8 + v];
        s0 += w * coord[v][0];
        s1 += w * coord[v][1];
        s2 += w * coord[v][2];
      }
      T* o = Tc + c * 36 + dm * 3;
      o[0] = s0;
      o[1] = s1;
      o[2] = s2;
    }
  }
}

template <typename T>
int coeffs_entry(T* Tc, const int32_t* x_dofs, const T* x_g, const T* M, int64_t ncells, void* stream) {
  if (ncells < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "trilinear_coeffs: ncells < 0");
  if (ncells == 0) return 0;
  if (!Tc || !x_dofs || !x_g || !M) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "trilinear_coeffs: null pointer");
  long long grid = (ncells + kCoeffThreads - 1) / kCoeffThreads;
  const long long cap = (long long)fus_num_sms() * 16;
  if (grid > cap) grid = cap;
  trilinear_coeffs_kernel<T><<<(unsigned)grid, kCoeffThreads, 0, static_cast<cudaStream_t>(stream)>>>(Tc, x_dofs, x_g, M,
                                                                                                      ncells);
  FUS_LAUNCH_CHECK("trilinear_coeffs_kernel");
  return 0;
}

template <typename T>
int set_vertex_tables(int P, const T* x1, const T* w1, cudaStream_t stream) {
  if (P < 2 || P > 7) return fus_set_error(FUS_ERR_BAD_DEGREE, "set_vertex_tables: degree must be 2..7");
  if (x1 == nullptr || w1 == nullptr) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "set_vertex_tables: null table");
  const int n = P + 1;
  if constexpr (sizeof(T) == 8) {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_X64, x1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_W64, w1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
  } else {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_X32, x1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_W32, w1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
  }
  return 0;
}

constexpr int kMassThreads = 256;

// Lumped mass on trilinear cells, one thread per (cell, point):
//   y[dm[c,q]] += coeff[c] * w_q |det J_c(X_q)| * x[dm[c,q]]
// with the tangents evaluated from the cell's 36 coefficients and the 1-D points and weights of
// fus_set_vertex_tables - the detJ table of fus_mass without ever storing it.  Set-up only.
template <typename T, int n>
__global__ void __launch_bounds__(kMassThreads)
    mass_vertex_kernel(const T* __restrict__ x, const T* __restrict__ coeff, T* y, const T* __restrict__ Tc,
                       const int32_t* __restrict__ dofmap, long long total) {
  using KT = KTable<T, n - 1>;
  constexpr int N2 = n * n, Nd = n * n * n;
  const long long stride = (long long)gridDim.x * kMassThreads;
  for (long long idx = (long long)blockIdx.x * kMassThreads + threadIdx.x; idx < total; idx += stride) {
    const long long c = idx / Nd;
    const int q = (int)(idx - c * Nd);
    const int i = q / N2, j = (q / n) % n, k = q % n;
    const T xi = KT::x(i), eta = KT::x(j), zeta = KT::x(k);
    const T* tc = Tc + c * 36;
    T t0[3], t1[3], t2[3];
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      t0[e] = tc[e] + eta * tc[3 + e] + zeta * tc[6 + e] + (eta * zeta) * tc[9 + e];
      t1[e] = tc[12 + e] + xi * tc[15 + e] + zeta * tc[18 + e] + (xi * zeta) * tc[21 + e];
      t2[e] = tc[24 + e] + xi * tc[27 + e] + eta * tc[30 + e] + (xi * eta) * tc[33 + e];
    }
    const T det = t0[0] * (t1[1] * t2[2] - t1[2] * t2[1]) + t0[1] * (t1[2] * t2[0] - t1[0] * t2[2]) +
                  t0[2] * (t1[0] * t2[1] - t1[1] * t2[0]);
    const T wdet = (KT::w(i) * (KT::w(j) * KT::w(k))) * fabs(det);
    const int d = dofmap[idx];
    atomicAdd(y + d, x[d] * wdet * coeff[c]);
  }
}

template <typename T>
int mass_vertex_entry(const T* x, const T* coeff, T* y, const T* Tc, const int32_t* dofmap, int64_t ncells, int P,
                      void* stream) {
  if (ncells < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "mass_vertex: ncells < 0");
  if (P < 2 || P > 7) return fus_set_error(FUS_ERR_BAD_DEGREE, "mass_vertex: degree must be 2..7");
  if (ncells == 0) return 0;
  if (!x || !coeff || !y || !Tc || !dofmap) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "mass_vertex: null pointer");
  const long long total = (long long)ncells * (P + 1) * (P + 1) * (P + 1);
  long long grid = (total + kMassThreads - 1) / kMassThreads;
  const long long cap = (long long)fus_num_sms() * 16;
  if (grid > cap) grid = cap;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define FUS_CASE(N)                                                                                   \
  case N - 1:                                                                                         \
    mass_vertex_kernel<T, N><<<(unsigned)grid, kMassThreads, 0, st>>>(x, coeff, y, Tc, dofmap, total); \
    break;
  switch (P) {
    FUS_CASE(3)
    FUS_CASE(4)
    FUS_CASE(5)
    FUS_CASE(6)
    FUS_CASE(7)
    FUS_CASE(8)
  }
#undef FUS_CASE
  FUS_LAUNCH_CHECK("mass_vertex_kernel");
  return 0;
}

}  // namespace

FUS_CELL_TABLES(vertex)

#define FUS_VERTEX_API(SFX, T) FUS_CELL_API(SFX, T, _vertex, 3, (const T* Tc), a.Tc = Tc, (const T* Tc), a.Tc = Tc)

extern "C" {

int fus_trilinear_coeffs_f64(double* Tc, const int32_t* x_dofs, const double* x_g, const double* M,
                             int64_t ncells, void* stream) {
  return coeffs_entry<double>(Tc, x_dofs, x_g, M, ncells, stream);
}
int fus_trilinear_coeffs_f32(float* Tc, const int32_t* x_dofs, const float* x_g, const float* M,
                             int64_t ncells, void* stream) {
  return coeffs_entry<float>(Tc, x_dofs, x_g, M, ncells, stream);
}
int fus_set_vertex_tables_f64(int P, const double* x1, const double* w1, void* stream) {
  return set_vertex_tables<double>(P, x1, w1, static_cast<cudaStream_t>(stream));
}
int fus_set_vertex_tables_f32(int P, const float* x1, const float* w1, void* stream) {
  return set_vertex_tables<float>(P, x1, w1, static_cast<cudaStream_t>(stream));
}
FUS_VERTEX_API(f64, double)
FUS_VERTEX_API(f32, float)
#undef FUS_VERTEX_API
int fus_mass_vertex_f64(const double* x, const double* coeff, double* y, const double* Tc, const int32_t* dofmap,
                        int64_t ncells, int P, void* stream) {
  return mass_vertex_entry<double>(x, coeff, y, Tc, dofmap, ncells, P, stream);
}
int fus_mass_vertex_f32(const float* x, const float* coeff, float* y, const float* Tc, const int32_t* dofmap,
                        int64_t ncells, int P, void* stream) {
  return mass_vertex_entry<float>(x, coeff, y, Tc, dofmap, ncells, P, stream);
}

}  // extern "C"
