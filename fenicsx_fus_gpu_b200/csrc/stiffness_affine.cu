// Stiffness action on AFFINE hexahedra (constant Jacobian), degree 2..7, sm_100a.
//
// The reference streams 6*n^3 geometric factors per cell whatever the cell
// (/root/reference/cuda/operators.py:154-164 reads G_entity[cell, q, 0..5];
// cuda/precompute.py:116-163 fills it).  On a parallelepiped J is constant, so
//     G[c, q, :] = wq[q] * Gc[c, :],     detJ[c, q] = wq[q] * detJc[c]
// and the action needs 6 (+1) values per cell instead of 6 (+1) n^3: the kernel is
// the AFF instantiation of stiffness_kernel.cuh - same pencil-ownership contractions
// and register prefetch of dofmap / x, no TMA ring - and is bound by the shared-memory
// pipe and the x / y / dofmap traffic instead of by the G stream.
// HBM bytes per cell: Nd*4 (dofmap) + 7s, plus 2s per global dof.

#include "stiffness_kernel.cuh"

namespace {

template <typename T>
int set_rect_tables(int P, const T* k1, const T* w1, cudaStream_t stream) {
  if (P < 2 || P > 7) return fus_set_error(FUS_ERR_BAD_DEGREE, "set_rect_tables: degree must be 2..7");
  if (k1 == nullptr || w1 == nullptr) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "set_rect_tables: null table");
  const int n = P + 1;
  if constexpr (sizeof(T) == 8) {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_K64, k1, sizeof(T) * n * n, sizeof(T) * 64 * (P - 2), cudaMemcpyDefault, stream));
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_W64, w1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
  } else {
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_K32, k1, sizeof(T) * n * n, sizeof(T) * 64 * (P - 2), cudaMemcpyDefault, stream));
    FUS_CUDA(cudaMemcpyToSymbolAsync(c_W32, w1, sizeof(T) * n, sizeof(T) * 8 * (P - 2), cudaMemcpyDefault, stream));
  }
  return 0;
}

// one CTA per cell: mean of the weight-normalised records and their largest deviation from it
template <typename T>
__global__ void compress_geometry_kernel(const T* __restrict__ G, const T* __restrict__ detJ,
                                         const T* __restrict__ wq, T* __restrict__ Gc,
                                         T* __restrict__ detJc, int32_t* __restrict__ affine,
                                         long long ncells, int nq, T tol) {
  __shared__ double red[7][8];
  __shared__ double mean[7];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (long long c = blockIdx.x; c < ncells; c += gridDim.x) {
    double acc[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int q = threadIdx.x; q < nq; q += blockDim.x) {
      const double w = 1.0 / (double)wq[q];
      const T* g = G + (c * nq + q) * 6;
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] += (double)g[k] * w;
      if (detJ) acc[6] += (double)detJ[c * nq + q] * w;
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      double v = acc[k];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[k][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
      double v = 0;
      for (int w = 0; w < nw; ++w) v += red[threadIdx.x][w];
      mean[threadIdx.x] = v / nq;
    }
    __syncthreads();
    double scale = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) scale = fmax(scale, fabs(mean[k]));
    double dev = 0;  // largest deviation relative to its scale
    for (int q = threadIdx.x; q < nq; q += blockDim.x) {
      const double w = 1.0 / (double)wq[q];
      const T* g = G + (c * nq + q) * 6;
#pragma unroll
      for (int k = 0; k < 6; ++k) dev = fmax(dev, fabs((double)g[k] * w - mean[k]) / scale);
      if (detJ) dev = fmax(dev, fabs((double)detJ[c * nq + q] * w - mean[6]) / fabs(mean[6]));
    }
    for (int o = 16; o; o >>= 1) dev = fmax(dev, __shfl_xor_sync(0xffffffffu, dev, o));
    __syncthreads();
    if (lane == 0) red[0][warp] = dev;
    __syncthreads();
    if (threadIdx.x == 0) {
      double v = 0;
      for (int w = 0; w < nw; ++w) v = fmax(v, red[0][w]);
      affine[c] = (v <= (double)tol) ? 1 : 0;  // NaN / zero scale compare false -> streamed
#pragma unroll
      for (int k = 0; k < 6; ++k) Gc[c * 6 + k] = (T)mean[k];
      if (detJc) detJc[c] = (T)mean[6];
    }
    __syncthreads();
  }
}

template <typename T>
int compress_entry(const T* G, const T* detJ, const T* wq, T* Gc, T* detJc, int32_t* affine,
                   int64_t ncells, int nq, T tol, void* stream) {
  if (ncells < 0 || nq <= 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "compress_geometry: bad sizes");
  if (ncells == 0) return 0;
  if (!G || !wq || !Gc || !affine) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "compress_geometry: null pointer");
  long long grid = (long long)fus_num_sms() * 16;
  if (grid > ncells) grid = ncells;
  compress_geometry_kernel<T><<<(unsigned)grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      G, detJ, wq, Gc, detJc, affine, ncells, nq, tol);
  FUS_LAUNCH_CHECK("compress_geometry_kernel");
  return 0;
}

}  // namespace

FUS_CELL_TABLES(affine)

// GEO 1 = affine cells (Gc x wq), GEO 2 = rectilinear cells (diagonal Gc, tensor-product weights
// from fus_set_rect_tables; no wq)
#define FUS_AFFINE_API(SFX, T)                                                                      \
  FUS_CELL_API(SFX, T, _affine, 1, (const T* Gc, const T* wq), a.Gc = Gc; a.wq = wq,                \
               (const T* Gc, const T* detJc, const T* wq), a.Gc = Gc; a.detJc = detJc; a.wq = wq)   \
  FUS_CELL_API(SFX, T, _rect, 2, (const T* Gc), a.Gc = Gc, (const T* Gc, const T* detJc),           \
               a.Gc = Gc; a.detJc = detJc)

extern "C" {

FUS_AFFINE_API(f64, double)
FUS_AFFINE_API(f32, float)
#undef FUS_AFFINE_API

int fus_set_rect_tables_f64(int P, const double* k1, const double* w1, void* stream) {
  return set_rect_tables<double>(P, k1, w1, static_cast<cudaStream_t>(stream));
}
int fus_set_rect_tables_f32(int P, const float* k1, const float* w1, void* stream) {
  return set_rect_tables<float>(P, k1, w1, static_cast<cudaStream_t>(stream));
}
int fus_compress_geometry_f64(const double* G, const double* detJ, const double* wq, double* Gc,
                              double* detJc, int32_t* affine, int64_t ncells, int nq, double tol,
                              void* stream) {
  return compress_entry<double>(G, detJ, wq, Gc, detJc, affine, ncells, nq, tol, stream);
}
int fus_compress_geometry_f32(const float* G, const float* detJ, const float* wq, float* Gc,
                              float* detJc, int32_t* affine, int64_t ncells, int nq, float tol,
                              void* stream) {
  return compress_entry<float>(G, detJ, wq, Gc, detJc, affine, ncells, nq, tol, stream);
}

}  // extern "C"
