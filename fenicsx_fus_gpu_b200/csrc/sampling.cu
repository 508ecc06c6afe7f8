// Field sampling on the device: u at arbitrary points of the mesh.
//
// Replaces the output path of /root/reference/cuda/demo_linear_piston.py:564-570
// (demo_nonlinear_bowl.py:641-655): `u_n_d.copy_to_host(u_n)` of the WHOLE vector
// followed by `Function.eval(x_eval, cell_eval)` on the host.  Here only the sampled
// values leave the device:
//     out[p] = sum_{i,j,k} l_i(X_p) l_j(Y_p) l_k(Z_p) u[dofmap[cell_p, i n^2 + j n + k]]
// with the 1-D Lagrange values phi[p, d, :] tabulated once on the host (sampling.py) at
// the reference coordinates of the points.  One warp per point; fixed reduction order, so
// the result is bit-reproducible.  Bytes are negligible (n^3 gathers per point).

#include "fus_common.cuh"

namespace {

// u at point p, summed by one warp in a fixed order (every lane returns the total): the one sum
// behind eval_points_kernel and record_points_kernel, so a recorded value is bit-identical to an
// evaluation of the same vector
template <typename T>
__device__ __forceinline__ T warp_point_value(const T* __restrict__ u, const int32_t* __restrict__ dofmap,
                                              const int32_t* __restrict__ cells, const T* __restrict__ phi,
                                              long long p, int n, int lane) {
  const int n2 = n * n, n3 = n2 * n;
  const int32_t* dm = dofmap + (long long)cells[p] * n3;
  const T* ph = phi + p * 3 * n;
  T acc = T(0);
  for (int e = lane; e < n3; e += 32) {
    const int i = e / n2, r = e - i * n2, j = r / n, k = r - j * n;
    acc += ph[i] * ph[n + j] * ph[2 * n + k] * u[dm[e]];
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

template <typename T>
__global__ void eval_points_kernel(const T* __restrict__ u, const int32_t* __restrict__ dofmap,
                                   const int32_t* __restrict__ cells, const T* __restrict__ phi,
                                   T* __restrict__ out, long long npts, int n) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long p = warp; p < npts; p += nwarps) {
    const T acc = warp_point_value(u, dofmap, cells, phi, p, n, lane);
    if (lane == 0) out[p] = acc;
  }
}

// One row of a recording: out[row * npts + p] for every point, row = *step_base + *step_dev - first
// read on the device (a captured launch fills the right row at every replay); a row outside
// [0, rows) writes nothing.
template <typename T>
__global__ void record_points_kernel(const T* __restrict__ u, const int32_t* __restrict__ dofmap,
                                     const int32_t* __restrict__ cells, const T* __restrict__ phi,
                                     T* __restrict__ out, long long npts, int n,
                                     const long long* __restrict__ step_dev,
                                     const long long* __restrict__ step_base, long long first,
                                     long long rows) {
  const long long row = *step_base + (step_dev != nullptr ? *step_dev : 0) - first;
  if (row < 0 || row >= rows) return;
  T* __restrict__ o = out + row * npts;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long p = warp; p < npts; p += nwarps) {
    const T acc = warp_point_value(u, dofmap, cells, phi, p, n, lane);
    if (lane == 0) o[p] = acc;
  }
}

template <typename T>
int eval_entry(const T* u, const int32_t* dofmap, const int32_t* cells, const T* phi, T* out,
               int64_t npts, int P, void* stream) {
  if (npts < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "eval_points: npts < 0");
  if (P < 1 || P > 15) return fus_set_error(FUS_ERR_BAD_DEGREE, "eval_points: degree must be 1..15");
  if (npts == 0) return 0;
  if (!u || !dofmap || !cells || !phi || !out)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "eval_points: null pointer");
  const int threads = 256;
  long long blocks = (npts * 32 + threads - 1) / threads;
  const long long cap = (long long)fus_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  eval_points_kernel<T><<<(unsigned)blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      u, dofmap, cells, phi, out, npts, P + 1);
  FUS_LAUNCH_CHECK("eval_points_kernel");
  return 0;
}

template <typename T>
int record_entry(const T* u, const int32_t* dofmap, const int32_t* cells, const T* phi, T* out, int64_t npts,
                 int P, const int64_t* step_dev, const int64_t* step_base, int64_t first, int64_t rows,
                 void* stream) {
  if (npts < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "record_points: npts < 0");
  if (rows < 1) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "record_points: rows < 1");
  if (first < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "record_points: first < 0");
  if (P < 1 || P > 15) return fus_set_error(FUS_ERR_BAD_DEGREE, "record_points: degree must be 1..15");
  if (npts == 0) return 0;
  if (!u || !dofmap || !cells || !phi || !out || !step_base)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "record_points: null pointer");
  const int threads = 256;
  long long blocks = (npts * 32 + threads - 1) / threads;
  const long long cap = (long long)fus_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  record_points_kernel<T><<<(unsigned)blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      u, dofmap, cells, phi, out, npts, P + 1, reinterpret_cast<const long long*>(step_dev),
      reinterpret_cast<const long long*>(step_base), first, rows);
  FUS_LAUNCH_CHECK("record_points_kernel");
  return 0;
}

}  // namespace

extern "C" {
int fus_eval_points_f64(const double* u, const int32_t* dofmap, const int32_t* cells,
                        const double* phi, double* out, int64_t npts, int P, void* stream) {
  return eval_entry<double>(u, dofmap, cells, phi, out, npts, P, stream);
}
int fus_eval_points_f32(const float* u, const int32_t* dofmap, const int32_t* cells,
                        const float* phi, float* out, int64_t npts, int P, void* stream) {
  return eval_entry<float>(u, dofmap, cells, phi, out, npts, P, stream);
}
int fus_record_points_f64(const double* u, const int32_t* dofmap, const int32_t* cells,
                          const double* phi, double* out, int64_t npts, int P, const int64_t* step_dev,
                          const int64_t* step_base, int64_t first, int64_t rows, void* stream) {
  return record_entry<double>(u, dofmap, cells, phi, out, npts, P, step_dev, step_base, first, rows, stream);
}
int fus_record_points_f32(const float* u, const int32_t* dofmap, const int32_t* cells,
                          const float* phi, float* out, int64_t npts, int P, const int64_t* step_dev,
                          const int64_t* step_base, int64_t first, int64_t rows, void* stream) {
  return record_entry<float>(u, dofmap, cells, phi, out, npts, P, step_dev, step_base, first, rows, stream);
}
}
