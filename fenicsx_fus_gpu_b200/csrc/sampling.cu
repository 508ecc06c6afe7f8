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
//
// Element receivers: out[e] = sum_k w[k] u[dof[k]] over the entries of element e, the part of
// the integral of u over the element's facets held by this rank (sampling.ElementReceiver).

#include <cstdio>

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

// Element receivers.  The entries (dof, w) are element-major, and cut into chunks that never
// straddle two elements: chunk c is entries [chunk_beg[c], chunk_beg[c + 1]), the chunks of
// element e are [elem_chunk[e], elem_chunk[e + 1]).  Two launches: one warp per chunk writes the
// chunk's partial sum, then one warp per element sums its partials.  Inside a warp the lanes
// stride the range and a fixed xor-shuffle tree combines them, so the order of every sum is set
// by the format alone: not by the grid size or the number of SMs.

// range [b, e) of x summed by one warp: lane l takes b + l, b + l + 32, ...; every lane returns the total
template <typename T, typename F>
__device__ __forceinline__ T warp_range_sum(long long b, long long e, int lane, F x) {
  T acc = T(0);
  for (long long k = b + lane; k < e; k += 32) acc += x(k);
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

// the recording row (eager: step_base == nullptr, row 0 of a one-row output)
__device__ __forceinline__ long long element_row(const long long* __restrict__ step_dev,
                                                 const long long* __restrict__ step_base, long long first) {
  return step_base == nullptr ? 0 : *step_base + (step_dev != nullptr ? *step_dev : 0) - first;
}

template <typename T>
__global__ void element_partials_kernel(const T* __restrict__ u, const int32_t* __restrict__ dof,
                                        const T* __restrict__ w, const int32_t* __restrict__ chunk_beg,
                                        T* __restrict__ partial, long long nchunks,
                                        const long long* __restrict__ step_dev,
                                        const long long* __restrict__ step_base, long long first,
                                        long long rows) {
  const long long row = element_row(step_dev, step_base, first);
  if (row < 0 || row >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long c = warp; c < nchunks; c += nwarps) {
    const T acc = warp_range_sum<T>(chunk_beg[c], chunk_beg[c + 1], lane,
                                    [&](long long k) { return w[k] * u[dof[k]]; });
    if (lane == 0) partial[c] = acc;
  }
}

template <typename T>
__global__ void element_sums_kernel(const T* __restrict__ partial, const int32_t* __restrict__ elem_chunk,
                                    T* __restrict__ out, long long E,
                                    const long long* __restrict__ step_dev,
                                    const long long* __restrict__ step_base, long long first,
                                    long long rows) {
  const long long row = element_row(step_dev, step_base, first);
  if (row < 0 || row >= rows) return;
  T* __restrict__ o = out + row * E;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long e = warp; e < E; e += nwarps) {
    const T acc = warp_range_sum<T>(elem_chunk[e], elem_chunk[e + 1], lane,
                                    [&](long long c) { return partial[c]; });
    if (lane == 0) o[e] = acc;
  }
}

// one warp per item, 256 threads a block, at most 8 blocks per SM (grid-stride loops beyond)
inline unsigned warp_blocks(long long items) {
  const int threads = 256;
  long long blocks = (items * 32 + threads - 1) / threads;
  const long long cap = (long long)fus_num_sms() * 8;
  return (unsigned)(blocks > cap ? cap : blocks);
}

template <typename T>
int elements_entry(const char* what, const T* u, const int32_t* dof, const T* w, const int32_t* chunk_beg,
                   const int32_t* elem_chunk, T* partial, T* out, int64_t nchunks, int64_t E,
                   const int64_t* step_dev, const int64_t* step_base, int64_t first, int64_t rows,
                   bool recording, void* stream) {
  char msg[96];
  auto bad = [&](const char* why) {
    snprintf(msg, sizeof msg, "%s: %s", what, why);
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, msg);
  };
  if (nchunks < 0) return bad("nchunks < 0");
  if (E < 0) return bad("E < 0");
  if (rows < 1) return bad("rows < 1");
  if (first < 0) return bad("first < 0");
  if (E == 0 || nchunks == 0) return 0;
  if (!u || !dof || !w || !chunk_beg || !elem_chunk || !partial || !out || (recording && !step_base))
    return bad("null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long* sd = reinterpret_cast<const long long*>(step_dev);
  const long long* sb = reinterpret_cast<const long long*>(step_base);
  element_partials_kernel<T><<<warp_blocks(nchunks), 256, 0, st>>>(u, dof, w, chunk_beg, partial, nchunks, sd, sb,
                                                                    first, rows);
  FUS_LAUNCH_CHECK("element_partials_kernel");
  element_sums_kernel<T><<<warp_blocks(E), 256, 0, st>>>(partial, elem_chunk, out, E, sd, sb, first, rows);
  FUS_LAUNCH_CHECK("element_sums_kernel");
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
int fus_eval_elements_f64(const double* u, const int32_t* dof, const double* w, const int32_t* chunk_beg,
                          const int32_t* elem_chunk, double* partial, double* out, int64_t nchunks, int64_t E,
                          void* stream) {
  return elements_entry<double>("eval_elements", u, dof, w, chunk_beg, elem_chunk, partial, out, nchunks, E,
                                nullptr, nullptr, 0, 1, false, stream);
}
int fus_eval_elements_f32(const float* u, const int32_t* dof, const float* w, const int32_t* chunk_beg,
                          const int32_t* elem_chunk, float* partial, float* out, int64_t nchunks, int64_t E,
                          void* stream) {
  return elements_entry<float>("eval_elements", u, dof, w, chunk_beg, elem_chunk, partial, out, nchunks, E,
                               nullptr, nullptr, 0, 1, false, stream);
}
int fus_record_elements_f64(const double* u, const int32_t* dof, const double* w, const int32_t* chunk_beg,
                            const int32_t* elem_chunk, double* partial, double* out, int64_t nchunks, int64_t E,
                            const int64_t* step_dev, const int64_t* step_base, int64_t first, int64_t rows,
                            void* stream) {
  return elements_entry<double>("record_elements", u, dof, w, chunk_beg, elem_chunk, partial, out, nchunks, E,
                                step_dev, step_base, first, rows, true, stream);
}
int fus_record_elements_f32(const float* u, const int32_t* dof, const float* w, const int32_t* chunk_beg,
                            const int32_t* elem_chunk, float* partial, float* out, int64_t nchunks, int64_t E,
                            const int64_t* step_dev, const int64_t* step_base, int64_t first, int64_t rows,
                            void* stream) {
  return elements_entry<float>("record_elements", u, dof, w, chunk_beg, elem_chunk, partial, out, nchunks, E,
                               step_dev, step_base, first, rows, true, stream);
}
}
