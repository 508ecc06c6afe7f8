// Sum-factorised stiffness action on hexahedra, degree 2..7, sm_100a.
//
// Replaces the Numba kernel of /root/reference/cuda/operators.py:73-192
// (one CTA of n^3 threads per cell, 4 smem tiles, 6n smem + 6n global loads
// per thread, AoS G read with 6 strided scalar loads, one fp atomic per
// node).  Same arithmetic:
//     g_d  = sum_l D[q_d, l] u[.. l ..]                     (:138-151)
//     f    = coeff * Gsym * g                               (:154-164)
//     y_j  = sum_d sum_q D[q, j_d] f_d[.. q ..]             (:171-187)
//     y[dofmap] += y_j                                      (:190)
//
// Design (B200 first).  ncu on the first version of this kernel showed the
// L1/shared-memory data pipe (not HBM, not FP64) as the limiter, so the kernel
// is organised to minimise shared-memory wavefronts per cell:
//   * persistent CTAs, one batch of B cells per iteration, n^2 threads per
//     cell.  Every 1-D contraction is done by the thread that owns the whole
//     pencil along the contraction direction, in registers, with the entries
//     of D as compile-time constant-bank operands: thread (j,k) owns x
//     pencils, thread (i,k) owns y pencils, thread (i,j) owns z pencils.
//     Moving between the three ownerships costs one write + one read of the
//     tile (n values per thread) instead of n^2 operand loads per thread;
//   * two shared-memory tiles per cell with different paddings, UY (plane
//     stride = n mod M) and UZ (plane stride = 1 mod M, M = banks per
//     wavefront), make ALL access patterns of the three ownerships
//     bank-conflict free (tools/smem_layout_search.py);
//   * G (the dominant HBM stream, 6*n^3 values per cell) of the NEXT batch is
//     fetched by the TMA unit (cp.async.bulk + mbarrier complete_tx, one copy
//     per cell into a slot padded so that 16-byte AoS record loads stay
//     conflict free across cell boundaries) into a 2-stage ring while the
//     current batch computes; the reference's AoS layout [cell][q][6] is
//     accepted as is;
//   * the dofmap entries and the gathered x values of the NEXT batch are
//     prefetched into registers (each thread gathers and scatters exactly its
//     own x pencil, coalesced over (j,k)), so no global-load latency is exposed
//     inside a batch; scatter is fire-and-forget RED atomics (or plain RMW when
//     the caller colours the cells).
//
// HBM-bound: algorithmic bytes per cell = Nd*4 (dofmap) + 6*Nd*s (G) + s
// (coeff) plus 2s per global dof for x and y (SURVEY.md section 8d).

#include "stiffness_kernel.cuh"

template <typename T>
int fus_affine_set_dphi(int P, const T* dphi, cudaStream_t stream);  // stiffness_affine.cu
template <typename T>
int fus_vertex_set_dphi(int P, const T* dphi, cudaStream_t stream);  // stiffness_vertex.cu

namespace {

// ---- host-buffer entry point: H2D of x (and y), the action, D2H of y, pipelined -------------
//
// The cells are cut into kHostChunks ranges.  A reduction over the dofmap gives the dof interval
// [lo_c, hi_c] every range touches; with H_c = max_{c' <= c} hi_c' and L_c = min_{c' >= c} lo_c',
// range c may run as soon as x[0, H_c] has arrived, and y[0, L_{c+1}) is final as soon as range c
// has run.  So the upload of piece c+1, the kernel of range c and the download of what range c-1
// finished proceed concurrently on three streams (PCIe is full duplex).  On a mesh whose cell
// order follows its dof order (every box mesh here, any mesh after a bandwidth-reducing
// renumbering) the pieces are ~1/kHostChunks of the vectors; on an unordered mesh H_0 ~ nd and
// the pipeline degenerates, correctly, into upload -> action -> download.
constexpr int kHostChunks = 8;

__global__ void __launch_bounds__(256) dof_range_kernel(const int32_t* __restrict__ dofmap, long long ncells,
                                                        int Nd, long long cells_per_chunk, int* lo, int* hi) {
  const int c = blockIdx.y;
  const long long c0 = c * cells_per_chunk;
  long long c1 = c0 + cells_per_chunk;
  if (c1 > ncells) c1 = ncells;
  const long long e0 = c0 * Nd, e1 = c1 * Nd;
  int mn = 0x7fffffff, mx = -1;
  for (long long e = e0 + (long long)blockIdx.x * 256 + threadIdx.x; e < e1; e += (long long)gridDim.x * 256) {
    const int d = dofmap[e];
    mn = d < mn ? d : mn;
    mx = d > mx ? d : mx;
  }
  mn = __reduce_min_sync(0xffffffffu, mn);
  mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0) {
    atomicMin(lo + c, mn);
    atomicMax(hi + c, mx);
  }
}

struct HostPipe {
  cudaStream_t in = nullptr, out = nullptr;
  cudaEvent_t start = nullptr, up[kHostChunks] = {}, done[kHostChunks] = {}, fin = nullptr;
  int* ranges_dev = nullptr;   // lo[kHostChunks], hi[kHostChunks]
  int* ranges_host = nullptr;  // pinned
  bool ok = false;
};

HostPipe* host_pipe() {
  static HostPipe pipes[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  HostPipe& p = pipes[dev];
  if (!p.ok) {
    bool good = cudaStreamCreateWithFlags(&p.in, cudaStreamNonBlocking) == cudaSuccess &&
                cudaStreamCreateWithFlags(&p.out, cudaStreamNonBlocking) == cudaSuccess &&
                cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming) == cudaSuccess &&
                cudaEventCreateWithFlags(&p.fin, cudaEventDisableTiming) == cudaSuccess &&
                cudaMalloc(&p.ranges_dev, 2 * kHostChunks * sizeof(int)) == cudaSuccess &&
                cudaMallocHost(&p.ranges_host, 2 * kHostChunks * sizeof(int)) == cudaSuccess;
    for (int c = 0; c < kHostChunks && good; ++c)
      good = cudaEventCreateWithFlags(&p.up[c], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&p.done[c], cudaEventDisableTiming) == cudaSuccess;
    if (!good) return nullptr;
    p.ok = true;
  }
  return &p;
}

template <typename T>
int stiffness_host(const T* x_host, T* y_host, int64_t nd, T* x_dev, T* y_dev, const T* coeff, const T* G,
                   const int32_t* dofmap, const T* dphi, int64_t ncells, int P, int flags, void* stream) {
  if (ncells < 0 || nd < 0) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "stiffness_host: negative size");
  if (P < 2 || P > 7) return fus_set_error(FUS_ERR_BAD_DEGREE, "stiffness_host: degree must be 2..7");
  if (nd == 0) return 0;
  if (x_host == nullptr || y_host == nullptr || x_dev == nullptr || y_dev == nullptr)
    return fus_set_error(FUS_ERR_BAD_ARGUMENT, "stiffness_host: null buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool yzero = (flags & FUS_HOST_Y_ZERO) != 0;
  const int kflags = flags & ~FUS_HOST_Y_ZERO;
  const int Nd = (P + 1) * (P + 1) * (P + 1);
  HostPipe* hp = host_pipe();
  auto action = [&](long long c0, long long nc, int fl) {  // y_dev += K x_dev on cells [c0, c0 + nc)
    StiffArgs<T> a{};
    a.xa = x_dev, a.ca = coeff + c0, a.y = y_dev, a.G = G + c0 * Nd * 6, a.dofmap = dofmap + c0 * Nd, a.ncells = nc;
    return cell_entry<T, 0, 0>(a, dphi, P, fl, stream, "stiffness_host");
  };
  // cells per range: even, so that every range's G slice keeps the 16-byte alignment of the base
  long long cpc = ((ncells + kHostChunks - 1) / kHostChunks + 1) / 2 * 2;
  if (hp == nullptr || ncells < 64 * kHostChunks) {
    // tiny problems (or no side streams): upload, action, download on the caller's stream
    FUS_CUDA(cudaMemcpyAsync(x_dev, x_host, sizeof(T) * nd, cudaMemcpyHostToDevice, st));
    if (yzero) {
      FUS_CUDA(cudaMemsetAsync(y_dev, 0, sizeof(T) * nd, st));
    } else {
      FUS_CUDA(cudaMemcpyAsync(y_dev, y_host, sizeof(T) * nd, cudaMemcpyHostToDevice, st));
    }
    if (int rc = action(0, ncells, kflags)) return rc;
    FUS_CUDA(cudaMemcpyAsync(y_host, y_dev, sizeof(T) * nd, cudaMemcpyDeviceToHost, st));
    FUS_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  // 1. dof interval of every cell range (one pass over the dofmap on the device)
  int init[2 * kHostChunks];
  for (int c = 0; c < kHostChunks; ++c) {
    init[c] = 0x7fffffff;
    init[kHostChunks + c] = -1;
  }
  FUS_CUDA(cudaMemcpyAsync(hp->ranges_dev, init, sizeof(init), cudaMemcpyHostToDevice, st));
  dof_range_kernel<<<dim3(64, kHostChunks), 256, 0, st>>>(dofmap, ncells, Nd, cpc, hp->ranges_dev,
                                                         hp->ranges_dev + kHostChunks);
  FUS_LAUNCH_CHECK("dof_range_kernel");
  FUS_CUDA(cudaMemcpyAsync(hp->ranges_host, hp->ranges_dev, sizeof(init), cudaMemcpyDeviceToHost, st));
  if (yzero) FUS_CUDA(cudaMemsetAsync(y_dev, 0, sizeof(T) * nd, st));
  if (!(kflags & FUS_TABLES_RESIDENT)) {
    if (int rc = set_dphi<T>(P, dphi, st)) return rc;
  }
  FUS_CUDA(cudaEventRecord(hp->start, st));
  FUS_CUDA(cudaStreamSynchronize(st));
  long long H[kHostChunks], L[kHostChunks + 1];
  long long run = -1;
  for (int c = 0; c < kHostChunks; ++c) {
    const long long hi = hp->ranges_host[kHostChunks + c];
    if (hi >= nd) return fus_set_error(FUS_ERR_BAD_ARGUMENT, "stiffness_host: dofmap entry >= nd");
    run = hi > run ? hi : run;
    H[c] = run + 1;  // x[0, H_c) must be resident before range c
  }
  H[kHostChunks - 1] = nd;
  L[kHostChunks] = nd;
  for (int c = kHostChunks - 1; c >= 0; --c) {
    long long lo = hp->ranges_host[c];
    if (lo == 0x7fffffff) lo = nd;  // empty range
    L[c] = lo < L[c + 1] ? lo : L[c + 1];
  }
  // 2. three-stream pipeline
  FUS_CUDA(cudaStreamWaitEvent(hp->in, hp->start, 0));
  FUS_CUDA(cudaStreamWaitEvent(hp->out, hp->start, 0));
  long long up0 = 0, down0 = 0;
  for (int c = 0; c < kHostChunks; ++c) {
    const long long c0 = c * cpc;
    long long nc = ncells - c0;
    if (nc > cpc) nc = cpc;
    if (H[c] > up0) {
      FUS_CUDA(cudaMemcpyAsync(x_dev + up0, x_host + up0, sizeof(T) * (H[c] - up0), cudaMemcpyHostToDevice, hp->in));
      if (!yzero)
        FUS_CUDA(cudaMemcpyAsync(y_dev + up0, y_host + up0, sizeof(T) * (H[c] - up0), cudaMemcpyHostToDevice, hp->in));
      up0 = H[c];
    }
    FUS_CUDA(cudaEventRecord(hp->up[c], hp->in));
    FUS_CUDA(cudaStreamWaitEvent(st, hp->up[c], 0));
    if (nc > 0) {
      if (int rc = action(c0, nc, kflags | FUS_TABLES_RESIDENT)) return rc;
    }
    FUS_CUDA(cudaEventRecord(hp->done[c], st));
    const long long fin = L[c + 1];  // y[0, fin) is final now
    if (fin > down0) {
      FUS_CUDA(cudaStreamWaitEvent(hp->out, hp->done[c], 0));
      FUS_CUDA(cudaMemcpyAsync(y_host + down0, y_dev + down0, sizeof(T) * (fin - down0), cudaMemcpyDeviceToHost, hp->out));
      down0 = fin;
    }
  }
  FUS_CUDA(cudaEventRecord(hp->fin, hp->out));
  FUS_CUDA(cudaStreamWaitEvent(st, hp->fin, 0));
  FUS_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// every unit that includes stiffness_kernel.cuh holds its own copy of the derivative table
template <typename T>
int set_dphi_all(int P, const T* dphi, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = set_dphi<T>(P, dphi, st);
  if (!rc) rc = fus_affine_set_dphi<T>(P, dphi, st);
  return rc ? rc : fus_vertex_set_dphi<T>(P, dphi, st);
}

}  // namespace

#define FUS_STREAMED_API(SFX, T)                                                        \
  FUS_CELL_API(SFX, T, , 0, (const T* G), a.G = G, (const T* G, const T* detJ), a.G = G; a.detJ = detJ) \
  int fus_set_dphi_##SFX(int P, const T* dphi, void* stream) { return set_dphi_all<T>(P, dphi, stream); } \
  int fus_stiffness_host_##SFX(const T* x_host, T* y_host, int64_t nd, T* x_dev, T* y_dev, const T* coeff,  \
                               const T* G, const int32_t* dofmap, const T* dphi, int64_t ncells, int P,     \
                               int flags, void* stream) {                                                    \
    return stiffness_host<T>(x_host, y_host, nd, x_dev, y_dev, coeff, G, dofmap, dphi, ncells, P, flags, stream); \
  }

extern "C" {
FUS_STREAMED_API(f64, double)
FUS_STREAMED_API(f32, float)
}  // extern "C"
#undef FUS_STREAMED_API
