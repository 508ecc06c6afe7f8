/*
 * fus_b200.h - C ABI of the B200-native (sm_100a) wave-propagation hot path.
 *
 * This is the drop-in boundary for fenicsx-fus-gpu's matrix-free explicit
 * spectral-element path.  The reference has no native ABI of its own: its
 * device code is Numba @cuda.jit kernels launched from Python
 * (/root/reference/cuda/operators.py, scatterer.py).  Each entry point below
 * names the reference kernel / function (file:line) it replaces; the Python
 * host layer (fenicsx_fus_gpu_b200/operators.py ...) binds them with ctypes
 * behind the reference's own call surface, see INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as
 *     void* (NULL = legacy default stream);
 *   - unless a name ends in `_host`, every data pointer is a DEVICE pointer
 *     owned by the caller; nothing is allocated or freed behind its back;
 *   - launches are asynchronous on `stream`; ordering is stream ordering, as
 *     with the reference's Numba launches;
 *   - return value 0 on success, otherwise a cudaError_t value (or
 *     FUS_ERR_* below); fus_last_error() gives the text.  Never throws.
 *   - `_f32` / `_f64` select the float type (the reference's `float_type`).
 *   - `P` is the polynomial degree, 2..7; n = P+1; Nd = n^3.
 */
#ifndef FUS_B200_H
#define FUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FUS_ABI_VERSION 2

/* error codes outside the cudaError_t range */
#define FUS_ERR_BAD_DEGREE 100001
#define FUS_ERR_BAD_ARGUMENT 100002
#define FUS_ERR_HALO_TIMEOUT 100003

/* flags for fus_stiffness* */
#define FUS_TABLES_RESIDENT 1 /* dphi for this (P, type) already uploaded: skip the table copy */
#define FUS_NO_ATOMICS 2      /* caller guarantees no two cells of this launch share a dof (colouring) */
#define FUS_HOST_Y_ZERO 4     /* fus_stiffness_host_*: y_host holds zeros - skip its upload, clear y on the device */

int fus_abi_version(void);
const char* fus_last_error(void);
/* Number of device kernels this library has launched since load / last reset
 * (bench.py's `gpu_launches`). */
int64_t fus_launch_count(void);
void fus_reset_launch_count(void);

/* --------------------------------------------------------------------- *
 * Element operators
 * --------------------------------------------------------------------- */

/* Upload the 1-D derivative table dphi[q*n + i] = l_i'(x_q) for degree P to
 * the constant bank the stiffness kernels read.  `dphi` may be a host or a
 * device pointer.  Replaces the `dphi` kernel argument of
 * cuda/operators.py:88-95 (read per thread from global at :138-151). */
int fus_set_dphi_f64(int P, const double* dphi, void* stream);
int fus_set_dphi_f32(int P, const float* dphi, void* stream);

/* Stiffness action  y[dm[c,:]] += D^T-apply( coeff[c] * Gsym[c,q] * (D-apply x[dm[c,:]]) ).
 * Replaces `stiffness_operator(P, float_type)[ncells, (n,n,n)](x, coeff, y, G, dofmap, dphi)`
 * - cuda/operators.py:73-192 (CPU twin numba-cpu/operators.py:71-227,
 * C++ cpp/common/spectral_op.hpp:173-243).
 *   x, y   : (nd,)            y is accumulated into (caller zero-fills)
 *   coeff  : (ncells,)
 *   G      : (ncells, Nd, 6)  C order, [G00 G01 G02 G11 G12 G22] (cuda/precompute.py:158-163)
 *   dofmap : (ncells, Nd)     int32, tensor-product order q = i*n*n + j*n + k
 *   dphi   : (n, n)           device or host; ignored with FUS_TABLES_RESIDENT */
int fus_stiffness_f64(const double* x, const double* coeff, double* y, const double* G,
                      const int32_t* dofmap, const double* dphi, int64_t ncells, int P,
                      int flags, void* stream);
int fus_stiffness_f32(const float* x, const float* coeff, float* y, const float* G,
                      const int32_t* dofmap, const float* dphi, int64_t ncells, int P,
                      int flags, void* stream);

/* Two stiffness actions sharing ONE read of G:
 *   y += K(coeff_a ; xa) + K(coeff_b ; xb)
 * Replaces the two back-to-back launches of the Westervelt stage,
 * cuda/demo_nonlinear_bowl.py:620-625. */
int fus_stiffness2_f64(const double* xa, const double* coeff_a, const double* xb,
                       const double* coeff_b, double* y, const double* G,
                       const int32_t* dofmap, const double* dphi, int64_t ncells, int P,
                       int flags, void* stream);
int fus_stiffness2_f32(const float* xa, const float* coeff_a, const float* xb,
                       const float* coeff_b, float* y, const float* G, const int32_t* dofmap,
                       const float* dphi, int64_t ncells, int P, int flags, void* stream);

/* The whole cell work of one Westervelt stage in ONE pass over G, detJ and the
 * dofmap (cuda/demo_nonlinear_bowl.py:609-612 and 620-628):
 *   b += K(c3 ; un) + K(c4 ; vn) + M(c5 ; vn^2)        m += M(c2 ; un)
 * with M(c ; w)[dm] = c * detJ * w[dm].  un and vn are gathered once. */
int fus_stiffness_westervelt_f64(const double* un, const double* c3, const double* vn,
                                 const double* c4, const double* c2, const double* c5, double* m,
                                 double* b, const double* G, const double* detJ,
                                 const int32_t* dofmap, const double* dphi, int64_t ncells, int P,
                                 int flags, void* stream);
int fus_stiffness_westervelt_f32(const float* un, const float* c3, const float* vn, const float* c4,
                                 const float* c2, const float* c5, float* m, float* b,
                                 const float* G, const float* detJ, const int32_t* dofmap,
                                 const float* dphi, int64_t ncells, int P, int flags, void* stream);

/* Affine-cell variants (no counterpart in the reference, which always streams the full
 * G of cuda/precompute.py:116-163).  On a cell with a constant Jacobian (parallelepiped:
 * every cell of the box demos) the tables factor exactly,
 *   G[c, q, :] = wq[q] * Gc[c, :]      detJ[c, q] = wq[q] * detJc[c],
 * wq (n^3) being the tensor quadrature weights, so a launch reads 6 (7) values per cell
 * instead of 6 (7) n^3.  Same arithmetic as fus_stiffness_* / fus_stiffness_westervelt_* with
 * the product wq[q] * Gc formed in registers; results agree with the streamed kernels to
 * rounding.  Gc: (ncells, 6), detJc: (ncells,), wq: (n^3,) in quadrature order q = i n^2 + j n + k
 * (fus_compress_geometry_* builds them from G and says which cells qualify). */
int fus_stiffness_affine_f64(const double* x, const double* coeff, double* y, const double* Gc,
                             const double* wq, const int32_t* dofmap, const double* dphi,
                             int64_t ncells, int P, int flags, void* stream);
int fus_stiffness_affine_f32(const float* x, const float* coeff, float* y, const float* Gc,
                             const float* wq, const int32_t* dofmap, const float* dphi,
                             int64_t ncells, int P, int flags, void* stream);
int fus_stiffness_westervelt_affine_f64(const double* un, const double* c3, const double* vn,
                                        const double* c4, const double* c2, const double* c5,
                                        double* m, double* b, const double* Gc,
                                        const double* detJc, const double* wq,
                                        const int32_t* dofmap, const double* dphi, int64_t ncells,
                                        int P, int flags, void* stream);
int fus_stiffness_westervelt_affine_f32(const float* un, const float* c3, const float* vn,
                                        const float* c4, const float* c2, const float* c5, float* m,
                                        float* b, const float* Gc, const float* detJc,
                                        const float* wq, const int32_t* dofmap, const float* dphi,
                                        int64_t ncells, int P, int flags, void* stream);

/* Rectilinear cells: affine AND Gc diagonal (axis-aligned box cells: Gc[c,1] = Gc[c,2] =
 * Gc[c,4] = 0) with tensor-product weights wq[i n^2 + j n + k] = w1[i] w1[j] w1[k].  The three
 * directions decouple,
 *   y = coeff * sum_d Gc[c,dd] * (w1 x w1) (x) K1 u,   K1 = D^T diag(w1) D  (n x n, constant),
 * so each pencil needs one n x n product per direction and no gradient ever changes
 * ownership: half the shared-memory traffic and FP work of the affine kernels.  Same operator
 * as fus_stiffness_* on such cells (results agree to rounding).  fus_set_rect_tables uploads
 * K1 (n*n, row-major) and w1 (n) for degree P (host or device pointers); Gc is (ncells, 6) as
 * above (entries 0, 3, 5 are read). */
int fus_set_rect_tables_f64(int P, const double* k1, const double* w1, void* stream);
int fus_set_rect_tables_f32(int P, const float* k1, const float* w1, void* stream);
int fus_stiffness_rect_f64(const double* x, const double* coeff, double* y, const double* Gc,
                           const int32_t* dofmap, const double* dphi, int64_t ncells, int P,
                           int flags, void* stream);
int fus_stiffness_rect_f32(const float* x, const float* coeff, float* y, const float* Gc,
                           const int32_t* dofmap, const float* dphi, int64_t ncells, int P, int flags,
                           void* stream);
int fus_stiffness_westervelt_rect_f64(const double* un, const double* c3, const double* vn,
                                      const double* c4, const double* c2, const double* c5,
                                      double* m, double* b, const double* Gc, const double* detJc,
                                      const int32_t* dofmap, const double* dphi, int64_t ncells,
                                      int P, int flags, void* stream);
int fus_stiffness_westervelt_rect_f32(const float* un, const float* c3, const float* vn,
                                      const float* c4, const float* c2, const float* c5, float* m,
                                      float* b, const float* Gc, const float* detJc,
                                      const int32_t* dofmap, const float* dphi, int64_t ncells, int P,
                                      int flags, void* stream);

/* y += K(ca; xa) + K(cb; xb) on affine / rectilinear cells (fus_stiffness2_* with compressed geometry). */
int fus_stiffness2_affine_f64(const double* xa, const double* ca, const double* xb, const double* cb,
                              double* y, const double* Gc, const double* wq, const int32_t* dofmap,
                              const double* dphi, int64_t ncells, int P, int flags, void* stream);
int fus_stiffness2_affine_f32(const float* xa, const float* ca, const float* xb, const float* cb,
                              float* y, const float* Gc, const float* wq, const int32_t* dofmap,
                              const float* dphi, int64_t ncells, int P, int flags, void* stream);
int fus_stiffness2_rect_f64(const double* xa, const double* ca, const double* xb, const double* cb,
                            double* y, const double* Gc, const int32_t* dofmap, const double* dphi,
                            int64_t ncells, int P, int flags, void* stream);
int fus_stiffness2_rect_f32(const float* xa, const float* ca, const float* xb, const float* cb,
                            float* y, const float* Gc, const int32_t* dofmap, const float* dphi,
                            int64_t ncells, int P, int flags, void* stream);

/* Trilinear cells with the geometry recomputed in the kernel (the on-the-fly-geometry mode; replaces the
 * G stream of cuda/operators.py:154-164 and the table cuda/precompute.py:115-163 fills): the map of a hexahedron
 * with 8 vertices is trilinear, so the tangent dx/dxi_d is bilinear in the other two reference coordinates
 * (u, v) = (eta, zeta), (xi, zeta), (xi, eta) for d = 0, 1, 2:
 *     t_d = Tc[c,d,0,:] + u Tc[c,d,1,:] + v Tc[c,d,2,:] + u v Tc[c,d,3,:]
 * fus_trilinear_coeffs_* : Tc (ncells, 3, 4, 3) = M (3, 4, 8) applied to the cell's vertex coordinates, where M is the
 *     bilinear expansion of the P1 derivative table, dphi[d, q, v] = sum_m M[d, m, v] {1, u, v, u v}_m (pts[q])
 *     (precompute.trilinear_expansion fits it from the same dphi / points cuda/precompute.py takes).
 * fus_set_vertex_tables_* : the n 1-D quadrature points and weights in dof order (host or device).
 * fus_stiffness_vertex_* / fus_stiffness2_vertex_* : y += K(coeff; x) / y += K(ca; xa) + K(cb; xb) with
 *     G = w |det J| J^-1 J^-T rebuilt at every point (same result as fus_stiffness_* to rounding);
 *     37 values per cell instead of 6 n^3 + 1. */
int fus_trilinear_coeffs_f64(double* Tc, const int32_t* x_dofs, const double* x_g, const double* M,
                             int64_t ncells, void* stream);
int fus_trilinear_coeffs_f32(float* Tc, const int32_t* x_dofs, const float* x_g, const float* M,
                             int64_t ncells, void* stream);
int fus_set_vertex_tables_f64(int P, const double* x1, const double* w1, void* stream);
int fus_set_vertex_tables_f32(int P, const float* x1, const float* w1, void* stream);
int fus_stiffness_vertex_f64(const double* x, const double* coeff, double* y, const double* Tc,
                             const int32_t* dofmap, const double* dphi, int64_t ncells, int P, int flags,
                             void* stream);
int fus_stiffness_vertex_f32(const float* x, const float* coeff, float* y, const float* Tc,
                             const int32_t* dofmap, const float* dphi, int64_t ncells, int P, int flags,
                             void* stream);
int fus_stiffness2_vertex_f64(const double* xa, const double* ca, const double* xb, const double* cb,
                              double* y, const double* Tc, const int32_t* dofmap, const double* dphi,
                              int64_t ncells, int P, int flags, void* stream);
int fus_stiffness2_vertex_f32(const float* xa, const float* ca, const float* xb, const float* cb, float* y,
                              const float* Tc, const int32_t* dofmap, const float* dphi, int64_t ncells,
                              int P, int flags, void* stream);
/* fus_stiffness_westervelt_vertex_* : fus_stiffness_westervelt_* on trilinear cells, Tc in place of G and detJ:
 *     b += K(c3 ; un) + K(c4 ; vn) + M(c5 ; vn^2)        m += M(c2 ; un)
 *     with M(c ; w)[dm] = c * w_q |det J(X_q)| * w[dm] taken from the same tangents as the stiffness.
 *     Not combinable with FUS_NO_ATOMICS.
 * fus_mass_vertex_* : the lumped mass y[dm[c,q]] += coeff[c] * w_q |det J_c(X_q)| * x[dm[c,q]] (fus_mass_* with
 *     ncols = n^3 and the detJ table recomputed from Tc); reads the tables of fus_set_vertex_tables_*.  A solver
 *     on trilinear cells builds its masses with it and never holds a (ncells, n^3) table. */
int fus_stiffness_westervelt_vertex_f64(const double* un, const double* c3, const double* vn, const double* c4,
                                        const double* c2, const double* c5, double* m, double* b, const double* Tc,
                                        const int32_t* dofmap, const double* dphi, int64_t ncells, int P, int flags,
                                        void* stream);
int fus_stiffness_westervelt_vertex_f32(const float* un, const float* c3, const float* vn, const float* c4,
                                        const float* c2, const float* c5, float* m, float* b, const float* Tc,
                                        const int32_t* dofmap, const float* dphi, int64_t ncells, int P, int flags,
                                        void* stream);
int fus_mass_vertex_f64(const double* x, const double* coeff, double* y, const double* Tc, const int32_t* dofmap,
                        int64_t ncells, int P, void* stream);
int fus_mass_vertex_f32(const float* x, const float* coeff, float* y, const float* Tc, const int32_t* dofmap,
                        int64_t ncells, int P, void* stream);

/* Per cell: Gc[c,:] = mean_q G[c,q,:] / wq[q], detJc[c] = mean_q detJ[c,q] / wq[q] (detJ may be
 * NULL) and affine[c] = 1 when every G[c,q,:] / wq[q] (and detJ[c,q] / wq[q]) lies within
 * tol * max|Gc[c,:]| (tol * |detJc[c]|) of that mean, else 0.  One CTA per cell. */
int fus_compress_geometry_f64(const double* G, const double* detJ, const double* wq, double* Gc,
                              double* detJc, int32_t* affine, int64_t ncells, int nq, double tol,
                              void* stream);
int fus_compress_geometry_f32(const float* G, const float* detJ, const float* wq, float* Gc,
                              float* detJc, int32_t* affine, int64_t ncells, int nq, float tol,
                              void* stream);

/* Mass (diagonal) action on cells or boundary facets
 *   y[dm[e,i]] += x[dm[e,i]] * detJ[e,i] * coeff[e]
 * Replaces `mass_operator[grid, block](x, coeff, y, detJ, dofmap)` -
 * cuda/operators.py:18-70 (numba-cpu/operators.py:19-68,
 * cpp/common/spectral_op.hpp:69-86).  ncols = Nd (cells) or n^2 (facets). */
int fus_mass_f64(const double* x, const double* coeff, double* y, const double* detJ,
                 const int32_t* dofmap, int64_t nent, int ncols, void* stream);
int fus_mass_f32(const float* x, const float* coeff, float* y, const float* detJ,
                 const int32_t* dofmap, int64_t nent, int ncols, void* stream);

/* --------------------------------------------------------------------- *
 * Vector kernels - cuda/operators.py:195-274
 * --------------------------------------------------------------------- */
int fus_axpy_f64(double alpha, const double* x, double* y, int64_t n, void* stream);
int fus_axpy_f32(float alpha, const float* x, float* y, int64_t n, void* stream);
int fus_copy_f64(const double* a, double* b, int64_t n, void* stream);
int fus_copy_f32(const float* a, float* b, int64_t n, void* stream);
int fus_fill_f64(double alpha, double* x, int64_t n, void* stream);
int fus_fill_f32(float alpha, float* x, int64_t n, void* stream);
int fus_pointwise_divide_f64(const double* a, const double* b, double* c, int64_t n, void* stream);
int fus_pointwise_divide_f32(const float* a, const float* b, float* c, int64_t n, void* stream);
int fus_square_f64(const double* a, double* b, int64_t n, void* stream);
int fus_square_f32(const float* a, float* b, int64_t n, void* stream);

/* --------------------------------------------------------------------- *
 * Halo pack / unpack - cuda/scatterer.py:18-101.  N = size_local.
 * --------------------------------------------------------------------- */
int fus_pack_fwd_f64(const double* in, double* out, const int64_t* index, int64_t n, void* stream);
int fus_pack_fwd_f32(const float* in, float* out, const int64_t* index, int64_t n, void* stream);
int fus_unpack_fwd_f64(const double* in, double* out, const int64_t* index, int64_t n, int64_t N, void* stream);
int fus_unpack_fwd_f32(const float* in, float* out, const int64_t* index, int64_t n, int64_t N, void* stream);
int fus_pack_rev_f64(const double* in, double* out, const int64_t* index, int64_t n, int64_t N, void* stream);
int fus_pack_rev_f32(const float* in, float* out, const int64_t* index, int64_t n, int64_t N, void* stream);
int fus_unpack_rev_f64(const double* in, double* out, const int64_t* index, int64_t n, void* stream);
int fus_unpack_rev_f32(const float* in, float* out, const int64_t* index, int64_t n, void* stream);
/* k vectors through one index list in one launch (the 2-3 forward scatters
 * of one RK stage, cuda/demo_linear_box.py:537-538, demo_nonlinear_bowl.py:604-606):
 *   out[i*nvec + v] = in_v[index[i] + offset]   /   out_v[index[i] + offset] (+)= in[i*nvec + v]
 * The buffer is entry-major so that a contiguous range of entries (one
 * neighbour's segment of a concatenated index list) carries all vectors:
 * ONE pack launch serves every neighbour. */
int fus_pack_multi_f64(const double* const* in, int nvec, double* out, const int64_t* index,
                       int64_t n, int64_t offset, void* stream);
int fus_pack_multi_f32(const float* const* in, int nvec, float* out, const int64_t* index,
                       int64_t n, int64_t offset, void* stream);
int fus_unpack_multi_f64(const double* in, double* const* out, int nvec, const int64_t* index,
                         int64_t n, int64_t offset, int add, void* stream);
int fus_unpack_multi_f32(const float* in, float* const* out, int nvec, const int64_t* index,
                         int64_t n, int64_t offset, int add, void* stream);

/* --------------------------------------------------------------------- *
 * Halo exchange through NVLink peer memory - the whole of
 * cuda/scatterer.py:104-277 (scatter_reverse / scatter_forward factories: per-neighbour
 * pack kernel, device synchronise, host-staged MPI Isend/Irecv + Waitall, unpack kernel)
 * behind ONE handle.  Data moves with plain loads / stores into peer-mapped memory;
 * ordering across GPUs is per-neighbour 64-bit epoch flags (st.release.sys /
 * ld.acquire.sys on a signal pad), issued by this library's own kernels: no host
 * synchronisation, no global barrier, capturable in a CUDA graph.
 *
 * The caller provides peer-addressable memory (CUDA VMM / cudaIpc mappings; the Python
 * layer uses torch's symmetric-memory allocator for the allocation and rendezvous only):
 * every exchanged vector must sit at the SAME byte offset of a symmetric arena on every
 * rank, so that its address on rank q is `local address + peer_delta[q]`.
 * --------------------------------------------------------------------- */
typedef struct fus_halo fus_halo_t;

typedef struct {
  int32_t rank, world;        /* flag slots are indexed by global rank                               */
  int32_t n_ghost_ranks;      /* neighbours holding ghost copies of dofs I own (ghosts_data[2])      */
  const int32_t* ghost_ranks; /* HOST [n_ghost_ranks]                                                */
  int32_t n_owner_ranks;      /* neighbours owning my ghosts (owners_data[2], cuda/utils.py:30-41)   */
  const int32_t* owner_ranks; /* HOST [n_owner_ranks]                                                */
  int64_t n;                  /* shared entries: ghosts_data index lists concatenated (utils.py:57-73) */
  const int64_t* idx;         /* HOST [n] local (owned) index of the entry                           */
  const int64_t* remote_pos;  /* HOST [n] index of the same dof in that neighbour's vector           */
  const int32_t* entry_seg;   /* HOST [n] position of the neighbour in ghost_ranks                   */
  int64_t size_local;         /* owned dofs: vectors are [owned | ghosts]                            */
  int64_t num_ghosts;
  void* signal_pad;           /* DEVICE my pad, fus_halo_pad_bytes(world) bytes, zeroed, peer-mapped */
  const uint64_t* peer_pad;   /* HOST [world] device address of rank q's pad as mapped HERE (0: unmapped) */
  const int64_t* peer_delta;  /* HOST [world] (rank q's arena base as mapped here) - (my arena base), bytes */
  int32_t close_group;        /* dofs per pack of the close kernel that will take the mask: 2 (f64), 4 (f32; default) */
} fus_halo_desc_t;

int64_t fus_halo_pad_bytes(int world);
/* Builds the device tables (one cudaMalloc owned by the handle, like the per-neighbour
 * buffers the reference's factories own: cuda/scatterer.py:133-138).  Host arrays of
 * `desc` are copied.  Collective only in the sense that every rank must create its own. */
int fus_halo_create(const fus_halo_desc_t* desc, fus_halo_t** out);
int fus_halo_destroy(fus_halo_t* h);
/* The owned dofs fus_rk_close_shared_* closes - those that are ghosts somewhere plus the other
 * members of their aligned groups of `close_group` (so the vectorised close kernel skips whole packs) - and
 * the bitmask over [0, size_local) marking them (bit d%8 of byte d/8), which fus_rk_close_* takes
 * as skip_mask (DEVICE pointer). */
int64_t fus_halo_num_shared(const fus_halo_t* h);
const uint8_t* fus_halo_shared_mask(const fus_halo_t* h);
/* t >= 0 when those dofs are exactly the tail [t, size_local) of the owned block (the local numbering
 * keeps the shared dofs last): fus_rk_close_* can then be given n = t and no mask.  -1 otherwise. */
int64_t fus_halo_shared_tail(const fus_halo_t* h);
/* 0, or FUS_ERR_HALO_TIMEOUT when a wait gave up (a neighbour never signalled). Synchronous. */
int fus_halo_status(fus_halo_t* h);

/* Stand-alone exchanges of up to 4 vectors (HOST array of DEVICE pointers), safe in any
 * call sequence that every rank makes identically:
 *   forward = scatter_forward(...)(buffer), cuda/scatterer.py:191-277: owner -> ghost overwrite
 *   reverse = scatter_reverse(...)(buffer), cuda/scatterer.py:104-188: ghost sums added into the
 *             owner; the ghost region keeps its values.
 * Asynchronous on `stream` (the reference synchronises the device: scatterer.py:186, 275). */
int fus_halo_forward_f64(fus_halo_t* h, double* const* vecs, int nvec, void* stream);
int fus_halo_forward_f32(fus_halo_t* h, float* const* vecs, int nvec, void* stream);
int fus_halo_reverse_f64(fus_halo_t* h, double* const* vecs, int nvec, void* stream);
int fus_halo_reverse_f32(fus_halo_t* h, float* const* vecs, int nvec, void* stream);

/* Split-phase pieces for a time-stepping loop that overlaps the exchange with compute
 * (used by the fused solvers; the ordering argument is in csrc/halo.cu):
 *   put          : owner values -> the neighbours' ghost slots, then the FWD epoch
 *   wait_forward : wait for the FWD epoch of every owner of my ghosts; then (nzero > 0) clear
 *                  the ghost part [size_local, size_local + num_ghosts) of `zero_vecs`
 *   signal_reverse : REV epoch -> every owner of my ghosts ("my partial sums are complete")
 *   get_add      : wait for the REV epoch of every ghosting neighbour, then
 *                  v[idx[e]] += peer_v[remote_pos[e]]
 *   barrier      : neighbour barrier
 * Every put must be matched by one wait_forward on the neighbours, every signal_reverse by
 * one get_add. */
int fus_halo_put_f64(fus_halo_t* h, double* const* vecs, int nvec, void* stream);
int fus_halo_put_f32(fus_halo_t* h, float* const* vecs, int nvec, void* stream);
int fus_halo_wait_forward_f64(fus_halo_t* h, double* const* zero_vecs, int nzero, void* stream);
int fus_halo_wait_forward_f32(fus_halo_t* h, float* const* zero_vecs, int nzero, void* stream);
int fus_halo_signal_reverse(fus_halo_t* h, void* stream);
/* wait (one warp) for the REV epoch of every ghosting neighbour - the first half of get_add, for
 * callers that fuse the gather into their own kernel (fus_rk_close_shared_* with gather != 0) */
int fus_halo_wait_reverse(fus_halo_t* h, void* stream);
int fus_halo_get_add_f64(fus_halo_t* h, double* const* vecs, int nvec, void* stream);
int fus_halo_get_add_f32(fus_halo_t* h, float* const* vecs, int nvec, void* stream);
int fus_halo_barrier(fus_halo_t* h, void* stream);

/* Forward halo overlapped with the interior cells INSIDE one stiffness launch.  Arms the NEXT
 * fus_stiffness* / fus_stiffness2* / fus_stiffness_westervelt* (streamed, affine or rectilinear)
 * launch issued by this host thread: cells [first_interface_cell, ncells) of that launch are the
 * ones that touch ghost dofs (the caller orders interior cells first).  Every CTA of the persistent
 * kernel works through its interior batches first and, before gathering for its first interface
 * batch, waits for the FWD epoch of every owner of this rank's ghosts (what fus_halo_wait_forward
 * would wait for); from then on it gathers x through L2.  The epoch is consumed by the
 * fus_boundary_terms_signal_* launch that follows (consume_forward != 0).  halo == NULL disarms.
 * Replaces scatter_forward(u_n), scatter_forward(v_n) -> stiffness of cuda/demo_linear_box.py:536-545
 * without a second launch for the interface cells.  Not combinable with FUS_NO_ATOMICS. */
int fus_stiffness_arm_halo_wait(const fus_halo_t* halo, int64_t first_interface_cell);

/* --------------------------------------------------------------------- *
 * Fused RK4 stage kernels.  Replace the 13 vector launches per stage of
 * cuda/demo_linear_box.py:491-563 (numba-cpu/demo_linear_box.py:425-459,
 * cpp/common/Linear.hpp:237-344).
 * --------------------------------------------------------------------- */

/* Stage opening (first stage of a step, or any stage when not chained):
 *   [first != 0: u0 = u; v0 = v]
 *   un = u0 + adt*ku ; vn = v0 + adt*kv ; ku = vn ; b = 0
 * (copy/axpy/copy/fill of :491-508, :541).  `vn` is stored in ku (f0: ku = vn). */
int fus_rk_open_f64(const double* u, const double* v, double* u0, double* v0, double* ku,
                    const double* kv, double* un, double* b, double adt, int first, int64_t n,
                    void* stream);
int fus_rk_open_f32(const float* u, const float* v, float* u0, float* v0, float* ku,
                    const float* kv, float* un, float* b, float adt, int first, int64_t n,
                    void* stream);

/* Stage closing, optionally chained with the next stage's opening:
 *   kv = b / m ; u += bdt*ku ; v += bdt*kv                       (:556-563)
 *   next_mode 1: un = u0 + adt_next*ku ; ku' = v0 + adt_next*kv ; b = 0
 *   next_mode 2: (step boundary) u0 = u ; v0 = v ; un = u ; ku' = v ; b = 0
 *   next_mode 0: nothing more
 *   next_mode 3: (first stage of a "ping-pong" step) u, v, ku are NOT read: the stage input was
 *                the base state itself (a_0 = 0: un = u0, vn = v0), so
 *                u = u0 + bdt*v0 ; v = v0 + bdt*kv ; un = u0 + adt_next*v0 ;
 *                ku' = v0 + adt_next*kv ; b = 0
 *   next_mode 4: (last stage of a ping-pong step) b = 0 and nothing else: the accumulators
 *                u, v ARE the new state; the caller swaps (u, v) with (u0, v0) between steps.
 *                A step run as 3 / 1 / 1 / 4 makes 9 + 12 + 12 + 8 vector passes instead of
 *                the 4 x 12 of 1 / 1 / 1 / 2, with the same arithmetic bit for bit.
 * kv is stored when non-NULL; it may be NULL in modes 1-4 (nothing reads
 * it again).  step_dev (may be NULL) is a device step counter incremented once per
 * call in modes 2 and 4, also when n == 0 - it indexes the source table of
 * fus_boundary_terms, so a whole RK step can be replayed as a CUDA graph with no host work.
 * skip_mask (DEVICE, may be NULL): bit d%8 of byte d/8 set => dof d is left untouched here
 * (multi-GPU: the shared dofs, closed by fus_rk_close_shared_* after the reverse halo). */
int fus_rk_close_f64(double* u, double* v, double* u0, double* v0, double* ku, double* kv,
                     double* un, double* b, const double* m, double bdt, double adt_next,
                     int next_mode, int64_t n, int64_t* step_dev, const uint8_t* skip_mask,
                     void* stream);
int fus_rk_close_f32(float* u, float* v, float* u0, float* v0, float* ku, float* kv, float* un,
                     float* b, const float* m, float bdt, float adt_next, int next_mode,
                     int64_t n, int64_t* step_dev, const uint8_t* skip_mask, void* stream);

/* Multi-GPU stage closing on the unique owned dofs that are ghosts on a neighbour - the dofs
 * fus_rk_close_* leaves out when given skip_mask = fus_halo_shared_mask(halo): their b is complete
 * only once the reverse halo has landed, so the bulk of the vector is closed while that exchange is
 * in flight and this (small, indexed) kernel runs after fus_halo_get_add.  With put_next != 0 it is
 * fused with the forward halo of the NEXT stage: the fresh stage input (un, ku; or u, v in
 * next_mode 4) is stored straight into the neighbours' ghost slots, followed by the FWD epoch
 * (= fus_halo_put of those two vectors).  With gather != 0 it is also fused with the reverse halo
 * (call fus_halo_wait_reverse first): each thread adds the neighbours' ghost partial sums of its
 * dof to b (and m, variant 1), loaded straight from their vectors, and clears them there - no
 * get_add pass, no atomics, no kernel to zero the ghost accumulators.  variant 0: fus_rk_close (m); 1: fus_rk_close_westervelt
 * (m, m0); 2: fus_rk_close_westervelt_pw (m0, m2, m5); 3: fus_leapfrog_close (m; next_mode 4, bdt =
 * dt_v, adt_next = dt_u); unused mass pointers may be NULL.
 * Replaces scatter_reverse(b) -> pointwise_divide/axpy -> (next stage) scatter_forward(un),
 * scatter_forward(vn) of cuda/demo_linear_box.py:536-563. */
int fus_rk_close_shared_f64(fus_halo_t* halo, int variant, int put_next, int gather, double* u,
                            double* v, double* u0, double* v0, double* ku, double* un, double* b,
                            double* m, const double* m0, const double* m2, const double* m5,
                            double bdt, double adt_next, int next_mode, void* stream);
int fus_rk_close_shared_f32(fus_halo_t* halo, int variant, int put_next, int gather, float* u,
                            float* v, float* u0, float* v0, float* ku, float* un, float* b, float* m,
                            const float* m0, const float* m2, const float* m5, float bdt,
                            float adt_next, int next_mode, void* stream);

/* One LEAPFROG step of the same second-order system (the north star names "RK4/leapfrog"; the
 * reference implements RK4 only - cuda/demo_linear_box.py:487-567 - so this has no reference
 * twin and is pinned to the oracle's restatement of the scheme and to its convergence order):
 *   v += dt_v * b / m ; u += dt_u * v ; b = 0        (u at whole steps, v at half steps)
 * b = K u + g src + absb v as assembled by fus_stiffness_* + fus_boundary_terms_*; with
 * m = m_lumped - (dt/2) absb the absorbing term is time-centred.  One stiffness action per step
 * instead of RK4's four; 4 reads + 3 writes per dof.  step_dev / skip_mask as for fus_rk_close_*;
 * the multi-GPU twin is fus_rk_close_shared_* with variant 3 (next_mode 4: u, v are put). */
int fus_leapfrog_close_f64(double* u, double* v, double* b, const double* m, double dt_v, double dt_u,
                           int64_t n, int64_t* step_dev, const uint8_t* skip_mask, void* stream);
int fus_leapfrog_close_f32(float* u, float* v, float* b, const float* m, float dt_v, float dt_u,
                           int64_t n, int64_t* step_dev, const uint8_t* skip_mask, void* stream);

/* Boundary-facet terms of one stage through precomputed diagonals on a compact
 * list of UNIQUE dofs: b[dof[i]] += g * src[i] + dg * src2[i] + vn[dof[i]] * absb[i].
 * Replaces the facet `mass_operator` launches of :546-551 (and
 * demo_nonlinear_bowl.py:629-639); src/src2/absb are those operators applied
 * to a vector of ones once at start-up.  Any of src, src2, absb may be NULL.
 * Source amplitudes: the scalars g, dg, or - when gtab != NULL - the device
 * table entries gtab[step*gstride + goff], gtab[step*gstride + goff + 1] with
 * step = *step_dev (0 when step_dev is NULL). */
int fus_boundary_terms_f64(double* b, const double* vn, const int32_t* dof, const double* src,
                           const double* src2, const double* absb, double g, double dg,
                           const double* gtab, const int64_t* step_dev, int gstride, int goff,
                           int64_t n, void* stream);
int fus_boundary_terms_f32(float* b, const float* vn, const int32_t* dof, const float* src,
                           const float* src2, const float* absb, float g, float dg,
                           const float* gtab, const int64_t* step_dev, int gstride, int goff,
                           int64_t n, void* stream);

/* The same, followed by fus_halo_signal_reverse(halo) from the kernel's last block: in a multi-GPU
 * stage the boundary terms are the last writes into the ghost partial sums, so the "my sums are
 * complete" epoch rides on this launch instead of needing one of its own (n may be 0).
 * consume_forward != 0: also advance the "forward epochs waited for" counter - the stage's stiffness
 * launches were armed with fus_stiffness_arm_halo_wait and have waited in-kernel. */
int fus_boundary_terms_signal_f64(fus_halo_t* halo, double* b, const double* vn, const int32_t* dof,
                                  const double* src, const double* src2, const double* absb, double g,
                                  double dg, const double* gtab, const int64_t* step_dev, int gstride,
                                  int goff, int64_t n, int consume_forward, void* stream);
int fus_boundary_terms_signal_f32(fus_halo_t* halo, float* b, const float* vn, const int32_t* dof,
                                  const float* src, const float* src2, const float* absb, float g,
                                  float dg, const float* gtab, const int64_t* step_dev, int gstride,
                                  int goff, int64_t n, int consume_forward, void* stream);

/* Multi-element (phased-array) source: the same boundary terms with one waveform per array element.
 * Over the compact list of unique dofs dof[0..n):
 *   b[dof[i]] += sum_{k = row[i]}^{row[i+1]-1} (w[k] G[elem[k]] + w2[k] DG[elem[k]]) + vn[dof[i]] absb[i]
 * with G = etab + s*8E + stage*2E, DG = G + E, s = *step_dev (0 when step_dev is NULL): the table has
 * the layout (rows, 4 stages, 2, E) - per step and RK stage the E amplitudes g_e, then the E dg_e/dt.
 * row: int32 CSR offsets, n + 1 entries (an absorbing-only dof has an empty row); elem: int32 element
 * ids in [0, E); w: the source facet mass diagonal of element elem[k] at the dof (facet coefficient
 * times detJ_f, summed over that element's facets containing the dof); w2: the same with the dg
 * coefficient (Westervelt), may be NULL; absb may be NULL.  A dof on the seam of two elements has one
 * entry per element.  One thread per dof, the sum in row order: deterministic, no atomics.
 * Rejected before any launch: n < 0, num_elements < 1, stage outside 0..3, and with n > 0 a NULL
 * b, dof, etab, row, elem or w. */
int fus_boundary_terms_elements_f64(double* b, const double* vn, const int32_t* dof, const int32_t* row,
                                    const int32_t* elem, const double* w, const double* w2,
                                    const double* absb, const double* etab, const int64_t* step_dev,
                                    int num_elements, int stage, int64_t n, void* stream);
int fus_boundary_terms_elements_f32(float* b, const float* vn, const int32_t* dof, const int32_t* row,
                                    const int32_t* elem, const float* w, const float* w2,
                                    const float* absb, const float* etab, const int64_t* step_dev,
                                    int num_elements, int stage, int64_t n, void* stream);
/* The same, followed by the "my ghost sums are complete" signal of fus_boundary_terms_signal_*
 * (n may be 0: the signalling block still runs). */
int fus_boundary_terms_elements_signal_f64(fus_halo_t* halo, double* b, const double* vn, const int32_t* dof,
                                           const int32_t* row, const int32_t* elem, const double* w,
                                           const double* w2, const double* absb, const double* etab,
                                           const int64_t* step_dev, int num_elements, int stage, int64_t n,
                                           int consume_forward, void* stream);
int fus_boundary_terms_elements_signal_f32(fus_halo_t* halo, float* b, const float* vn, const int32_t* dof,
                                           const int32_t* row, const int32_t* elem, const float* w,
                                           const float* w2, const float* absb, const float* etab,
                                           const int64_t* step_dev, int num_elements, int stage, int64_t n,
                                           int consume_forward, void* stream);

/* Westervelt stage helpers (cuda/demo_nonlinear_bowl.py:603-650):
 *   w = vn*vn                                                   (:603)
 *   fused cell-mass pair sharing one read of detJ and the dofmap:
 *     m[dm] += c2 * detJ * un[dm]       (state-dependent LHS, :610-612)
 *     b[dm] += c5 * detJ * vn[dm]^2     (:626-628)
 *   m += m0 is folded into the closing kernel below. */
int fus_westervelt_mass_f64(const double* un, const double* vn, const double* c2,
                            const double* c5, double* m, double* b, const double* detJ,
                            const int32_t* dofmap, int64_t ncells, int ncols, void* stream);
int fus_westervelt_mass_f32(const float* un, const float* vn, const float* c2, const float* c5,
                            float* m, float* b, const float* detJ, const int32_t* dofmap,
                            int64_t ncells, int ncols, void* stream);
/* kv = b / (m + m0); u += bdt*ku; v += bdt*kv; m = 0; then as fus_rk_close. */
int fus_rk_close_westervelt_f64(double* u, double* v, double* u0, double* v0, double* ku,
                                double* kv, double* un, double* b, double* m, const double* m0,
                                double bdt, double adt_next, int next_mode, int64_t n,
                                int64_t* step_dev, const uint8_t* skip_mask, void* stream);
int fus_rk_close_westervelt_f32(float* u, float* v, float* u0, float* v0, float* ku, float* kv,
                                float* un, float* b, float* m, const float* m0, float bdt,
                                float adt_next, int next_mode, int64_t n, int64_t* step_dev,
                                const uint8_t* skip_mask, void* stream);

/* Pointwise form of the Westervelt stage closing.  The lumped mass is diagonal, so the cell-mass
 * pair of cuda/demo_nonlinear_bowl.py:609-612, 626-628 needs no pass over the cells:
 *   M(c2; un) = un * m2,  M(c5; vn^2) = vn^2 * m5   with m2 = M(c2; 1), m5 = M(c5; 1) assembled once.
 *   kv = (b + vn^2 m5) / (m0 + un m2) ; u += bdt*ku ; v += bdt*kv ; then as fus_rk_close
 * (un, vn = ku: the stage input; in next_mode 3 they are u0, v0).  The stage kernel is then
 * fus_stiffness2_* (both stiffness terms, one pass over G) and only b is reverse-exchanged. */
int fus_rk_close_westervelt_pw_f64(double* u, double* v, double* u0, double* v0, double* ku,
                                   double* kv, double* un, double* b, const double* m0,
                                   const double* m2, const double* m5, double bdt,
                                   double adt_next, int next_mode, int64_t n, int64_t* step_dev,
                                   const uint8_t* skip_mask, void* stream);
int fus_rk_close_westervelt_pw_f32(float* u, float* v, float* u0, float* v0, float* ku, float* kv,
                                   float* un, float* b, const float* m0, const float* m2,
                                   const float* m5, float bdt, float adt_next, int next_mode,
                                   int64_t n, int64_t* step_dev, const uint8_t* skip_mask,
                                   void* stream);

/* --------------------------------------------------------------------- *
 * Geometry precompute on the device - cuda/precompute.py:17-163
 * (cpp/common/precompute.hpp:33-213).
 *   x_dofs (ncells, 8) int32; x_g (nv, 3); dphi (3, nq, 8); w (nq,)
 *   G (ncells, nq, 6); detJ (ncells, nq); either output may be NULL.
 * --------------------------------------------------------------------- */
int fus_geometry_f64(double* G, double* detJ, const int32_t* x_dofs, const double* x_g,
                     const double* dphi, const double* w, int64_t ncells, int nq, void* stream);
int fus_geometry_f32(float* G, float* detJ, const int32_t* x_dofs, const float* x_g,
                     const float* dphi, const float* w, int64_t ncells, int nq, void* stream);
/* boundary_data (nf, 2) int32 = (cell, local facet); dphi_f (6, 3, nq_f, 8) */
int fus_facet_geometry_f64(double* detJ_f, const int32_t* x_dofs, const double* x_g,
                           const int32_t* boundary_data, const double* dphi_f, const double* w,
                           int64_t nf, int nq_f, void* stream);
int fus_facet_geometry_f32(float* detJ_f, const int32_t* x_dofs, const float* x_g,
                           const int32_t* boundary_data, const float* dphi_f, const float* w,
                           int64_t nf, int nq_f, void* stream);

/* --------------------------------------------------------------------- *
 * Field sampling (output path)
 * --------------------------------------------------------------------- */

/* out[p] = sum_{ijk} phi[p,0,i] phi[p,1,j] phi[p,2,k] u[dofmap[cells[p], i n^2 + j n + k]],
 * phi: (npts, 3, n) 1-D Lagrange values at the points' reference coordinates.  Replaces
 * `u_n_d.copy_to_host(u_n); u_n_.eval(x_eval, cell_eval)` of
 * cuda/demo_linear_piston.py:564-570 - the whole vector no longer crosses PCIe per dump. */
int fus_eval_points_f64(const double* u, const int32_t* dofmap, const int32_t* cells,
                        const double* phi, double* out, int64_t npts, int P, void* stream);
int fus_eval_points_f32(const float* u, const int32_t* dofmap, const int32_t* cells,
                        const float* phi, float* out, int64_t npts, int P, void* stream);

/* --------------------------------------------------------------------- *
 * Host-buffer entry points (the end-to-end path: host <-> device copies are
 * inside the call).  x_host / y_host are HOST pointers (pinned for full
 * speed); every other pointer is a device pointer as above.
 * y_host += K x_host, staged through the caller-provided device scratch
 * x_dev / y_dev (nd each).  Synchronous on return.  The cells are cut into 8 ranges; the
 * upload of the x (and y) piece the next range needs, the action on the current range and the
 * download of the part of y the previous range completed run concurrently on three streams
 * (full-duplex PCIe).  With FUS_HOST_Y_ZERO (y_host holds zeros, the reference's calling
 * pattern: cuda/time_operators.py:276-279 zero-fills b before every launch) y is not uploaded.
 * --------------------------------------------------------------------- */
int fus_stiffness_host_f64(const double* x_host, double* y_host, int64_t nd, double* x_dev,
                           double* y_dev, const double* coeff, const double* G,
                           const int32_t* dofmap, const double* dphi, int64_t ncells, int P,
                           int flags, void* stream);
int fus_stiffness_host_f32(const float* x_host, float* y_host, int64_t nd, float* x_dev,
                           float* y_dev, const float* coeff, const float* G,
                           const int32_t* dofmap, const float* dphi, int64_t ncells, int P,
                           int flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FUS_B200_H */
