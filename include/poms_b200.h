/*
 * poms_b200.h -- C ABI of libpoms_b200.so: hand-written sm_100a fp64 kernels for the POMS
 * multigrid solve path (tensor-product B-spline discretisations).
 *
 * The reference (pyccel/poms) is pure Python and has no FFI; its hot-path "interface" is a
 * set of Python functions over `spl` stencil objects.  Each entry point below replaces the
 * arithmetic of one of them; the Python package poms_b200/ keeps the reference names and
 * signatures and binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer (tensor.data_ptr()); no torch types cross this ABI;
 *  - vectors are fp64, C order, axis 1 slowest (sources/mg_jac.py:106-108).  A d-dim vector
 *    is described by its owned extent (n1[,n2],n3), the row pitch `ld` and the plane pitch
 *    `pld` in doubles, and `glo`/`ghi` = number of readable ghost planes stored directly
 *    below / above the owned planes along axis 1 (slab partition; 0 on one GPU);
 *  - a 1-D banded matrix is an (n, 2p+1) row-major array, band[i][k] = A[i, i+k-p]
 *    (pyccel/pyccel_functions.py:15,19); out-of-matrix entries must be zero;
 *  - all launches go to the caller's `stream` (cudaStream_t cast to void*); nothing
 *    allocates or synchronises; `ws` is a caller-owned workspace of poms_workspace_bytes()
 *    bytes, zero-initialised once, private to one stream;
 *  - return value: 0 ok, <0 = -(index of the bad argument), >0 = cudaError_t.
 */
#ifndef POMS_B200_H
#define POMS_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int poms_version(void);
int64_t poms_workspace_bytes(void);
const char* poms_last_error(void);
/* number of kernel launches issued through this library since load (bench "gpu_launches") */
int64_t poms_launch_count(void);
/* kernels replayed from a captured CUDA graph are not seen by the library: the caller adds them */
void poms_launch_count_add(int64_t n);

/* operator forms for poms_kron_matvec_* */
#define POMS_FORM_SINGLE 0 /* Y = (A1 (x) A2 [(x) A3]) X; the A's are passed in the m* slots   */
#define POMS_FORM_SUM    1 /* Y = sum_a (M (x)..(x) K_a (x)..(x) M) X, separable elliptic form */
/* epilogues: v = (A x)[i] */
#define POMS_EPI_STORE  0  /* y = v                      ; dot += x*v   (p.q of CG)          */
#define POMS_EPI_RESID  1  /* y = b - v                  ; dot += y*y   (r.r)                */
#define POMS_EPI_JACOBI 2  /* y = x + om*(b - v)/diag(A) ; dot += dr*dr (damped Jacobi sweep) */
#define POMS_EPI_DINV   3  /* y = om*(b - v)/diag(A)     ; dot += y*y   (Jacobi-preconditioned residual) */
#define POMS_EPI_AXPY   4  /* y = b + om*v (b NULL: om*v) ; dot += (om*v)^2 (EXTENSION: smoother update) */

/*
 * Kronecker-structured banded mat-vec, one fused pass (16 B/DOF algorithmic).
 * Replaces: kron_dot_v2 / kron_dot_v1 (sources/kron_product.py:56-89, 10-52),
 *           kron_dot_pyccel_2d (pyccel/pyccel_functions.py:4-21),
 *           StencilMatrix.dot as used by the solvers (sources/solvers.py:85,103,209,256,274),
 *           and, with POMS_EPI_JACOBI, the sweep of damped_jacobi (sources/solvers.py:209-219).
 * All bands have the same half-bandwidth p (narrower ones are zero-padded by the caller).
 * FORM_SINGLE: m1,m2[,m3] are the factors, k* ignored.  FORM_SUM: k of the LAST axis must
 * already contain K+M (the "+u" term of sources/matrix_assembler.py:82-83).
 * dot_out (may be NULL = no reduction): the fused reduction OVERWRITES *dot_out.
 */
int poms_kron_matvec_2d(const double* x, double* y, const double* b,
                        int n1, int n2, int64_t ld, int glo, int ghi, int p, int form,
                        const double* m1, const double* k1, const double* m2, const double* k2,
                        int epilogue, double omega, double* dot_out, void* ws, void* stream);
int poms_kron_matvec_3d(const double* x, double* y, const double* b,
                        int n1, int n2, int n3, int64_t ld, int64_t pld, int glo, int ghi,
                        int p, int form,
                        const double* m1, const double* k1, const double* m2, const double* k2,
                        const double* m3, const double* k3,
                        int epilogue, double omega, double* dot_out, void* ws, void* stream);

/* poms_kron_matvec_2d plus HOST-side hints for the TMA kernel: toep_host[axis(0,1)][m,k][2p+1] = the
 * interior (Toeplitz) band rows, toep_rng_host = {lo1, hi1, lo2, hi2} (rows [lo, hi) equal them bit for
 * bit); NULL = no hint (every coefficient from global memory).  poms_set_matvec2d_variant(0) selects the
 * round-1 kernel (A/B timing, tests); initial value from POMS_B200_MV2_VARIANT. */
int poms_kron_matvec_2d_ex(const double* x, double* y, const double* b,
                           int n1, int n2, int64_t ld, int glo, int ghi, int p, int form,
                           const double* m1, const double* k1, const double* m2, const double* k2,
                           int epilogue, double omega, double* dot_out, void* ws, void* stream,
                           const double* toep_host, const int* toep_rng_host);
void poms_set_matvec2d_variant(int variant);

/*
 * Same as poms_kron_matvec_3d plus HOST-side hints that unlock the constant-bank coefficient path
 * of the TMA kernel: toep_host[axis(0,1,2)][m,k][2p+1] = the interior (Toeplitz) band row of the
 * matrices of each axis, toep_rng_host = {lo1, hi1, lo2, hi2, lo3, hi3}: rows [lo, hi) of that axis equal
 * it bit for bit (uniform knots: all rows but the first / last 2p).  NULL = no hint.
 * The TMA path is taken when x is 16-byte aligned and ld, pld are even; otherwise the generic
 * kernel runs.  poms_set_force_generic(1) forces the generic kernel (tests / A-B timing).
 */
int poms_kron_matvec_3d_ex(const double* x, double* y, const double* b,
                           int n1, int n2, int n3, int64_t ld, int64_t pld, int glo, int ghi,
                           int p, int form,
                           const double* m1, const double* k1, const double* m2, const double* k2,
                           const double* m3, const double* k3,
                           int epilogue, double omega, double* dot_out, void* ws, void* stream,
                           const double* toep_host, const int* toep_rng_host);
/* poms_kron_matvec_3d_ex with a fused dot product against a THIRD vector: with POMS_EPI_AXPY and
 * dot_with != NULL the reduction written to *dot_out is sum y[i] * dot_with[i] (y = the epilogue's
 * output) instead of sum (om*v)^2 -- the s.r of the CG drivers (sources/solvers.py:117-118) computed by the
 * last smoother pass.  dot_with has the layout of x (same ghost planes).  *fused_host = 1 when the TMA
 * kernel did it, 0 when the launch fell back to a kernel without this epilogue (*dot_out then holds the
 * standard reduction and the caller computes the dot product itself). */
int poms_kron_matvec_3d_dotv(const double* x, double* y, const double* b,
                             int n1, int n2, int n3, int64_t ld, int64_t pld, int glo, int ghi,
                             int p, int form,
                             const double* m1, const double* k1, const double* m2, const double* k2,
                             const double* m3, const double* k3,
                             int epilogue, double omega, double* dot_out, void* ws, void* stream,
                             const double* toep_host, const int* toep_rng_host,
                             const double* dot_with, int* fused_host);
void poms_set_force_generic(int flag);
/* A/B timing only: fix the axis-1 chunk (planes per CTA) of the 3-D mat-vec; 0 = automatic. */
void poms_set_matvec3d_chunk(int chunk);
/* Kernel variant of the TMA path: 1 = split-barrier kernel with TMA epilogue tiles and shared pair sums
 * (default), 0 = round-1 kernel (one CTA barrier per plane); initial value from the environment variable
 * POMS_B200_MV3_VARIANT.  A/B timing and tests. */
void poms_set_matvec3d_variant(int variant);

/*
 * Full (non-separable) 2-D stencil mat-vec: y[i1,i2] = sum_{k1,k2} S[i1,i2,k1,k2] x[i1+k1-p1,i2+k2-p2]
 * = spl StencilMatrix.dot (slides/content.tex:285-290; sources/solvers.py:85).  S is
 * (n1, n2, 2p1+1, 2p2+1) row-major.  Same epilogues; diag = S[i1,i2,p1,p2].
 */
int poms_stencil_matvec_2d(const double* x, double* y, const double* b, const double* S,
                           int n1, int n2, int64_t ld, int glo, int ghi, int p1, int p2,
                           int epilogue, double omega, double* dot_out, void* ws, void* stream);

/* The same in 3-D: S is (n1, n2, n3, 2p1+1, 2p2+1, 2p3+1) row-major ((2p+1)^3 coefficients per row: the
 * kernel streams coefficients, one warp per output point).  EXTENSION to 3-D of the operator type the
 * reference's solvers take (sources/solvers.py:85,103,209). */
int poms_stencil_matvec_3d(const double* x, double* y, const double* b, const double* S,
                           int n1, int n2, int n3, int64_t ld, int64_t pld, int glo, int ghi,
                           int p1, int p2, int p3, int epilogue, double omega, double* dot_out,
                           void* ws, void* stream);
/* x[i] += d[i] on the points with (i1 + i2 + i3 + off) % 2 == colour (n1 = 1 for 2-D arrays): the half
 * sweep of a two-colour (red-black) damped Jacobi smoother, named as future work in the reference's talk
 * (slides/content.tex:393).  EXTENSION. */
int poms_color_add(double* x, const double* d, int n1, int n2, int n3, int64_t ld, int64_t pld,
                   int off, int colour, void* stream);

/*
 * BLAS-1 pieces of the CG drivers over a flat range of `n` doubles (the owned planes are
 * contiguous because axis 1 is slowest).  Scalars live on the device: alpha = *num / *den.
 */
/* x += a p ; r -= a q ; *rr = r.r      (sources/solvers.py:104-111; 48 B/DOF)            */
int poms_cg_update(double* x, double* r, const double* p, const double* q, int64_t n,
                   const double* num, const double* den, double* rr_out, void* ws, void* stream);
/* p = s + (num/den) p                  (sources/solvers.py:120-124)                         */
int poms_p_update(double* p, const double* s, int64_t n, const double* num, const double* den,
                  void* stream);
/* *out = x.y                           (StencilVector.dot, local part)                      */
int poms_dot(const double* x, const double* y, int64_t n, double* out, void* ws, void* stream);
/* z = a x + b y  (y may be NULL -> z = a x); a, b host scalars                              */
int poms_axpby(double* z, double a, const double* x, double b, const double* y, int64_t n,
               void* stream);
/* y += (num/den) * x with device scalars (crl: sources/solvers.py:44-54)                    */
int poms_axpy_dev(double* y, const double* x, int64_t n, const double* num, const double* den,
                  double sign, void* stream);
/* x = om * b / diag(A) and *dot = x.x : first damped-Jacobi sweep from x0 = 0, and jacobi()
 * with om = 1 (sources/solvers.py:139-163, 209-219).  diag from the Kronecker-sum bands. */
int poms_jacobi_first_2d(double* x, const double* b, int n1, int n2, int64_t ld, int p, int form,
                         const double* m1, const double* k1, const double* m2, const double* k2,
                         double omega, double* dot_out, void* ws, void* stream);
int poms_jacobi_first_3d(double* x, const double* b, int n1, int n2, int n3, int64_t ld,
                         int64_t pld, int p, int form,
                         const double* m1, const double* k1, const double* m2, const double* k2,
                         const double* m3, const double* k3,
                         double omega, double* dot_out, void* ws, void* stream);
/* d = c1*d + c2*z ; x += d : one step of the Chebyshev smoother recurrence (40 B/DOF).
 * EXTENSION (not in the reference): linear, symmetric form of the reference's PCG smoothers */
int poms_cheb_update(double* x, double* d, const double* z, double c1, double c2, int64_t n,
                     void* stream);
/* x = om * b / d (d = explicit diagonal array, same layout), *dot = x.x                     */
int poms_diag_scale(double* x, const double* b, const double* d, int64_t n, double omega,
                    double* dot_out, void* ws, void* stream);

/*
 * Banded triangular solves of dgbtrs along one axis of a 2-D/3-D array, all lines at once.
 * Replaces the per-line dgbtrs of kron_solve_bnd_par (sources/kron_product.py:226,232) and
 * kron_solve_par_bnd_pyccel_{2d,3d} (pyccel/pyccel_functions.py:160,166,229-244).
 * `ab` is the dgbtrf output in LAPACK band storage as a row-major (2kl+ku+1, n) array,
 * `ipiv` the 0-based pivots (int32); ipiv == NULL states that dgbtrf made no row interchange
 * (ipiv[j] == j: SPD / diagonally dominant bands such as mass and GLT matrices) and selects the
 * streaming kernels: one thread per line for a strided axis, warp-tiled shared-memory transposition
 * for the contiguous axis.  The array is viewed as (n_outer, n, n_inner) with strides
 * (s_outer, s_axis, 1); y -> x (may alias).
 */
int poms_band_solve_axis(const double* y, double* x, const double* ab, const int32_t* ipiv,
                         int n, int kl, int ku, int64_t n_outer, int64_t s_outer, int64_t s_axis,
                         int64_t n_inner, void* stream);

/*
 * No-pivot banded solve for FEW lines (2-D grids: only n lines of length n exist, far too few
 * for 148 SMs): every line is cut into chunks of `chunk` entries that start `warm_*` entries early
 * from a zero state.  Valid when the homogeneous solutions of the two triangular recurrences decay
 * below rounding within the warm-up (diagonally dominant SPD bands: mass, GLT); the caller checks
 * that on the host for the given factor.  y -> work (forward), work -> x (backward); work must not
 * alias y or x.
 */
int poms_band_solve_axis_chunked(const double* y, double* x, double* work, const double* ab, int n,
                                 int kl, int ku, int64_t n_outer, int64_t s_outer, int64_t s_axis,
                                 int64_t n_inner, int chunk, int warm_fwd, int warm_bwd,
                                 void* stream);

/*
 * No-pivot banded solve along the CONTIGUOUS axis with a fused epilogue:
 *   out = [add +] scale * T^-1 y      (work receives the forward-substitution intermediate)
 * EXTENSION used by the multi-level smoother: the Chebyshev / Richardson update
 * x += (1/theta) B^-1 r is folded into the last line solve of the Kronecker solve, so the
 * correction is never written to and re-read from HBM.  n_lines lines, s_line doubles apart.
 */
int poms_band_solve_axis_fused(const double* y, double* work, const double* ab, int n, int kl,
                               int ku, int64_t n_lines, int64_t s_line, double scale,
                               const double* add, double* out, void* stream);

/*
 * Per-axis sparse row-gather: out[o, i, c] (+)= sum_{w<W} coef[i*W+w] * in[o, start[i]+w, c].
 * With the rows of P1 it is the prolongation, with the rows of P1^T the restriction of
 * sources/mg_jac.py:67-70,94,102 applied one axis at a time (knot-insertion transfer).
 * accumulate != 0 adds into out (prolong + correct, sources/mg_jac.py:112).
 */
int poms_axis_gather(const double* in, double* out, const int32_t* start, const double* coef,
                     int W, int n_in, int n_out, int64_t n_outer, int64_t so_in, int64_t sa_in,
                     int64_t so_out, int64_t sa_out, int64_t n_inner, int accumulate,
                     void* stream);

/*
 * Fused 3-D transfers (EXTENSION of the per-axis gathers above: same rows, one pass).
 *   poms_restrict_3d: coarse = (R1 (x) R2 (x) R3) fine     -- R.dot of sources/mg_jac.py:94
 *   poms_prolong_3d:  fine (+)= (P1 (x) P2 (x) P3) coarse  -- P.dot + correction, mg_jac.py:102,112
 * sN, cN: device rows (start, coef) of axis N in the poms_axis_gather format, WN taps per row
 * (<= 8); sN_host: host copies of the starts, checked against the kernels' static tile bounds (a
 * negative status means the caller must use poms_axis_gather).  ld / pld: row and plane pitches.
 */
int poms_restrict_3d(const double* fine, double* coarse, int n1f, int n2f, int n3f, int64_t ldf,
                     int64_t pldf, int n1c, int n2c, int n3c, int64_t ldc, int64_t pldc,
                     const int32_t* s1, const double* c1, int W1, const int32_t* s2,
                     const double* c2, int W2, const int32_t* s3, const double* c3, int W3,
                     const int32_t* s1_host, const int32_t* s2_host, const int32_t* s3_host,
                     void* stream);
int poms_prolong_3d(const double* coarse, double* fine, int n1f, int n2f, int n3f, int64_t ldf,
                    int64_t pldf, int n1c, int n2c, int n3c, int64_t ldc, int64_t pldc,
                    const int32_t* s1, const double* c1, int W1, const int32_t* s2,
                    const double* c2, int W2, const int32_t* s3, const double* c3, int W3,
                    const int32_t* s2_host, const int32_t* s3_host, int accumulate, void* stream);

/*
 * Round-2 one-pass transfers for the big levels (poms_transfer3d_v2.cu): same arguments, rows and
 * results as poms_restrict_3d / poms_prolong_3d, but ONE row width on all three axes (restriction
 * 3..7, prolongation 2..6).  The in-plane passes run once per COARSE plane and the axis-1 pass lives
 * in registers, so that 9 (restriction) / 17 (prolongation + correction, mg_jac.py:112) bytes per
 * fine point move through HBM instead of the 21 / 29 of three per-axis gathers.  A negative status
 * means "rows do not fit": fall back to poms_restrict_3d / poms_prolong_3d / poms_axis_gather.
 */
int poms_restrict_3d_v2(const double* fine, double* coarse, int n1f, int n2f, int n3f, int64_t ldf,
                        int64_t pldf, int n1c, int n2c, int n3c, int64_t ldc, int64_t pldc,
                        const int32_t* s1, const double* c1, int W1, const int32_t* s2,
                        const double* c2, int W2, const int32_t* s3, const double* c3, int W3,
                        const int32_t* s1_host, const int32_t* s2_host, const int32_t* s3_host,
                        void* stream);
int poms_prolong_3d_v2(const double* coarse, double* fine, int n1f, int n2f, int n3f, int64_t ldf,
                       int64_t pldf, int n1c, int n2c, int n3c, int64_t ldc, int64_t pldc,
                       const int32_t* s1, const double* c1, int W1, const int32_t* s2,
                       const double* c2, int W2, const int32_t* s3, const double* c3, int W3,
                       const int32_t* s2_host, const int32_t* s3_host, int accumulate, void* stream);

/* y = Ainv x, dense row-major n x n (replicated coarse direct solve, sources/mg_jac.py:98-99) */
int poms_dense_matvec(const double* Ainv, const double* x, double* y, int n, void* stream);

/*
 * Device-side 1-D setup (EXTENSION, SURVEY section 8f-2): the O(n p^2) pieces the reference computes in
 * Python on the host.  All pointers are device pointers.
 *  poms_assemble_1d: mass M and stiffness K bands (n, 2p+1) on the knot vector `knots` (n + p + 1
 *    entries) by Gauss-Legendre quadrature with the p+1 nodes / weights gauss_x, gauss_w on [-1, 1]
 *    (assembly_1d, sources/matrix_assembler.py:10-77; it computes K and returns only M, Appendix B).
 *  poms_knot_insertion_rows: rows of the knot-insertion matrix P1 (n_f x n_c) between the nested knot
 *    vectors Tc, Tf by the Oslo recursion: P1[i, start[i] + w] = coef[i*(p+1) + w]
 *    (matrix_multi_stages, sources/mg_jac.py:67).
 *  poms_band_lu_nopiv: LU without row interchanges of an (n, 2q+1) band into dgbtrf storage, row-major
 *    (3q+1, n) with kl = ku = q (the factor kron_solve_bnd_par takes, sources/kron_product.py:191-197);
 *    *info_dev = 0, or j+1 when column j has a zero pivot.
 */
int poms_assemble_1d(const double* knots, int n, int p, const double* gauss_x, const double* gauss_w,
                     double* M, double* K, void* stream);
int poms_knot_insertion_rows(const double* Tc, int nc, const double* Tf, int nf, int p,
                             int32_t* start, double* coef, void* stream);
int poms_band_lu_nopiv(const double* band, int n, int q, double* ab, int* info_dev, void* stream);

/*
 * Dense per-axis contraction out[o,i,c] = sum_j Q[i,j] in[o,j,c] on the fp64 tensor cores (DMMA):
 * the 1-D eigenbasis contractions of the fast-diagonalisation coarse solve that replaces
 * splu(csc_matrix(Ac)).solve(rc) (sources/mg_jac.py:98-99; dense Kronecker solve of
 * sources/kron_product.py:93-117).  Same array view as poms_axis_gather; Q is n_out x n_in row-major.
 */
int poms_axis_dense_dmma(const double* in, double* out, const double* Q, int n_in, int n_out,
                         int64_t n_outer, int64_t so_in, int64_t sa_in, int64_t so_out,
                         int64_t sa_out, int64_t n_inner, void* stream);

/*
 * Peer-memory halo exchange (one process per GPU, one box): replaces the MPI ghost update of spl's
 * `update_ghost_regions` (sources/kron_product.py:76,87; sources/solvers.py:162,215) without NCCL.
 * poms_ipc_*: thin wrappers of cudaMalloc / cudaIpc{Get,Open,Close}MemHandle so that the Python
 * host side can map the vector arenas and flag words of the two slab neighbours (handles travel
 * over torch.distributed); `handle` buffers hold poms_ipc_handle_bytes() bytes.
 * poms_halo_exchange_p2p: ONE kernel that pushes `n_doubles` doubles (the outermost owned planes,
 * contiguous because axis 1 is slowest) from src_lo / src_hi into the neighbours' ghost planes
 * dst_lo / dst_hi (peer pointers) and handshakes through the flag words (poms_halo_flags_bytes()
 * zero-initialised bytes per rank; lo_flags / hi_flags = the neighbours' words, NULL = no
 * neighbour on that side).  Collective over the neighbours: every rank must launch the same
 * sequence of exchanges.  Graph-capturable (the sequence number lives on the device).
 */
int poms_ipc_alloc(int64_t bytes, void** ptr_out);
int poms_ipc_free(void* ptr);
int poms_ipc_handle_bytes(void);
int poms_ipc_get_handle(void* ptr, void* handle_out);
int poms_ipc_open(const void* handle, void** ptr_out);
int poms_ipc_close(void* ptr);
int poms_halo_flags_bytes(void);
int poms_halo_exchange_p2p(const double* src_lo, double* dst_lo, const double* src_hi, double* dst_hi,
                           int64_t n_doubles, void* my_flags, void* lo_flags, void* hi_flags,
                           void* stream);

/*
 * Finite-element quadrature on tensor-product B-spline spaces (poms_fem3d.cu; poms_b200/fem.py builds the
 * tables).  Both entry points march along axis 1 over one chunk of element planes; a 2-D space is passed
 * with a middle axis of one coefficient and one quadrature point.
 *  poms_quad_to_coef_3d: y (+)= (B1^T (x) B2^T (x) B3^T) F, F = (e1_hi - e1_lo) * q1n quadrature planes of
 *    shape (m2, m3) with pitches fld / fpld.  Axis 1: element e touches rows s1[e] .. s1[e]+k1n-1 with the
 *    weighted values b1[(e * k1n + k) * q1n + q]; rows below `store_from` are added to y, the others
 *    stored.  Axis 2: row r = sum_t c2[r * w2 + t] * (quadrature row st2[r] + t).  Axis 3: row r =
 *    sum_{m, q} c3[r * (p+1)^2 + m (p+1) + q] * F[(e3[r] + m)(p+1) + q], ne3 elements.  The *_host
 *    arrays are host copies of s1, st2, e3 (checks and tile sizes).  Deterministic, no atomics.
 *  poms_quad_error_3d: out[0] (+)= sum w (ref[0] - u_h)^2, and with grad out[1] (+)= sum w |ref[1..3] -
 *    grad u_h|^2 (a null gradient component is skipped) over quadrature planes j1_lo .. j1_lo+nq1-1 of
 *    m1; ref[c] has row / plane pitches rld[c] / rpld[c] (host arrays of 4).  Per quadrature point j of
 *    axis a: first coefficient s_a[j], k_a values v_a[j * k_a + i] and derivatives d_a, weight w_a[j];
 *    k3 = p+1.  ws: the library workspace (deterministic grid reduction).
 */
int poms_quad_to_coef_3d(const double* F, int64_t fld, int64_t fpld, double* y, int64_t ld, int64_t pld,
                         int n1, int n2, int n3, int m2, int m3, int p, int e1_lo, int e1_hi, int k1n,
                         int q1n, const int32_t* s1, const double* b1, int store_from, const int32_t* st2,
                         const double* c2, int w2, const int32_t* e3, const double* c3, int ne3,
                         const int32_t* s1_host, const int32_t* st2_host, const int32_t* e3_host,
                         void* stream);
int poms_quad_error_3d(const double* x, int64_t ld, int64_t pld, int n1, int n2, int n3, int m2, int m3, int p,
                       const double* const* ref, const int64_t* rld, const int64_t* rpld, int j1_lo, int nq1,
                       int k1n, const int32_t* s1, const double* v1, const double* d1, const double* w1,
                       int k2n, const int32_t* s2, const double* v2, const double* d2, const double* w2,
                       const int32_t* s3, const double* v3, const double* d3, const double* w3,
                       const int32_t* s1_host, const int32_t* s2_host, const int32_t* s3_host, int m1,
                       int grad, int accumulate, double* out, void* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif
