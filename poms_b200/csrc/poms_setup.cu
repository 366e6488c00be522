// poms_setup.cu -- device-side 1-D SETUP of the multigrid hierarchy (SURVEY.md section 8f-2):
//   * poms_assemble_1d        1-D mass / stiffness bands by Gauss-Legendre quadrature
//                             (/root/reference/sources/matrix_assembler.py:10-77, assembly_1d)
//   * poms_assemble_1d_advection  1-D advection band G[i, k] = int B_{i+k-p}' B_i (convection term)
//   * poms_knot_insertion_rows  rows of the knot-insertion (prolongation) matrix P1 by the Oslo
//                             recursion (matrix_multi_stages, /root/reference/sources/mg_jac.py:67)
//   * poms_band_lu_nopiv      banded LU without row interchanges in dgbtrf storage (the factor
//                             kron_solve_bnd_par takes, /root/reference/sources/kron_product.py:191-197)
// All of it is O(n p^2) work on arrays of a few thousand entries: the kernels are written for
// latency (one small grid each), not for bandwidth.  The dense generalised eigenproblems of the
// coarse solve / smoother bounds use torch.linalg on the device (setup-time library calls).
#include <string.h>
#define POMS_TU 99
#include "poms_kernels.cu"

#define POMS_MAXP 5

// p+1 non-zero B-splines of degree p and of degree p-1 at x in knot span `span` (de Boor triangle;
// The NURBS Book A2.2).  N[r] = B_{span-p+r, p}(x); Nm[r] = B_{span-p+1+r, p-1}(x), r < p.
__device__ __forceinline__ void basis_funs(const double* __restrict__ T, int p, int span, double x,
                                           double (&N)[POMS_MAXP + 1], double (&Nm)[POMS_MAXP + 1]) {
    double left[POMS_MAXP + 1], right[POMS_MAXP + 1];
    N[0] = 1.0;
#pragma unroll
    for (int r = 0; r <= POMS_MAXP; ++r) Nm[r] = 0.0;
    if (p == 1) Nm[0] = 1.0;
    for (int d = 1; d <= p; ++d) {
        left[d] = x - T[span + 1 - d];
        right[d] = T[span + d] - x;
        if (d == p)
            for (int r = 0; r < p; ++r) Nm[r] = N[r];     // degree p-1 values
        double saved = 0.0;
        for (int r = 0; r < d; ++r) {
            const double den = right[r + 1] + left[d - r];
            const double tmp = N[r] / den;
            N[r] = saved + right[r + 1] * tmp;
            saved = left[d - r] * tmp;
        }
        N[d] = saved;
    }
}

// one thread per band entry (i, k), j = i+k-p: M[i, k] = int B_i B_j, K[i, k] = int B_i' B_j',
// G[i, k] = int B_i B_j' (advection).  One quadrature loop serves both entry points; an output whose
// pointer is null is neither computed into memory nor written.
__global__ void __launch_bounds__(128) assemble_1d_kernel(const double* __restrict__ T, int n, int p,
                                                          const double* __restrict__ gx, const double* __restrict__ gw,
                                                          double* __restrict__ M, double* __restrict__ K,
                                                          double* __restrict__ G) {
    const int W = 2 * p + 1;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * W) return;
    const int i = t / W, kk = t - i * W;
    const int j = i + kk - p;
    double m = 0.0, s = 0.0, g = 0.0;
    if (j >= 0 && j < n) {
        const int e_lo = max(max(i, j), p), e_hi = min(min(i, j) + p, n - 1);
        for (int e = e_lo; e <= e_hi; ++e) {
            const double a = T[e], b = T[e + 1];
            if (!(b > a)) continue;
            const int il = i - (e - p), jl = j - (e - p);
            for (int q = 0; q <= p; ++q) {
                const double x = 0.5 * (a + b) + 0.5 * (b - a) * gx[q];
                const double w = 0.5 * (b - a) * gw[q];
                double N[POMS_MAXP + 1], Nm[POMS_MAXP + 1];
                basis_funs(T, p, e, x, N, Nm);
                // derivative of local function r (global g = e-p+r):
                //   p * ( B_{g,p-1} / (T[g+p]-T[g]) - B_{g+1,p-1} / (T[g+p+1]-T[g+1]) ),  B_{g,p-1} = Nm[r-1]
                auto der = [&](int r) {
                    const int g = e - p + r;
                    double d = 0.0;
                    if (r >= 1) d += p * Nm[r - 1] / (T[g + p] - T[g]);
                    if (r <= p - 1) d -= p * Nm[r] / (T[g + p + 1] - T[g + 1]);
                    return d;
                };
                const double djl = der(jl);
                m = fma(w * N[il], N[jl], m);
                s = fma(w * der(il), djl, s);
                g = fma(w * N[il], djl, g);
            }
        }
    }
    if (M) M[t] = m;
    if (K) K[t] = s;
    if (G) G[t] = g;
}

static int launch_assemble_1d(const double* knots, int n, int p, const double* gauss_x, const double* gauss_w,
                              double* M, double* K, double* G, void* stream) {
    if (!knots || !gauss_x || !gauss_w) return bad_arg(1, "null pointer");
    if (p < 1 || p > POMS_MAXP) return bad_arg(3, "p must be 1..5");
    if (n < p + 1) return bad_arg(2, "n");
    const int total = n * (2 * p + 1);
    assemble_1d_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(knots, n, p, gauss_x, gauss_w, M, K, G);
    return 0;
}

extern "C" int poms_assemble_1d(const double* knots, int n, int p, const double* gauss_x, const double* gauss_w,
                                double* M, double* K, void* stream) {
    if (!M || !K) return bad_arg(1, "null pointer");
    const int rc = launch_assemble_1d(knots, n, p, gauss_x, gauss_w, M, K, nullptr, stream);
    if (rc) return rc;
    CHECK_LAUNCH("poms_assemble_1d");
    return 0;
}

extern "C" int poms_assemble_1d_advection(const double* knots, int n, int p, const double* gauss_x,
                                          const double* gauss_w, double* G, void* stream) {
    if (!G) return bad_arg(1, "null pointer");
    const int rc = launch_assemble_1d(knots, n, p, gauss_x, gauss_w, nullptr, nullptr, G, stream);
    if (rc) return rc;
    CHECK_LAUNCH("poms_assemble_1d_advection");
    return 0;
}

// one thread per fine row i: P1[i, start[i] + w] = coef[i, w], w = 0..p  (Oslo algorithm 1)
__global__ void __launch_bounds__(128) knot_insertion_rows_kernel(const double* __restrict__ Tc, int nc,
                                                                  const double* __restrict__ Tf, int nf, int p,
                                                                  int32_t* __restrict__ start,
                                                                  double* __restrict__ coef) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nf) return;
    // coarse span mu: Tc[mu] <= Tf[i] < Tc[mu+1]  (searchsorted right - 1), clamped to [p, nc-1]
    const double tf = Tf[i];
    int lo = 0, hi = nc + p + 1;            // first index with Tc[idx] > tf
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (Tc[mid] <= tf) lo = mid + 1; else hi = mid;
    }
    int mu = lo - 1;
    mu = min(max(mu, p), nc - 1);
    double alpha[POMS_MAXP + 1], nw[POMS_MAXP + 1];
    alpha[0] = 1.0;
    for (int w = 1; w <= POMS_MAXP; ++w) alpha[w] = 0.0;
    for (int k = 1; k <= p; ++k) {
        const double tau = Tf[i + k];
        for (int w = 0; w <= k; ++w) {
            const int j = mu - k + w;
            double acc = 0.0;
            if (w >= 1) {
                const double den = Tc[j + k] - Tc[j];
                if (den > 0.0) acc += (tau - Tc[j]) / den * alpha[w - 1];
            }
            if (w <= k - 1) {
                const double den = Tc[j + k + 1] - Tc[j + 1];
                if (den > 0.0) acc += (Tc[j + k + 1] - tau) / den * alpha[w];
            }
            nw[w] = acc;
        }
        for (int w = 0; w <= k; ++w) alpha[w] = nw[w];
    }
    start[i] = mu - p;
    for (int w = 0; w <= p; ++w) coef[(int64_t)i * (p + 1) + w] = alpha[w];
}

extern "C" int poms_knot_insertion_rows(const double* Tc, int nc, const double* Tf, int nf, int p, int32_t* start,
                                        double* coef, void* stream) {
    if (!Tc || !Tf || !start || !coef) return bad_arg(1, "null pointer");
    if (p < 1 || p > POMS_MAXP) return bad_arg(5, "p must be 1..5");
    if (nc < p + 1 || nf < nc) return bad_arg(2, "nc / nf");
    knot_insertion_rows_kernel<<<(nf + 127) / 128, 128, 0, (cudaStream_t)stream>>>(Tc, nc, Tf, nf, p, start, coef);
    CHECK_LAUNCH("poms_knot_insertion_rows");
    return 0;
}

// Banded LU without row interchanges, one CTA: the band (n, 2q+1) is copied into dgbtrf storage
// AB[kl+ku+i-j, j] = A[i, j] (row-major (2kl+ku+1, n), kl = ku = q), then column by column the
// q multipliers are formed and the q x q trailing block is updated by the threads of the CTA.
__global__ void __launch_bounds__(128) band_lu_nopiv_kernel(const double* __restrict__ band, int n, int q,
                                                            double* __restrict__ ab, int* __restrict__ info) {
    const int W = 2 * q + 1, R = 3 * q + 1, kd = 2 * q;
    for (int64_t t = threadIdx.x; t < (int64_t)R * n; t += blockDim.x) ab[t] = 0.0;
    __syncthreads();
    for (int64_t t = threadIdx.x; t < (int64_t)n * W; t += blockDim.x) {
        const int i = (int)(t / W), k = (int)(t - (int64_t)i * W) - q;     // A[i, i+k]
        const int j = i + k;
        if (j >= 0 && j < n) ab[(int64_t)(kd - k) * n + j] = band[t];
    }
    __syncthreads();
    for (int j = 0; j < n; ++j) {
        const double piv = ab[(int64_t)kd * n + j];
        if (piv == 0.0) {
            if (threadIdx.x == 0) *info = j + 1;
            return;
        }
        const int km = min(q, n - 1 - j);          // rows below the diagonal in this column
        if ((int)threadIdx.x < km) ab[(int64_t)(kd + 1 + threadIdx.x) * n + j] /= piv;
        __syncthreads();
        const int ju = min(q, n - 1 - j);          // columns right of the diagonal
        for (int t = threadIdx.x; t < km * ju; t += blockDim.x) {
            const int i = t / ju + 1, c = t - (t / ju) * ju + 1;     // A[j+i, j+c] -= l_i * A[j, j+c]
            ab[(int64_t)(kd + i - c) * n + (j + c)] -= ab[(int64_t)(kd + i) * n + j] * ab[(int64_t)(kd - c) * n + (j + c)];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *info = 0;
}

extern "C" int poms_band_lu_nopiv(const double* band, int n, int q, double* ab, int* info_dev, void* stream) {
    if (!band || !ab || !info_dev) return bad_arg(1, "null pointer");
    if (n < 1) return bad_arg(2, "n");
    if (q < 0 || q > 9) return bad_arg(3, "half-bandwidth");
    band_lu_nopiv_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(band, n, q, ab, info_dev);
    CHECK_LAUNCH("poms_band_lu_nopiv");
    return 0;
}
