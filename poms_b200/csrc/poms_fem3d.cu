// poms_fem3d.cu -- load-vector assembly and error integration on tensor-product B-spline spaces.
// Self-contained unit of libpoms_b200.so (own kernels + C ABI, see include/poms_b200.h).
//
//   poms_quad_to_coef_3d:  b (+)= (B1^T (x) B2^T (x) B3^T) F    F = f at the Gauss points of a chunk of
//                          element planes, B_a = basis values with the quadrature weights folded in
//   poms_quad_error_3d:    sum_q w_q (u - u_h)^2 and sum_q w_q |grad u - grad u_h|^2 over a chunk,
//                          u_h and grad u_h evaluated from the coefficients inside the kernel
//
// Both march along axis 1 (the chunk axis of poms_b200/fem.py).  2-D spaces use the same kernels with a
// middle axis of one coefficient and one quadrature point (weight 1, basis value 1): the chunks then still
// run along the first axis.
//
// Load vector (output-centric, no atomics).  CTA: tile of TC2 x 32 coefficient rows of axes (2, 3); it
// reads the quadrature points of every element that touches the tile (halo of p elements per axis:
// (1 + p/TC2)(1 + p/32) <= 1.34 read amplification, 1.30 at p = 3) and marches over the quadrature
// planes of the chunk:
//   per group of 8 quadrature rows:  global -> registers (one group ahead) -> shared (double buffer),
//                                    contracted along axis 3 into H (one row per warp, one output
//                                    column per lane, the 16..36 row weights of the lane in registers)
//   per quadrature plane:            H contracted along axis 2 (weights broadcast from shared memory),
//                                    added into the p+1 axis-1 partial sums (registers) of each point
//   per element plane:               the rows the element plane completes are stored (first chunk) or
//                                    added (rows that an earlier chunk already touched).
// The quadrature row is stored in shared memory DE-interleaved (point q of element e at q * exte + e), so
// that the lanes of a warp, whose rows start at consecutive elements, read consecutive words.
//
// Error (gather form).  CTA: 32 x 32 quadrature points of axes (2, 3) and a range of quadrature planes.
// Per plane: the p+1 coefficient planes it needs (re-read only when the element plane changes) are
// contracted along axis 1 (values and derivatives), then along axis 3, then along axis 2 per point; the
// weighted squares are reduced per CTA and summed by the last CTA in a fixed order (per-CTA slots and a
// ticket in the workspace): deterministic.
//
// POMS_HOST_EMU is never defined by build.py.  tests/test_fem_host_emulation.py defines it to compile THIS
// file for the host over tests/host_emu/cuda_emu.h under AddressSanitizer and ThreadSanitizer, with the
// dynamic shared memory of each launch exactly sized.
#ifdef POMS_HOST_EMU
#include "cuda_emu.h"
#define POMS_LAUNCH_SMEM(kernel, grid, smem, stream, arg) EMU_LAUNCH_EX(kernel, grid, 256, smem, stream, arg)
#define FEM_DYN_SMEM(name) double* const name = reinterpret_cast<double*>(emu_dyn_smem)
[[maybe_unused]] static int fail_cuda(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof(g_err), "%s: error %d", where, (int)e);
    return (int)e;
}
#else
#define POMS_TU 99
#include "poms_kernels.cu"
#define POMS_LAUNCH_SMEM(kernel, grid, smem, stream, arg) kernel<<<grid, 256, smem, stream>>>(arg)
#define FEM_DYN_SMEM(name) extern __shared__ double name[]
#endif

namespace {

constexpr int FEM_MAXP = 5;
constexpr int FEM_WS_HEADER = 256;            // = POMS_WS_HEADER: ticket, then the per-CTA slots
constexpr int FEM_MAX_SLOTS = 65536;          // = POMS_MAX_PARTIALS doubles (two per CTA)

int f_bad_arg(int idx, const char* what) {
    snprintf(g_err, sizeof(g_err), "bad argument %d: %s", idx, what);
    return -idx;
}

// ---------------------------------------------------------------------------------------------
// quadrature values -> coefficients
// ---------------------------------------------------------------------------------------------
struct Q2C {
    const double* F;            // F[j1 * fpld + j2 * fld + j3], j1 relative to the chunk
    int64_t fld, fpld;
    double* y;                  // y[r1 * pld + r2 * ld + r3]
    int64_t ld, pld;
    int n1, n2, n3, m2, m3;
    // axis 1: element planes e1_lo .. e1_hi-1 of the chunk; row s1[e] + k gets b1[(e * k1n + k) * q1n + q]
    int e1_lo, e1_hi, k1n, q1n;
    const int32_t* s1;
    const double* b1;
    int store_from;             // rows r1 < store_from are accumulated, the others stored
    // axis 2: row r2 = sum_t c2[r2 * w2 + t] * (quadrature row st2[r2] + t)
    const int32_t* st2;
    const double* c2;
    int w2, ext2;               // ext2: H rows (>= st2[last] + w2 - st2[first] over every tile)
    // axis 3: row r3 = sum_{m, q} c3[r3 * W + m * Q + q] * F[(e3[r3] + m) * Q + q]
    const int32_t* e3;
    const double* c3;
    int ne3, exte;              // exte: staged elements per quadrature point of a row (>= every tile's taps)
};

template <int P>
struct Q2CTile {
    static constexpr int TC2 = P == 1 ? 8 : P <= 3 ? 16 : P == 4 ? 24 : 32;
    static constexpr int NO = TC2 / 8;                                       // output rows per thread
    static constexpr int NPT = (8 * (P + 1) * (32 + P) + 255) / 256;         // staged values per thread
};

template <int P>
__global__ void __launch_bounds__(256) quad_to_coef3d_kernel(const Q2C a) {
    constexpr int Q = P + 1, W = Q * Q, TC2 = Q2CTile<P>::TC2, NO = Q2CTile<P>::NO, NPT = Q2CTile<P>::NPT;
    FEM_DYN_SMEM(sm);
    const int grow = Q * a.exte;                    // one staged quadrature row
    double* const fin = sm;                         // [2][8][Q][exte]
    double* const H = fin + 2 * 8 * grow;           // [ext2][32]
    double* const c2s = H + a.ext2 * 32;            // [TC2][w2]
    const int tid = threadIdx.x, lane = tid & 31, wp = tid >> 5;
    const int r3_0 = blockIdx.x * 32, r2_0 = blockIdx.y * TC2;
    const int r3n = min(32, a.n3 - r3_0), r2n = min(TC2, a.n2 - r2_0);
    const int elo = a.e3[r3_0];
    const int ne = min(a.ne3, a.e3[r3_0 + r3n - 1] + P + 1) - elo;
    const int qlen = ne * Q;
    const int j2lo = a.st2[r2_0];
    const int nr = min(a.m2, a.st2[r2_0 + r2n - 1] + a.w2) - j2lo;
    const int ng = (nr + 7) >> 3;

    for (int t = tid; t < 2 * 8 * grow; t += 256) fin[t] = 0.0;
    for (int t = tid; t < a.ext2 * 32; t += 256) H[t] = 0.0;
    for (int t = tid; t < TC2 * a.w2; t += 256) {
        const int r = t / a.w2;
        c2s[t] = r < r2n ? a.c2[(int64_t)r2_0 * a.w2 + t] : 0.0;
    }
    const bool v3 = lane < r3n;
    double c3r[W];
#pragma unroll
    for (int t = 0; t < W; ++t) c3r[t] = v3 ? a.c3[(int64_t)(r3_0 + lane) * W + t] : 0.0;
    const int o3 = v3 ? a.e3[r3_0 + lane] - elo : 0;
    int o2[NO];
#pragma unroll
    for (int i = 0; i < NO; ++i) {
        const int r = wp + 8 * i;
        o2[i] = r < r2n ? a.st2[r2_0 + r] - j2lo : 0;
    }
    // this thread's slots of a staged group (8 rows x qlen points)
    int64_t go[NPT];
    int so[NPT], srow[NPT];
#pragma unroll
    for (int m = 0; m < NPT; ++m) {
        const int slot = tid + 256 * m;
        const int row = slot / qlen, col = slot - row * qlen;
        srow[m] = row < 8 ? row : 8;
        go[m] = row < 8 ? (int64_t)row * a.fld + col : 0;
        so[m] = row < 8 ? row * grow + (col % Q) * a.exte + col / Q : 0;
    }
    const int nq1 = (a.e1_hi - a.e1_lo) * a.q1n;
    const int total = nq1 * ng;
    const double* const fbase = a.F + (int64_t)j2lo * a.fld + (int64_t)elo * Q;
    double pre[NPT];
    auto load = [&](const int G) {
        const int j1 = G / ng, g = G - j1 * ng;
        const double* const p = fbase + (int64_t)j1 * a.fpld + (int64_t)(8 * g) * a.fld;
        const int rows = nr - 8 * g;
#pragma unroll
        for (int m = 0; m < NPT; ++m) pre[m] = srow[m] < rows ? __ldg(p + go[m]) : 0.0;
    };
    double acc[P + 1][NO];
#pragma unroll
    for (int k = 0; k <= P; ++k)
#pragma unroll
        for (int i = 0; i < NO; ++i) acc[k][i] = 0.0;
    load(0);
    __syncthreads();

#pragma unroll 1
    for (int G = 0; G < total; ++G) {
        double* const buf = fin + (G & 1) * 8 * grow;
#pragma unroll
        for (int m = 0; m < NPT; ++m)
            if (srow[m] < 8) buf[so[m]] = pre[m];
        if (G + 1 < total) load(G + 1);
        __syncthreads();
        const int j1 = G / ng, g = G - j1 * ng;
        const int jrow = 8 * g + wp;
        if (jrow < nr) {
            const double* const br = buf + wp * grow + o3;
            double h = 0.0;
#pragma unroll
            for (int m = 0; m <= P; ++m)
#pragma unroll
                for (int q = 0; q < Q; ++q) h = fma(c3r[m * Q + q], br[q * a.exte + m], h);
            H[jrow * 32 + lane] = h;
        }
        if (g != ng - 1) continue;
        // quadrature plane j1 complete: axis 2, then the axis-1 partial sums
        __syncthreads();
        const int e1 = a.e1_lo + j1 / a.q1n, q1 = j1 - (j1 / a.q1n) * a.q1n;
        double val[NO];
#pragma unroll
        for (int i = 0; i < NO; ++i) {
            const double* const cr = c2s + (wp + 8 * i) * a.w2;
            const double* const hp = H + o2[i] * 32 + lane;
            double v = 0.0;
#pragma unroll 4
            for (int t = 0; t < a.w2; ++t) v = fma(cr[t], hp[t * 32], v);
            val[i] = v;
        }
#pragma unroll
        for (int k = 0; k <= P; ++k) {
            if (k < a.k1n) {
                const double b = __ldg(a.b1 + ((int64_t)e1 * a.k1n + k) * a.q1n + q1);
#pragma unroll
                for (int i = 0; i < NO; ++i) acc[k][i] = fma(b, val[i], acc[k][i]);
            }
        }
        if (q1 != a.q1n - 1) continue;
        // element plane e1 complete: emit the rows no later element plane of the chunk touches
        const int s = a.s1[e1];
        const int nxt = e1 + 1 < a.e1_hi ? a.s1[e1 + 1] : s + a.k1n;
#pragma unroll 1
        for (int r1 = s; r1 < nxt; ++r1) {
            if (v3) {
#pragma unroll
                for (int i = 0; i < NO; ++i) {
                    const int r2 = wp + 8 * i;
                    if (r2 < r2n) {
                        double* const yp = a.y + (int64_t)r1 * a.pld + (int64_t)(r2_0 + r2) * a.ld + r3_0 + lane;
                        *yp = r1 < a.store_from ? *yp + acc[0][i] : acc[0][i];
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < P; ++k)
#pragma unroll
                for (int i = 0; i < NO; ++i) acc[k][i] = acc[k + 1][i];
#pragma unroll
            for (int i = 0; i < NO; ++i) acc[P][i] = 0.0;
        }
    }
}

template <int P>
int launch_q2c(const Q2C& a, cudaStream_t st) {
    constexpr int TC2 = Q2CTile<P>::TC2;
    const size_t smem = sizeof(double) * ((size_t)2 * 8 * (P + 1) * a.exte + (size_t)a.ext2 * 32 + (size_t)TC2 * a.w2);
    if (smem > 227 * 1024) return f_bad_arg(2, "quadrature tile does not fit the shared memory");
    const dim3 grid((a.n3 + 31) / 32, (a.n2 + TC2 - 1) / TC2, 1);
    if (grid.y > 65535) return f_bad_arg(2, "grid too large");
    if (smem > 48 * 1024) {        // above the default limit: opt in (per device context, so on every launch)
        const cudaError_t e = cudaFuncSetAttribute(quad_to_coef3d_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail_cuda(e, "poms_quad_to_coef_3d: cudaFuncSetAttribute");
    }
    POMS_LAUNCH_SMEM(quad_to_coef3d_kernel<P>, grid, smem, st, a);
    CHECK_LAUNCH("poms_quad_to_coef_3d");
    return 0;
}

// rows of one axis: starts nondecreasing and inside [0, n_in)
bool starts_ok(const int32_t* s, int n, int n_in) {
    for (int i = 0; i < n; ++i)
        if (s[i] < 0 || s[i] >= n_in || (i && s[i] < s[i - 1])) return false;
    return true;
}

// ---------------------------------------------------------------------------------------------
// error integration
// ---------------------------------------------------------------------------------------------
struct QErr {
    const double* x;            // x[r1 * pld + r2 * ld + r3]
    int64_t ld, pld;
    int n1, n2, n3, m2, m3;
    const double* ref[4];       // u, du/dx1, du/dx2, du/dx3 at the chunk's points (gradient: null = skip)
    int64_t rld[4], rpld[4];
    int j1_lo, nq1, ppc;        // first (global) quadrature plane, planes of the chunk, planes per CTA
    // per quadrature point j of axis a: first coefficient s[j], values v[j * k + i], derivatives d, weight w
    int k1n, k2n;
    const int32_t *s1, *s2, *s3;
    const double *v1, *d1, *w1, *v2, *d2, *w2, *v3, *d3, *w3;
    int c2max, c3max, grad, accumulate;
    double* out;                // out[0] (+)= L2 squared, out[1] (+)= H1 seminorm squared
    void* ws;
};

// sum of v over the CTA, in a fixed order (result in thread 0); red: 256 doubles
__device__ __forceinline__ double cta_sum(double v, double* red) {
    const int tid = threadIdx.x;
    red[tid] = v;
    __syncthreads();
#pragma unroll 1
    for (int h = 128; h > 0; h >>= 1) {
        if (tid < h) red[tid] += red[tid + h];
        __syncthreads();
    }
    const double s = red[0];
    __syncthreads();
    return s;
}

template <int P>
__global__ void __launch_bounds__(256) quad_error3d_kernel(const QErr a) {
    constexpr int K3 = P + 1;
    FEM_DYN_SMEM(sm);
    const int cpl = a.c2max * a.c3max;
    double* const X = sm;                               // [P+1][c2max][c3max]
    double* const A0 = X + (P + 1) * cpl;               // [c2max][c3max]  axis-1 values
    double* const A1 = A0 + cpl;                        //                 axis-1 derivatives
    double* const B0 = A1 + cpl;                        // [c2max][32]     then axis-3 values
    double* const B3 = B0 + a.c2max * 32;               //                 axis-3 derivative of A0
    double* const B1 = B3 + a.c2max * 32;               //                 axis-3 values of A1
    double* const red = B1 + a.c2max * 32;              // [256]
    __shared__ unsigned s_last;
    const int tid = threadIdx.x, lane = tid & 31, wp = tid >> 5;
    const int J3 = blockIdx.x * 32;
    const int n3q = min(32, a.m3 - J3);
    const int g2 = (a.m2 + 31) / 32;
    const bool v3 = lane < n3q;
    const int j3 = J3 + (v3 ? lane : 0);
    const int c3lo = a.s3[J3];
    const int c3n = a.s3[J3 + n3q - 1] + K3 - c3lo;
    double v3r[K3], d3r[K3];
#pragma unroll
    for (int k = 0; k < K3; ++k) {
        v3r[k] = a.v3[(int64_t)j3 * K3 + k];
        d3r[k] = a.d3[(int64_t)j3 * K3 + k];
    }
    const int o3 = a.s3[j3] - c3lo;
    const double w3 = v3 ? a.w3[j3] : 0.0;
    const int jj_lo = blockIdx.z * a.ppc, jj_hi = min(a.nq1, jj_lo + a.ppc);
    double sl2 = 0.0, sh1 = 0.0;

#pragma unroll 1
    for (int ty = blockIdx.y; ty < g2; ty += gridDim.y) {
        const int J2 = ty * 32;
        const int n2q = min(32, a.m2 - J2);
        const int c2lo = a.s2[J2];
        const int c2n = a.s2[J2 + n2q - 1] + a.k2n - c2lo;
        int cur = -1;
#pragma unroll 1
        for (int jj = jj_lo; jj < jj_hi; ++jj) {
            const int j = a.j1_lo + jj;
            const int s = a.s1[j];
            if (s != cur) {            // coefficient planes s .. s+k1n-1 of the tile
                cur = s;
                for (int t = tid; t < a.k1n * c2n * c3n; t += 256) {
                    const int k = t / (c2n * c3n), rem = t - k * (c2n * c3n);
                    const int r2 = rem / c3n, r3 = rem - r2 * c3n;
                    X[k * cpl + r2 * a.c3max + r3] =
                        a.x[(int64_t)(s + k) * a.pld + (int64_t)(c2lo + r2) * a.ld + c3lo + r3];
                }
            }
            __syncthreads();
            for (int t = tid; t < c2n * c3n; t += 256) {
                const int r2 = t / c3n, r3 = t - r2 * c3n;
                const int o = r2 * a.c3max + r3;
                double u = 0.0, du = 0.0;
                for (int k = 0; k < a.k1n; ++k) {
                    const double xv = X[k * cpl + o];
                    u = fma(a.v1[(int64_t)j * a.k1n + k], xv, u);
                    du = fma(a.d1[(int64_t)j * a.k1n + k], xv, du);
                }
                A0[o] = u;
                A1[o] = du;
            }
            __syncthreads();
            for (int r2 = wp; r2 < c2n; r2 += 8) {
                const double* const a0 = A0 + r2 * a.c3max + o3;
                const double* const a1 = A1 + r2 * a.c3max + o3;
                double b0 = 0.0, b3 = 0.0, b1 = 0.0;
#pragma unroll
                for (int k = 0; k < K3; ++k) {
                    b0 = fma(v3r[k], a0[k], b0);
                    b3 = fma(d3r[k], a0[k], b3);
                    b1 = fma(v3r[k], a1[k], b1);
                }
                B0[r2 * 32 + lane] = b0;
                B3[r2 * 32 + lane] = b3;
                B1[r2 * 32 + lane] = b1;
            }
            __syncthreads();
            const double w1 = a.w1[j];
#pragma unroll 1
            for (int r = wp; r < n2q; r += 8) {
                if (!v3) continue;
                const int j2 = J2 + r;
                const int o2 = a.s2[j2] - c2lo;
                double uh = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;
                for (int k = 0; k < a.k2n; ++k) {
                    const double vv = a.v2[(int64_t)j2 * a.k2n + k], dd = a.d2[(int64_t)j2 * a.k2n + k];
                    const int o = (o2 + k) * 32 + lane;
                    uh = fma(vv, B0[o], uh);
                    e1 = fma(vv, B1[o], e1);
                    e2 = fma(dd, B0[o], e2);
                    e3 = fma(vv, B3[o], e3);
                }
                const double wq = w1 * a.w2[j2] * w3;
                const int64_t off = j3;
                const double du0 = a.ref[0][(int64_t)jj * a.rpld[0] + (int64_t)j2 * a.rld[0] + off] - uh;
                sl2 = fma(wq * du0, du0, sl2);
                if (a.grad) {
                    double g = 0.0, t;
                    if (a.ref[1]) { t = a.ref[1][(int64_t)jj * a.rpld[1] + (int64_t)j2 * a.rld[1] + off] - e1; g = fma(t, t, g); }
                    if (a.ref[2]) { t = a.ref[2][(int64_t)jj * a.rpld[2] + (int64_t)j2 * a.rld[2] + off] - e2; g = fma(t, t, g); }
                    if (a.ref[3]) { t = a.ref[3][(int64_t)jj * a.rpld[3] + (int64_t)j2 * a.rld[3] + off] - e3; g = fma(t, t, g); }
                    sh1 = fma(wq, g, sh1);
                }
            }
            __syncthreads();
        }
    }
    // deterministic grid reduction: per-CTA slots, ticket, fixed-order sum in the last CTA
    const double t0 = cta_sum(sl2, red), t1 = cta_sum(sh1, red);
    const unsigned nb = gridDim.x * gridDim.y * gridDim.z;
    const unsigned bid = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
    unsigned* const ticket = (unsigned*)a.ws;
    double* const part = (double*)((char*)a.ws + FEM_WS_HEADER);
    if (tid == 0) {
        part[2 * bid] = t0;
        part[2 * bid + 1] = t1;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == nb - 1 ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        double q0 = 0.0, q1 = 0.0;
        for (unsigned i = tid; i < nb; i += 256) {
            q0 += __ldcg(part + 2 * i);
            q1 += __ldcg(part + 2 * i + 1);
        }
        q0 = cta_sum(q0, red);
        q1 = cta_sum(q1, red);
        if (tid == 0) {
            a.out[0] = a.accumulate ? a.out[0] + q0 : q0;
            a.out[1] = a.accumulate ? a.out[1] + q1 : q1;
            *ticket = 0u;
        }
    }
}

template <int P>
int launch_err(const QErr& a, dim3 grid, cudaStream_t st) {
    const size_t smem = sizeof(double) * ((size_t)(P + 3) * a.c2max * a.c3max + (size_t)3 * a.c2max * 32 + 256);
    if (smem > 227 * 1024) return f_bad_arg(2, "quadrature tile does not fit the shared memory");
    if (smem > 48 * 1024) {        // above the default limit: opt in (per device context, so on every launch)
        const cudaError_t e = cudaFuncSetAttribute(quad_error3d_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail_cuda(e, "poms_quad_error_3d: cudaFuncSetAttribute");
    }
    POMS_LAUNCH_SMEM(quad_error3d_kernel<P>, grid, smem, st, a);
    CHECK_LAUNCH("poms_quad_error_3d");
    return 0;
}

// largest coefficient window of a tile of `tile` consecutive quadrature points
int quad_window(const int32_t* s, int m, int k, int tile) {
    int w = 0;
    for (int j0 = 0; j0 < m; j0 += tile) {
        const int j1 = min(m, j0 + tile) - 1;
        w = max(w, s[j1] + k - s[j0]);
    }
    return w;
}

}  // namespace

// F: quadrature values of element planes e1_lo .. e1_hi-1 (Q1 = q1n planes each), shape (nq1, m2, m3) with
// row pitch fld and plane pitch fpld.  Rows r1 < store_from are added to y, the others overwritten.
// Host copies of the small index tables (s1_host, st2_host, e3_host) are used for argument checks and
// tile sizes; the device copies for the kernel.
extern "C" int poms_quad_to_coef_3d(const double* F, int64_t fld, int64_t fpld, double* y, int64_t ld,
                                    int64_t pld, int n1, int n2, int n3, int m2, int m3, int p, int e1_lo,
                                    int e1_hi, int k1n, int q1n, const int32_t* s1, const double* b1,
                                    int store_from, const int32_t* st2, const double* c2, int w2,
                                    const int32_t* e3, const double* c3, int ne3, const int32_t* s1_host,
                                    const int32_t* st2_host, const int32_t* e3_host, void* stream) {
    if (!F || !y || !s1 || !b1 || !st2 || !c2 || !e3 || !c3 || !s1_host || !st2_host || !e3_host)
        return f_bad_arg(1, "null pointer");
    if (n1 < 1 || n2 < 1 || n3 < 1 || m2 < 1 || m3 < 1) return f_bad_arg(7, "empty grid");
    if (p < 1 || p > FEM_MAXP) return f_bad_arg(12, "p must be 1..5");
    if (e1_lo < 0 || e1_hi <= e1_lo || k1n < 1 || k1n > p + 1 || q1n < 1) return f_bad_arg(13, "axis-1 elements");
    if (ld < n3 || pld < (int64_t)n2 * ld || fld < m3 || fpld < (int64_t)m2 * fld) return f_bad_arg(2, "pitch");
    if (w2 < 1 || w2 > (p + 1) * (p + 1)) return f_bad_arg(22, "axis-2 row width");
    if (ne3 * (p + 1) != m3) return f_bad_arg(25, "axis-3 elements do not match m3");
    for (int e = e1_lo; e < e1_hi; ++e)
        if (s1_host[e] < 0 || s1_host[e] + k1n > n1 || (e > e1_lo && s1_host[e] < s1_host[e - 1]))
            return f_bad_arg(17, "axis-1 element starts");
    if (!starts_ok(st2_host, n2, m2) || !starts_ok(e3_host, n3, ne3)) return f_bad_arg(20, "row starts");
    Q2C a;
    a.F = F; a.fld = fld; a.fpld = fpld; a.y = y; a.ld = ld; a.pld = pld;
    a.n1 = n1; a.n2 = n2; a.n3 = n3; a.m2 = m2; a.m3 = m3;
    a.e1_lo = e1_lo; a.e1_hi = e1_hi; a.k1n = k1n; a.q1n = q1n; a.s1 = s1; a.b1 = b1; a.store_from = store_from;
    a.st2 = st2; a.c2 = c2; a.w2 = w2; a.e3 = e3; a.c3 = c3; a.ne3 = ne3;
    int tc2;
    switch (p) {
        case 1: tc2 = Q2CTile<1>::TC2; break;
        case 2: tc2 = Q2CTile<2>::TC2; break;
        case 3: tc2 = Q2CTile<3>::TC2; break;
        case 4: tc2 = Q2CTile<4>::TC2; break;
        default: tc2 = Q2CTile<5>::TC2; break;
    }
    a.ext2 = 0;
    for (int i0 = 0; i0 < n2; i0 += tc2) {
        const int i1 = min(n2, i0 + tc2) - 1;
        a.ext2 = max(a.ext2, st2_host[i1] + w2 - st2_host[i0]);
    }
    a.exte = 0;
    for (int i0 = 0; i0 < n3; i0 += 32) {
        const int i1 = min(n3, i0 + 32) - 1;
        a.exte = max(a.exte, e3_host[i1] + p + 1 - e3_host[i0]);    // (taps past ne3: zero weights)
    }
    if (a.exte > 32 + p) return f_bad_arg(23, "axis-3 rows span too many elements");
    cudaStream_t st = (cudaStream_t)stream;
    switch (p) {
        case 1: return launch_q2c<1>(a, st);
        case 2: return launch_q2c<2>(a, st);
        case 3: return launch_q2c<3>(a, st);
        case 4: return launch_q2c<4>(a, st);
        default: return launch_q2c<5>(a, st);
    }
}

// Reference values ref[0] (u) and, with grad, ref[1..3] (the gradient; a null component is skipped) at the
// quadrature planes j1_lo .. j1_lo+nq1-1, each of shape (nq1, m2, m3) with its own pitches.  Per-point
// tables of axis a: s_a (first coefficient), v_a / d_a (k_a values / derivatives), w_a (weight); k3 = p+1.
// out[0] (+)= sum w (u - u_h)^2, out[1] (+)= sum w |grad u - grad u_h|^2.  ws: the library workspace.
extern "C" int poms_quad_error_3d(const double* x, int64_t ld, int64_t pld, int n1, int n2, int n3, int m2, int m3,
                                  int p, const double* const* ref, const int64_t* rld, const int64_t* rpld,
                                  int j1_lo, int nq1, int k1n, const int32_t* s1, const double* v1,
                                  const double* d1, const double* w1, int k2n, const int32_t* s2,
                                  const double* v2, const double* d2, const double* w2, const int32_t* s3,
                                  const double* v3, const double* d3, const double* w3,
                                  const int32_t* s1_host, const int32_t* s2_host, const int32_t* s3_host,
                                  int m1, int grad, int accumulate, double* out, void* ws, void* stream) {
    if (!x || !ref || !ref[0] || !rld || !rpld || !s1 || !v1 || !d1 || !w1 || !s2 || !v2 || !d2 || !w2 || !s3 ||
        !v3 || !d3 || !w3 || !s1_host || !s2_host || !s3_host || !out || !ws)
        return f_bad_arg(1, "null pointer");
    if (n1 < 1 || n2 < 1 || n3 < 1 || m1 < 1 || m2 < 1 || m3 < 1 || nq1 < 1) return f_bad_arg(4, "empty grid");
    if (p < 1 || p > FEM_MAXP) return f_bad_arg(9, "p must be 1..5");
    if (j1_lo < 0 || j1_lo + nq1 > m1) return f_bad_arg(13, "chunk outside the quadrature planes");
    if (k1n < 1 || k1n > p + 1 || k2n < 1 || k2n > p + 1) return f_bad_arg(15, "basis functions per point");
    if (ld < n3 || pld < (int64_t)n2 * ld) return f_bad_arg(2, "pitch");
    for (int c = 0; c < 4; ++c)
        if (ref[c] && (rld[c] < 0 || rpld[c] < 0)) return f_bad_arg(11, "reference pitch");
    for (int j = 0; j < m1; ++j)
        if (s1_host[j] < 0 || s1_host[j] + k1n > n1 || (j && s1_host[j] < s1_host[j - 1]))
            return f_bad_arg(31, "axis-1 starts");
    for (int j = 0; j < m2; ++j)
        if (s2_host[j] < 0 || s2_host[j] + k2n > n2 || (j && s2_host[j] < s2_host[j - 1]))
            return f_bad_arg(32, "axis-2 starts");
    for (int j = 0; j < m3; ++j)
        if (s3_host[j] < 0 || s3_host[j] + p + 1 > n3 || (j && s3_host[j] < s3_host[j - 1]))
            return f_bad_arg(33, "axis-3 starts");
    QErr a;
    a.x = x; a.ld = ld; a.pld = pld; a.n1 = n1; a.n2 = n2; a.n3 = n3; a.m2 = m2; a.m3 = m3;
    for (int c = 0; c < 4; ++c) {
        a.ref[c] = (c == 0 || grad) ? ref[c] : nullptr;
        a.rld[c] = rld[c];
        a.rpld[c] = rpld[c];
    }
    a.j1_lo = j1_lo; a.nq1 = nq1; a.k1n = k1n; a.k2n = k2n;
    a.s1 = s1; a.s2 = s2; a.s3 = s3; a.v1 = v1; a.d1 = d1; a.w1 = w1; a.v2 = v2; a.d2 = d2; a.w2 = w2;
    a.v3 = v3; a.d3 = d3; a.w3 = w3;
    a.grad = grad; a.accumulate = accumulate; a.out = out; a.ws = ws;
    a.c2max = quad_window(s2_host, m2, k2n, 32);
    a.c3max = quad_window(s3_host, m3, p + 1, 32);
    // grid: 32 x 32 point tiles x ranges of planes; at most FEM_MAX_SLOTS / 2 CTAs (two slots each), the
    // tiles of axis 2 are looped over when there are more
    const int g3 = (m3 + 31) / 32, g2 = (m2 + 31) / 32;
    if (g3 > FEM_MAX_SLOTS / 2) return f_bad_arg(8, "grid too large");
    int64_t gz = (1184 + (int64_t)g3 * g2 - 1) / ((int64_t)g3 * g2);
    if (gz > nq1) gz = nq1;
    a.ppc = (int)((nq1 + gz - 1) / gz);
    gz = (nq1 + a.ppc - 1) / a.ppc;
    int64_t gy = g2;
    if ((int64_t)g3 * gy * gz > FEM_MAX_SLOTS / 2) gy = (FEM_MAX_SLOTS / 2) / ((int64_t)g3 * gz);
    if (gy < 1) {
        gz = 1;
        a.ppc = nq1;
        gy = max((int64_t)1, (int64_t)(FEM_MAX_SLOTS / 2) / g3);
        if (gy > g2) gy = g2;
    }
    const dim3 grid(g3, (unsigned)gy, (unsigned)gz);
    if (grid.y > 65535 || grid.z > 65535) return f_bad_arg(8, "grid too large");
    cudaStream_t st = (cudaStream_t)stream;
    switch (p) {
        case 1: return launch_err<1>(a, grid, st);
        case 2: return launch_err<2>(a, grid, st);
        case 3: return launch_err<3>(a, grid, st);
        case 4: return launch_err<4>(a, grid, st);
        default: return launch_err<5>(a, grid, st);
    }
}
