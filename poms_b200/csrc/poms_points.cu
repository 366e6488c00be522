// poms_points.cu -- particle coupling on tensor-product B-spline spaces: u_h and grad u_h at scattered points,
// and the deposit of point weights into a load vector, b_i = sum_k w_k phi_i(X_k).
// Self-contained unit of libpoms_b200.so (own kernels + C ABI, see include/poms_b200.h).
//
//   poms_points_eval:      u[k] = u_h(X_k), g[k, :] = grad u_h(X_k)      one thread per point
//   poms_points_locate:    key[k] = the cell of X_k                       one thread per point
//   poms_points_moments:   M[c, i] = sum_{k in c} w_k phi_i(X_k)          one warp per cell of a chunk
//   poms_points_assemble:  b (+)= the moments of the <= (p+1)^d cells of each coefficient
//
// Cells are the knot spans: axis a has C_a = n_a - p spans k = p .. n_a - 1, cell coordinate c = k - p (a
// span of zero length, at a repeated knot, is a cell no point falls into), key = (c1 C2 + c2) C3 + c3.  A
// point belongs to the span with T[k] <= x < T[k+1]; a point at T[n] to the last non-empty span (the
// convention of scipy's BSpline and of fem.evaluate), so derivatives on a breakpoint are right-hand ones.
// Per axis: a binary search of the knot vector, then the Cox-de Boor triangle with first derivatives in
// registers (the recursion of bsplines._all_basis).
//
// The deposit has no atomics and is deterministic: the points are sorted by cell (poms_b200/fem.py, a stable
// sort), a warp sums the points of its cell in that order, in batches of 32 (lane l evaluates the basis of
// point l of the batch into warp-private shared memory, then every lane accumulates its targets over the
// batch), and the assembly is output-centric: each coefficient adds the moments of its cells in a fixed
// order.  The moments of a chunk of cell planes along axis 1 are the only scratch besides the sort; rows
// shared with the previous chunk are added to (rows r1 < store_from), the others stored.
//
// A 2-D space runs through the same kernels with T2 = NULL and n2 = 1: a middle axis of one coefficient and
// one cell, basis value 1, derivative 0.  Points then have d = 2 coordinates (axes 1 and 3).
//
// POMS_HOST_EMU is never defined by build.py.  tests/test_points_host_emulation.py defines it to compile THIS
// file for the host over tests/host_emu/cuda_emu.h under AddressSanitizer and ThreadSanitizer, with the
// dynamic shared memory of each launch exactly sized.
#ifdef POMS_HOST_EMU
#include "cuda_emu.h"
#define PT_LAUNCH(kernel, grid, smem, stream, arg) EMU_LAUNCH_EX(kernel, grid, 256, smem, stream, arg)
#define PT_DYN_SMEM(name) double* const name = reinterpret_cast<double*>(emu_dyn_smem)
[[maybe_unused]] static int fail_cuda(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof(g_err), "%s: error %d", where, (int)e);
    return (int)e;
}
#else
#define POMS_TU 99
#include "poms_kernels.cu"
#define PT_LAUNCH(kernel, grid, smem, stream, arg) kernel<<<grid, 256, smem, stream>>>(arg)
#define PT_DYN_SMEM(name) extern __shared__ double name[]
#endif

namespace {

constexpr int PT_MAXP = 5;
constexpr int64_t PT_MAX_POINTS = (int64_t)1 << 31;        // m < 2^31 (fem.py checks it too)
constexpr int PT_WARPS = 8;                                 // warps (cells) per CTA of the moments kernel

int pt_bad_arg(int idx, const char* what) {
    snprintf(g_err, sizeof(g_err), "bad argument %d: %s", idx, what);
    return -idx;
}

struct PtAxes {
    const double* T[3];         // knot vectors (n_a + p + 1 entries); T[1] == NULL: 2-D, singleton middle axis
    int n[3];                   // coefficients per axis
};

// largest span k in [p, n-1] with T[k] <= x and T[k] < T[n] (x inside [T[p], T[n]])
__device__ __forceinline__ int find_span(const double* T, int n, int p, double x) {
    const double tn = __ldg(T + n);
    int lo = p, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        const double t = __ldg(T + mid);
        if (t <= x && t < tn)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// values N[j] and (DER) first derivatives dN[j] of the P+1 B-splines k-P+j that are non-zero on span k
template <int P, bool DER>
__device__ __forceinline__ void basis(const double* T, int k, double x, double (&N)[P + 1], double (&dN)[P + 1]) {
    double left[P + 1], right[P + 1], Np[P + 1];
    N[0] = 1.0;
#pragma unroll
    for (int d = 1; d <= P; ++d) {
        left[d] = x - __ldg(T + k + 1 - d);
        right[d] = __ldg(T + k + d) - x;
        if (d == P) {
#pragma unroll
            for (int r = 0; r < P; ++r) Np[r] = N[r];      // degree P-1 values
        }
        double saved = 0.0;
#pragma unroll
        for (int r = 0; r < d; ++r) {
            const double tmp = N[r] / (right[r + 1] + left[d - r]);
            N[r] = saved + right[r + 1] * tmp;
            saved = left[d - r] * tmp;
        }
        N[d] = saved;
    }
    if (DER) {
#pragma unroll
        for (int j = 0; j <= P; ++j) {
            const int i = k - P + j;
            double v = 0.0;
            if (j >= 1) v += P * Np[j - 1] / (__ldg(T + i + P) - __ldg(T + i));
            if (j <= P - 1) v -= P * Np[j] / (__ldg(T + i + P + 1) - __ldg(T + i + 1));
            dN[j] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// evaluation
// ---------------------------------------------------------------------------------------------
struct PtEval {
    const double* x;            // x[r1 * pld + r2 * ld + r3]
    int64_t ld, pld;
    PtAxes ax;
    const double* pts;          // pts[k * d + a]
    int d;
    int64_t m;
    double* u;                  // u[k]
    double* g;                  // g[k * d + a] (GRAD)
};

template <int P, bool GRAD>
__global__ void __launch_bounds__(256) points_eval_kernel(const PtEval a) {
    constexpr int K = P + 1;
    const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (k >= a.m) return;
    const double* const X = a.pts + k * a.d;
    double N1[K], D1[K], N2[K], D2[K], N3[K], D3[K];
    const int k1 = find_span(a.ax.T[0], a.ax.n[0], P, __ldg(X));
    basis<P, GRAD>(a.ax.T[0], k1, __ldg(X), N1, D1);
    const int k3 = find_span(a.ax.T[2], a.ax.n[2], P, __ldg(X + a.d - 1));
    basis<P, GRAD>(a.ax.T[2], k3, __ldg(X + a.d - 1), N3, D3);
    const bool three = a.ax.T[1] != nullptr;
    int s2 = 0;
    if (three) {
        const int k2 = find_span(a.ax.T[1], a.ax.n[1], P, __ldg(X + 1));
        basis<P, GRAD>(a.ax.T[1], k2, __ldg(X + 1), N2, D2);
        s2 = k2 - P;
    } else {
#pragma unroll
        for (int i = 0; i < K; ++i) N2[i] = D2[i] = 0.0;
        N2[0] = 1.0;
    }
    const int k2n = three ? K : 1;
    const double* const xb = a.x + (int64_t)(k1 - P) * a.pld + (int64_t)s2 * a.ld + (k3 - P);
    double u = 0.0, g1 = 0.0, g2 = 0.0, g3 = 0.0;
#pragma unroll
    for (int i1 = 0; i1 < K; ++i1) {
        double r0 = 0.0, r2 = 0.0, r3 = 0.0;
#pragma unroll
        for (int i2 = 0; i2 < K; ++i2) {
            if (i2 < k2n) {
                const double* const row = xb + (int64_t)i1 * a.pld + (int64_t)i2 * a.ld;
                double c0 = 0.0, c3 = 0.0;
#pragma unroll
                for (int i3 = 0; i3 < K; ++i3) {
                    const double c = __ldg(row + i3);
                    c0 = fma(N3[i3], c, c0);
                    if (GRAD) c3 = fma(D3[i3], c, c3);
                }
                r0 = fma(N2[i2], c0, r0);
                if (GRAD) {
                    r2 = fma(D2[i2], c0, r2);
                    r3 = fma(N2[i2], c3, r3);
                }
            }
        }
        u = fma(N1[i1], r0, u);
        if (GRAD) {
            g1 = fma(D1[i1], r0, g1);
            g2 = fma(N1[i1], r2, g2);
            g3 = fma(N1[i1], r3, g3);
        }
    }
    a.u[k] = u;
    if (GRAD) {
        double* const G = a.g + k * a.d;
        G[0] = g1;
        if (three) {
            G[1] = g2;
            G[2] = g3;
        } else {
            G[1] = g3;
        }
    }
}

template <int P>
int launch_eval(const PtEval& a, cudaStream_t st) {
    const dim3 grid((unsigned)((a.m + 255) / 256));
    if (a.g)
        PT_LAUNCH((points_eval_kernel<P, true>), grid, 0, st, a);
    else
        PT_LAUNCH((points_eval_kernel<P, false>), grid, 0, st, a);
    CHECK_LAUNCH("poms_points_eval");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// deposit: locate, moments, assemble
// ---------------------------------------------------------------------------------------------
struct PtLocate {
    PtAxes ax;
    int p;
    const double* pts;
    int d;
    int64_t m;
    int64_t C2, C3;             // cells of axes 2 and 3
    int64_t* key;
};

__global__ void __launch_bounds__(256) points_locate_kernel(const PtLocate a) {
    const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (k >= a.m) return;
    const double* const X = a.pts + k * a.d;
    const int64_t c1 = find_span(a.ax.T[0], a.ax.n[0], a.p, __ldg(X)) - a.p;
    const int64_t c2 = a.ax.T[1] ? find_span(a.ax.T[1], a.ax.n[1], a.p, __ldg(X + 1)) - a.p : 0;
    const int64_t c3 = find_span(a.ax.T[2], a.ax.n[2], a.p, __ldg(X + a.d - 1)) - a.p;
    a.key[k] = (c1 * a.C2 + c2) * a.C3 + c3;
}

struct PtMom {
    PtAxes ax;
    const double* pts;
    const double* w;
    int d;
    const int64_t* perm;        // point indices in cell order
    const int64_t* offs;        // the points of cell cell_lo + l are perm[offs[l] .. offs[l+1]-1]
    int64_t cell_lo, ncells;
    int C2, C3;
    double* mom;                // mom[l * nt + (i1 k2n + i2)(P+1) + i3], l = cell - cell_lo
};

template <int P>
__global__ void __launch_bounds__(256) points_moments_kernel(const PtMom a) {
    constexpr int K = P + 1, NA = (K * K * K + 31) / 32;
    PT_DYN_SMEM(sm);
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int64_t l = (int64_t)blockIdx.x * PT_WARPS + wp;
    if (l >= a.ncells) return;                          // (the whole warp)
    double* const sb = sm + wp * (3 * K * 32);          // [3][K][32]: w phi_1, phi_2, phi_3 of the batch
    const bool three = a.ax.T[1] != nullptr;
    const int k2n = three ? K : 1, nt = K * k2n * K;
    const int64_t c = a.cell_lo + l;
    const int c3 = (int)(c % a.C3), c2 = (int)((c / a.C3) % a.C2), c1 = (int)(c / ((int64_t)a.C2 * a.C3));
    int o1[NA], o2[NA], o3[NA];
    double acc[NA];
#pragma unroll
    for (int s = 0; s < NA; ++s) {
        const int t = min(lane + 32 * s, nt - 1);
        o1[s] = (t / (k2n * K)) * 32;
        o2[s] = (K + (t / K) % k2n) * 32;
        o3[s] = (2 * K + t % K) * 32;
        acc[s] = 0.0;
    }
    const int64_t j0 = a.offs[l], j1 = a.offs[l + 1];
#pragma unroll 1
    for (int64_t b = j0; b < j1; b += 32) {
        const int nb = j1 - b < 32 ? (int)(j1 - b) : 32;
        if (lane < nb) {
            const int64_t q = a.perm[b + lane];
            const double* const X = a.pts + q * a.d;
            const double wq = __ldg(a.w + q);
            double N[K], D[K];
            basis<P, false>(a.ax.T[0], c1 + P, __ldg(X), N, D);
#pragma unroll
            for (int i = 0; i < K; ++i) sb[i * 32 + lane] = wq * N[i];
            if (three) {
                basis<P, false>(a.ax.T[1], c2 + P, __ldg(X + 1), N, D);
#pragma unroll
                for (int i = 0; i < K; ++i) sb[(K + i) * 32 + lane] = N[i];
            } else {
                sb[K * 32 + lane] = 1.0;
            }
            basis<P, false>(a.ax.T[2], c3 + P, __ldg(X + a.d - 1), N, D);
#pragma unroll
            for (int i = 0; i < K; ++i) sb[(2 * K + i) * 32 + lane] = N[i];
        }
        __syncwarp();
#pragma unroll 1
        for (int j = 0; j < nb; ++j) {
#pragma unroll
            for (int s = 0; s < NA; ++s) acc[s] = fma(sb[o1[s] + j] * sb[o2[s] + j], sb[o3[s] + j], acc[s]);
        }
        __syncwarp();                                   // the batch is read before the next one is written
    }
    double* const out = a.mom + l * nt;
#pragma unroll
    for (int s = 0; s < NA; ++s)
        if (lane + 32 * s < nt) out[lane + 32 * s] = acc[s];
}

template <int P>
int launch_moments(const PtMom& a, cudaStream_t st) {
    const size_t smem = sizeof(double) * PT_WARPS * 3 * (P + 1) * 32;      // <= 36 KB: no opt-in needed
    const int64_t nblk = (a.ncells + PT_WARPS - 1) / PT_WARPS;
    if (nblk > 0x7fffffff) return pt_bad_arg(6, "chunk has too many cells");
    PT_LAUNCH(points_moments_kernel<P>, dim3((unsigned)nblk), smem, st, a);
    CHECK_LAUNCH("poms_points_moments");
    return 0;
}

struct PtAsm {
    const double* mom;          // moments of the cell planes c1_lo .. c1_hi-1 (poms_points_moments)
    int c1_lo, c1_hi, C2, C3, k2n;
    double* y;                  // y[r1 * pld + r2 * ld + r3]
    int64_t ld, pld;
    int n2, n3, r1_lo, store_from;
    int64_t count;              // rows r1_lo .. : count = (rows) n2 n3
};

template <int P>
__global__ void __launch_bounds__(256) points_assemble_kernel(const PtAsm a) {
    constexpr int K = P + 1;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= a.count) return;
    const int r3 = (int)(idx % a.n3);
    const int64_t t = idx / a.n3;
    const int r2 = (int)(t % a.n2), r1 = a.r1_lo + (int)(t / a.n2);
    const int nt = K * a.k2n * K, p2 = a.k2n - 1;
    const int b1 = max(a.c1_lo, r1 - P), e1 = min(a.c1_hi - 1, r1);
    const int b2 = max(0, r2 - p2), e2 = min(a.C2 - 1, r2);
    const int b3 = max(0, r3 - P), e3 = min(a.C3 - 1, r3);
    double s = 0.0;
    for (int c1 = b1; c1 <= e1; ++c1)
        for (int c2 = b2; c2 <= e2; ++c2) {
            const double* const m = a.mom + (((int64_t)(c1 - a.c1_lo) * a.C2 + c2) * a.C3) * nt +
                                     ((r1 - c1) * a.k2n + (r2 - c2)) * K + r3;
            for (int c3 = b3; c3 <= e3; ++c3) s += __ldg(m + (int64_t)c3 * nt - c3);
        }
    double* const yp = a.y + (int64_t)r1 * a.pld + (int64_t)r2 * a.ld + r3;
    *yp = r1 < a.store_from ? *yp + s : s;
}

template <int P>
int launch_assemble(const PtAsm& a, cudaStream_t st) {
    const int64_t nblk = (a.count + 255) / 256;
    if (nblk > 0x7fffffff) return pt_bad_arg(2, "too many rows");
    PT_LAUNCH(points_assemble_kernel<P>, dim3((unsigned)nblk), 0, st, a);
    CHECK_LAUNCH("poms_points_assemble");
    return 0;
}

// shared checks of the space: returns 0 or a negative status (idx: index of n1 in the caller's arguments)
int check_space(int n1, int n2, int n3, int p, const double* T1, const double* T2, const double* T3, int idx) {
    if (p < 1 || p > PT_MAXP) return pt_bad_arg(idx + 3, "p must be 1..5");
    if (n1 < p + 1 || n3 < p + 1) return pt_bad_arg(idx, "an axis needs n > p coefficients");
    if (T2 ? n2 < p + 1 : n2 != 1) return pt_bad_arg(idx + 1, "n2 (1 with T2 = NULL, 2-D; else > p)");
    if (!T1 || !T3) return pt_bad_arg(idx + 4, "null knot vector");
    return 0;
}

PtAxes make_axes(int n1, int n2, int n3, const double* T1, const double* T2, const double* T3) {
    PtAxes ax;
    ax.T[0] = T1; ax.T[1] = T2; ax.T[2] = T3;
    ax.n[0] = n1; ax.n[1] = n2; ax.n[2] = n3;
    return ax;
}

}  // namespace

extern "C" int poms_points_eval(const double* x, int64_t ld, int64_t pld, int n1, int n2, int n3, int p,
                                const double* T1, const double* T2, const double* T3, const double* pts, int d,
                                int64_t m, double* u, double* g, void* stream) {
    if (!x) return pt_bad_arg(1, "null coefficients");
    if (const int rc = check_space(n1, n2, n3, p, T1, T2, T3, 4)) return rc;
    if (ld < n3 || pld < (int64_t)n2 * ld) return pt_bad_arg(2, "pitch");
    if (d != (T2 ? 3 : 2)) return pt_bad_arg(12, "d must be 3 (T2 given) or 2 (T2 = NULL)");
    if (m < 0 || m >= PT_MAX_POINTS) return pt_bad_arg(13, "m must be in [0, 2^31)");
    if (m > 0 && (!pts || !u)) return pt_bad_arg(11, "null points or output");
    if (m == 0) return 0;
    PtEval a;
    a.x = x; a.ld = ld; a.pld = pld; a.ax = make_axes(n1, n2, n3, T1, T2, T3);
    a.pts = pts; a.d = d; a.m = m; a.u = u; a.g = g;
    cudaStream_t st = (cudaStream_t)stream;
    switch (p) {
        case 1: return launch_eval<1>(a, st);
        case 2: return launch_eval<2>(a, st);
        case 3: return launch_eval<3>(a, st);
        case 4: return launch_eval<4>(a, st);
        default: return launch_eval<5>(a, st);
    }
}

extern "C" int poms_points_locate(const double* pts, int d, int64_t m, int n1, int n2, int n3, int p,
                                  const double* T1, const double* T2, const double* T3, int64_t* key,
                                  void* stream) {
    if (const int rc = check_space(n1, n2, n3, p, T1, T2, T3, 4)) return rc;
    if (d != (T2 ? 3 : 2)) return pt_bad_arg(2, "d must be 3 (T2 given) or 2 (T2 = NULL)");
    if (m < 0 || m >= PT_MAX_POINTS) return pt_bad_arg(3, "m must be in [0, 2^31)");
    if (m > 0 && (!pts || !key)) return pt_bad_arg(1, "null points or keys");
    if (m == 0) return 0;
    PtLocate a;
    a.ax = make_axes(n1, n2, n3, T1, T2, T3);
    a.p = p; a.pts = pts; a.d = d; a.m = m; a.key = key;
    a.C2 = T2 ? n2 - p : 1;
    a.C3 = n3 - p;
    PT_LAUNCH(points_locate_kernel, dim3((unsigned)((m + 255) / 256)), 0, (cudaStream_t)stream, a);
    CHECK_LAUNCH("poms_points_locate");
    return 0;
}

extern "C" int poms_points_moments(const double* pts, const double* w, int d, const int64_t* perm,
                                   const int64_t* offs, int c1_lo, int c1_hi, int n1, int n2, int n3, int p,
                                   const double* T1, const double* T2, const double* T3, double* mom,
                                   void* stream) {
    if (!pts || !w || !perm || !offs || !mom) return pt_bad_arg(1, "null pointer");
    if (const int rc = check_space(n1, n2, n3, p, T1, T2, T3, 8)) return rc;
    if (d != (T2 ? 3 : 2)) return pt_bad_arg(3, "d must be 3 (T2 given) or 2 (T2 = NULL)");
    if (c1_lo < 0 || c1_hi <= c1_lo || c1_hi > n1 - p) return pt_bad_arg(6, "cell planes outside 0 .. n1-p");
    PtMom a;
    a.ax = make_axes(n1, n2, n3, T1, T2, T3);
    a.pts = pts; a.w = w; a.d = d; a.perm = perm; a.offs = offs; a.mom = mom;
    a.C2 = T2 ? n2 - p : 1;
    a.C3 = n3 - p;
    a.cell_lo = (int64_t)c1_lo * a.C2 * a.C3;
    a.ncells = (int64_t)(c1_hi - c1_lo) * a.C2 * a.C3;
    cudaStream_t st = (cudaStream_t)stream;
    switch (p) {
        case 1: return launch_moments<1>(a, st);
        case 2: return launch_moments<2>(a, st);
        case 3: return launch_moments<3>(a, st);
        case 4: return launch_moments<4>(a, st);
        default: return launch_moments<5>(a, st);
    }
}

extern "C" int poms_points_assemble(const double* mom, int c1_lo, int c1_hi, int n1, int n2, int n3, int p,
                                    double* y, int64_t ld, int64_t pld, int store_from, void* stream) {
    if (!mom || !y) return pt_bad_arg(1, "null pointer");
    if (p < 1 || p > PT_MAXP) return pt_bad_arg(7, "p must be 1..5");
    if (n1 < p + 1 || n3 < p + 1 || (n2 != 1 && n2 < p + 1)) return pt_bad_arg(4, "an axis needs n > p coefficients");
    if (c1_lo < 0 || c1_hi <= c1_lo || c1_hi > n1 - p) return pt_bad_arg(2, "cell planes outside 0 .. n1-p");
    if (ld < n3 || pld < (int64_t)n2 * ld) return pt_bad_arg(9, "pitch");
    if (store_from < 0 || store_from > n1) return pt_bad_arg(11, "store_from outside 0 .. n1");
    PtAsm a;
    a.mom = mom; a.c1_lo = c1_lo; a.c1_hi = c1_hi;
    a.k2n = n2 == 1 ? 1 : p + 1;
    a.C2 = n2 == 1 ? 1 : n2 - p;
    a.C3 = n3 - p;
    a.y = y; a.ld = ld; a.pld = pld; a.n2 = n2; a.n3 = n3;
    a.r1_lo = c1_lo;
    a.store_from = store_from;
    a.count = (int64_t)(c1_hi - 1 + p + 1 - c1_lo) * n2 * n3;        // rows c1_lo .. c1_hi-1+p
    cudaStream_t st = (cudaStream_t)stream;
    switch (p) {
        case 1: return launch_assemble<1>(a, st);
        case 2: return launch_assemble<2>(a, st);
        case 3: return launch_assemble<3>(a, st);
        case 4: return launch_assemble<4>(a, st);
        default: return launch_assemble<5>(a, st);
    }
}
