// emu_points.cpp -- TEST INFRASTRUCTURE ONLY (see cuda_emu.h): runs the entry points of
// poms_b200/csrc/poms_points.cu, compiled for the host, on a problem read from a file.  Every array is copied
// into an exactly sized heap block, so that AddressSanitizer sees any access outside it.
//   emu_points <in> <out>
// in:  int32 header of 32 entries {op, n1, n2, n3, p, d, m, grad | chunk, ld}, then the arrays
//      (tests/test_points_host_emulation.py); n2 = 1 and d = 2: a 2-D space (no T2)
//   op 0 (poms_points_eval):  T1, [T2], T3, x (n1 n2 ld), pts (m d)      out: int32 status, u (m), [g (m d)]
//   op 1 (deposit, the sequence of poms_b200.fem.deposit with a stable sort on the host and chunks of `chunk`
//         cell planes):  T1, [T2], T3, pts (m d), w (m), y (n1 n2 ld)   out: int32 status, y
#define POMS_HOST_EMU 1
#include "../../poms_b200/csrc/poms_points.cu"

#include <algorithm>
#include <cstdlib>
#include <memory>
#include <numeric>

static FILE* g_in;
template <class T>
static std::unique_ptr<T[]> rd(size_t n) {
    std::unique_ptr<T[]> p(new T[n ? n : 1]);
    if (fread(p.get(), sizeof(T), n, g_in) != n) {
        fprintf(stderr, "short read\n");
        exit(3);
    }
    return p;
}

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    g_in = fopen(argv[1], "rb");
    if (!g_in) return 2;
    auto h = rd<int32_t>(32);
    FILE* o = fopen(argv[2], "wb");
    const int op = h[0], n1 = h[1], n2 = h[2], n3 = h[3], p = h[4], d = h[5], ld = h[8];
    const int64_t m = h[6];
    auto T1 = rd<double>(n1 + p + 1);
    std::unique_ptr<double[]> T2;
    if (d == 3) T2 = rd<double>(n2 + p + 1);
    auto T3 = rd<double>(n3 + p + 1);
    const int64_t ny = (int64_t)n1 * n2 * ld;
    int rc = 0;
    if (op == 0) {
        const int grad = h[7];
        auto x = rd<double>(ny);
        auto pts = rd<double>(m * d);
        std::unique_ptr<double[]> u(new double[m ? m : 1]), g(grad ? new double[m * d ? m * d : 1] : nullptr);
        rc = poms_points_eval(x.get(), ld, (int64_t)n2 * ld, n1, n2, n3, p, T1.get(), T2.get(), T3.get(), pts.get(),
                              d, m, u.get(), g.get(), nullptr);
        const int32_t rc32 = rc;
        fwrite(&rc32, 4, 1, o);
        fwrite(u.get(), 8, m, o);
        if (grad) fwrite(g.get(), 8, m * d, o);
    } else {
        const int chunk = h[7];
        auto pts = rd<double>(m * d);
        auto w = rd<double>(m);
        auto y = rd<double>(ny);
        const int C1 = n1 - p, C2 = d == 3 ? n2 - p : 1, C3 = n3 - p;
        const int nt = (p + 1) * (p + 1) * (d == 3 ? p + 1 : 1);
        std::unique_ptr<int64_t[]> key(new int64_t[m ? m : 1]), perm(new int64_t[m ? m : 1]);
        rc = poms_points_locate(pts.get(), d, m, n1, n2, n3, p, T1.get(), T2.get(), T3.get(), key.get(), nullptr);
        std::iota(perm.get(), perm.get() + m, (int64_t)0);
        std::stable_sort(perm.get(), perm.get() + m, [&](int64_t a, int64_t b) { return key[a] < key[b]; });
        std::vector<int64_t> skey(m);
        for (int64_t k = 0; k < m; ++k) skey[k] = key[perm[k]];
        for (int c0 = 0; rc == 0 && c0 < C1; c0 += chunk) {
            const int c1 = std::min(C1, c0 + chunk);
            const int64_t ncells = (int64_t)(c1 - c0) * C2 * C3;
            std::unique_ptr<int64_t[]> offs(new int64_t[ncells + 1]);
            for (int64_t l = 0; l <= ncells; ++l)
                offs[l] = std::lower_bound(skey.begin(), skey.end(), (int64_t)c0 * C2 * C3 + l) - skey.begin();
            std::unique_ptr<double[]> mom(new double[ncells * nt]);
            rc = poms_points_moments(pts.get(), w.get(), d, perm.get(), offs.get(), c0, c1, n1, n2, n3, p, T1.get(),
                                     T2.get(), T3.get(), mom.get(), nullptr);
            if (rc == 0)
                rc = poms_points_assemble(mom.get(), c0, c1, n1, n2, n3, p, y.get(), ld, (int64_t)n2 * ld,
                                          c0 == 0 ? 0 : c0 + p, nullptr);
        }
        const int32_t rc32 = rc;
        fwrite(&rc32, 4, 1, o);
        fwrite(y.get(), 8, ny, o);
    }
    if (rc != 0) fprintf(stderr, "status %d: %s\n", rc, g_err);
    fclose(g_in);
    fclose(o);
    return 0;
}
