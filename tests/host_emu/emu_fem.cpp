// emu_fem.cpp -- TEST INFRASTRUCTURE ONLY (see cuda_emu.h): runs poms_quad_to_coef_3d / poms_quad_error_3d of
// poms_b200/csrc/poms_fem3d.cu, compiled for the host, on a problem read from a file.  Every array is copied
// into an exactly sized heap block, so that AddressSanitizer sees any access outside it.
//   emu_fem <in> <out>
// in:  int32 header of 32 entries, then the arrays (tests/test_fem_host_emulation.py, _run_q2c / _run_err).
//   op 0: {0, n1, n2, n3, m2, m3, p, e1_lo, e1_hi, k1n, q1n, store_from, w2, ne3, nq1, E1, fld, fpld, ld}
//         s1 (E1), b1 (E1 k1n q1n), st2 (n2), c2 (n2 w2), e3 (n3), c3 (n3 (p+1)^2), F (nq1 fpld), y (n1 n2 ld)
//         out: int32 status, y
//   op 1: {1, n1, n2, n3, m2, m3, p, j1_lo, nq1, k1n, k2n, m1, grad, ld, has[4], rld[4], rpld[4]}
//         x (n1 n2 ld), s1 v1 d1 w1 (m1, m1 k1n, m1 k1n, m1), s2 v2 d2 w2 (axis 2, k2n), s3 v3 d3 w3 (axis 3,
//         p+1), the present reference arrays (nq1 rpld each), out (2)
//         out: int32 status, out (2)
#define POMS_HOST_EMU 1
#include "../../poms_b200/csrc/poms_fem3d.cu"

#include <cstdlib>
#include <memory>

static FILE* g_in;
template <class T>
static std::unique_ptr<T[]> rd(size_t n) {
    std::unique_ptr<T[]> p(new T[n]);
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
    int rc;
    if (h[0] == 0) {
        const int n1 = h[1], n2 = h[2], n3 = h[3], m2 = h[4], m3 = h[5], p = h[6], e1_lo = h[7], e1_hi = h[8];
        const int k1n = h[9], q1n = h[10], store_from = h[11], w2 = h[12], ne3 = h[13], nq1 = h[14], E1 = h[15];
        const int fld = h[16], fpld = h[17], ld = h[18];
        auto s1 = rd<int32_t>(E1);
        auto b1 = rd<double>((size_t)E1 * k1n * q1n);
        auto st2 = rd<int32_t>(n2);
        auto c2 = rd<double>((size_t)n2 * w2);
        auto e3 = rd<int32_t>(n3);
        auto c3 = rd<double>((size_t)n3 * (p + 1) * (p + 1));
        auto F = rd<double>((size_t)nq1 * fpld);
        auto y = rd<double>((size_t)n1 * n2 * ld);
        rc = poms_quad_to_coef_3d(F.get(), fld, fpld, y.get(), ld, (int64_t)n2 * ld, n1, n2, n3, m2, m3, p, e1_lo,
                                  e1_hi, k1n, q1n, s1.get(), b1.get(), store_from, st2.get(), c2.get(), w2, e3.get(),
                                  c3.get(), ne3, s1.get(), st2.get(), e3.get(), nullptr);
        const int32_t rc32 = rc;
        fwrite(&rc32, 4, 1, o);
        fwrite(y.get(), 8, (size_t)n1 * n2 * ld, o);
    } else {
        const int n1 = h[1], n2 = h[2], n3 = h[3], m2 = h[4], m3 = h[5], p = h[6], j1_lo = h[7], nq1 = h[8];
        const int k1n = h[9], k2n = h[10], m1 = h[11], grad = h[12], ld = h[13];
        auto x = rd<double>((size_t)n1 * n2 * ld);
        auto s1 = rd<int32_t>(m1);
        auto v1 = rd<double>((size_t)m1 * k1n);
        auto d1 = rd<double>((size_t)m1 * k1n);
        auto w1 = rd<double>(m1);
        auto s2 = rd<int32_t>(m2);
        auto v2 = rd<double>((size_t)m2 * k2n);
        auto d2 = rd<double>((size_t)m2 * k2n);
        auto w2 = rd<double>(m2);
        auto s3 = rd<int32_t>(m3);
        auto v3 = rd<double>((size_t)m3 * (p + 1));
        auto d3 = rd<double>((size_t)m3 * (p + 1));
        auto w3 = rd<double>(m3);
        std::unique_ptr<double[]> refs[4];
        const double* ref[4];
        int64_t rld[4], rpld[4];
        for (int c = 0; c < 4; ++c) {
            rld[c] = h[18 + c];
            rpld[c] = h[22 + c];
            if (h[14 + c]) refs[c] = rd<double>((size_t)nq1 * rpld[c]);
            ref[c] = refs[c].get();
        }
        auto out = rd<double>(2);
        std::unique_ptr<unsigned char[]> ws(new unsigned char[256 + 65536 * 8]());
        rc = poms_quad_error_3d(x.get(), ld, (int64_t)n2 * ld, n1, n2, n3, m2, m3, p, ref, rld, rpld, j1_lo, nq1, k1n,
                                s1.get(), v1.get(), d1.get(), w1.get(), k2n, s2.get(), v2.get(), d2.get(), w2.get(),
                                s3.get(), v3.get(), d3.get(), w3.get(), s1.get(), s2.get(), s3.get(), m1, grad,
                                j1_lo > 0, out.get(), ws.get(), nullptr);
        const int32_t rc32 = rc;
        fwrite(&rc32, 4, 1, o);
        fwrite(out.get(), 8, 2, o);
    }
    if (rc != 0) fprintf(stderr, "status %d: %s\n", rc, g_err);
    fclose(g_in);
    fclose(o);
    return 0;
}
