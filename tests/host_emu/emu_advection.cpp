// emu_advection.cpp -- TEST INFRASTRUCTURE ONLY (see cuda_emu.h): poms_assemble_1d_advection of poms_setup.cu
// (rewritten for g++ by make_emu_source.py into setup_emu.cuh) on exactly sized buffers.
//   emu_advection <in> <out>
// in:  int32 header (16): {n, p, 0...}, then knots (n+p+1), gauss_x (p+1), gauss_w (p+1), each as int64 length + data
// out: int32 status, then G (n * (2p+1))
#define POMS_HOST_EMU 1
#include "cuda_emu.h"
#include "poms_b200.h"
#include "setup_emu.cuh"

#include <cstdlib>

static double* read_arr(FILE* f, int64_t expect) {
    int64_t len;
    if (fread(&len, 8, 1, f) != 1 || len != expect) exit(3);
    double* a = new double[len];                   // exactly sized: the sanitizer sees every overrun
    if (fread(a, 8, len, f) != (size_t)len) exit(3);
    return a;
}

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    int32_t h[16];
    if (fread(h, 4, 16, f) != 16) return 3;
    const int n = h[0], p = h[1];
    double* T = read_arr(f, n + p + 1);
    double* gx = read_arr(f, p + 1);
    double* gw = read_arr(f, p + 1);
    const size_t len = (size_t)n * (2 * p + 1);
    double* G = new double[len];
    const int32_t rc = poms_assemble_1d_advection(T, n, p, gx, gw, G, nullptr);
    FILE* o = fopen(argv[2], "wb");
    fwrite(&rc, 4, 1, o);
    if (rc == 0) fwrite(G, 8, len, o);
    else fprintf(stderr, "status %d: %s\n", rc, g_err);
    delete[] T; delete[] gx; delete[] gw; delete[] G;
    fclose(f);
    fclose(o);
    return 0;
}
