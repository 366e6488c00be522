"""poms_b200 -- B200-native (sm_100a) implementation of the POMS multigrid solve path.

Module names mirror the reference's `sources/` directory so that
`from poms_b200.kron_product import kron_dot_v2` etc. read like the originals:

    kron_product  kron_dot_v1/v2, kron_solve_serial/par/bnd_par, to_bnd (+ 3-D variants)
    solvers       crl, pcg, jacobi, damped_jacobi, pcg_glt
    multilevels   knots_to_insert
    mg_jac/mg_glt the two-grid scripts as functions
    utils         populate_*, array_to_vect_stencil, array_to_mat_stencil
    stencil       StencilVectorSpace / StencilVector / StencilMatrix (spl-compatible, on device),
                  KronSumMatrix
    mg            Transfer, CoarseSolver, two_grid; EXTENSION: Hierarchy, vcycle, mg_pcg
    dist          slab partition along axis 1, halo exchange, all-reduce (NCCL)
    fem           EXTENSION: load_vector (b_i = int f phi_i), error_norms (L2 / H1), evaluate

All arithmetic runs in hand-written CUDA kernels (csrc/poms_kernels.cu) behind the C ABI of
include/poms_b200.h; there is no CPU fallback.
"""
__version__ = "0.1.0"
