"""ctypes binding of libpoms_b200.so (include/poms_b200.h).  There is NO fallback: if the
shared library is missing or a call fails, the product raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POMS_B200_LIB", os.path.join(HERE, "libpoms_b200.so"))

_vp, _i, _l, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double

_PROTOS = {
    "poms_version": (C.c_int, []),
    "poms_workspace_bytes": (_l, []),
    "poms_last_error": (C.c_char_p, []),
    "poms_launch_count": (_l, []),
    "poms_launch_count_add": (None, [_l]),
    "poms_kron_matvec_2d": (C.c_int, [_vp, _vp, _vp, _i, _i, _l, _i, _i, _i, _i,
                                     _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp]),
    "poms_kron_matvec_2d_ex": (C.c_int, [_vp, _vp, _vp, _i, _i, _l, _i, _i, _i, _i,
                                        _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _vp]),
    "poms_set_matvec2d_variant": (None, [_i]),
    "poms_kron_matvec_3d": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _i,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp]),
    "poms_kron_matvec_3d_ex": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _i,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp,
                                        _vp, _vp]),
    "poms_kron_matvec_3d_dotv": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _i,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp,
                                          _vp, _vp, _vp, C.POINTER(C.c_int)]),
    "poms_set_force_generic": (None, [_i]),
    "poms_set_matvec3d_chunk": (None, [_i]),
    "poms_set_matvec3d_variant": (None, [_i]),
    "poms_stencil_matvec_2d": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _l, _i, _i, _i, _i,
                                        _i, _d, _vp, _vp, _vp]),
    "poms_cg_update": (C.c_int, [_vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _vp, _vp]),
    "poms_p_update": (C.c_int, [_vp, _vp, _l, _vp, _vp, _vp]),
    "poms_dot": (C.c_int, [_vp, _vp, _l, _vp, _vp, _vp]),
    "poms_axpby": (C.c_int, [_vp, _d, _vp, _d, _vp, _l, _vp]),
    "poms_axpy_dev": (C.c_int, [_vp, _vp, _l, _vp, _vp, _d, _vp]),
    "poms_jacobi_first_2d": (C.c_int, [_vp, _vp, _i, _i, _l, _i, _i, _vp, _vp, _vp, _vp,
                                      _d, _vp, _vp, _vp]),
    "poms_jacobi_first_3d": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i,
                                      _vp, _vp, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp]),
    "poms_cheb_update": (C.c_int, [_vp, _vp, _vp, _d, _d, _l, _vp]),
    "poms_diag_scale": (C.c_int, [_vp, _vp, _vp, _l, _d, _vp, _vp, _vp]),
    "poms_band_solve_axis": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _l, _l, _l, _l, _vp]),
    "poms_band_solve_axis_chunked": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _l, _l, _l, _l,
                                              _i, _i, _i, _vp]),
    "poms_band_solve_axis_fused": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _l, _l, _d, _vp, _vp, _vp]),
    "poms_axis_gather": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _l, _l, _l, _l, _l, _l,
                                  _i, _vp]),
    "poms_dense_matvec": (C.c_int, [_vp, _vp, _vp, _i, _vp]),
    "poms_restrict_3d": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _l, _l,
                                  _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "poms_prolong_3d": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _l, _l,
                                 _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "poms_restrict_3d_v2": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _l, _l,
                                     _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "poms_prolong_3d_v2": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _l, _l,
                                    _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "poms_stencil_matvec_3d": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _l, _l, _i, _i, _i, _i, _i,
                                        _i, _d, _vp, _vp, _vp]),
    "poms_color_add": (C.c_int, [_vp, _vp, _i, _i, _i, _l, _l, _i, _i, _vp]),
    "poms_assemble_1d": (C.c_int, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "poms_knot_insertion_rows": (C.c_int, [_vp, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "poms_band_lu_nopiv": (C.c_int, [_vp, _i, _i, _vp, _vp, _vp]),
    "poms_axis_dense_dmma": (C.c_int, [_vp, _vp, _vp, _i, _i, _l, _l, _l, _l, _l, _l, _vp]),
    "poms_quad_to_coef_3d": (C.c_int, [_vp, _l, _l, _vp, _l, _l, _i, _i, _i, _i, _i, _i, _i, _i, _i,
                                      _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "poms_quad_error_3d": (C.c_int, [_vp, _l, _l, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _i,
                                    _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                    _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "poms_ipc_alloc": (C.c_int, [_l, C.POINTER(C.c_void_p)]),
    "poms_ipc_free": (C.c_int, [_vp]),
    "poms_ipc_handle_bytes": (C.c_int, []),
    "poms_ipc_get_handle": (C.c_int, [_vp, C.c_char_p]),
    "poms_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "poms_ipc_close": (C.c_int, [_vp]),
    "poms_halo_flags_bytes": (C.c_int, []),
    "poms_halo_exchange_p2p": (C.c_int, [_vp, _vp, _vp, _vp, _l, _vp, _vp, _vp, _vp]),
}

EXPORTS = tuple(_PROTOS)


class PomsError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library (once).  Raises if it has not been built: no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PomsError(
                "libpoms_b200.so not found at %s -- run `python -m poms_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().poms_last_error().decode()
        raise PomsError("%s failed with status %d: %s" % (what or "libpoms_b200 call", rc, msg))
