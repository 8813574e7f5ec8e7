"""ctypes binding of libpnb200.so -- the C ABI declared in include/pnb200.h.

The CUDA library is the product: there is NO fallback.  If the shared object is missing or a call
fails, an exception is raised (PnbError carries pnb_last_error()).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libpnb200.so")

MAX_K = 8
MAX_SR = 128


class PnbError(RuntimeError):
    pass


class PnbOverflow(PnbError):
    """The shading workspace was smaller than the number of valid samples of a call (the extra samples were dropped)."""


class Grid(C.Structure):
    _fields_ = [("lo", C.c_float * 3), ("svs", C.c_float * 3), ("dim", C.c_int32 * 3), ("P", C.c_int32),
                ("parity_slot0", C.c_int32), ("n_points", C.c_int32), ("n_words", C.c_uint32),
                ("occ_bits", C.c_void_p), ("pt_bits", C.c_void_p), ("word_rank", C.c_void_p),
                ("cell_start", C.c_void_p), ("spts", C.c_void_p), ("counters", C.c_void_p)]


class Query(C.Structure):
    _fields_ = [("R", C.c_int32), ("SR", C.c_int32), ("K", C.c_int32), ("D", C.c_int32), ("cap_samples", C.c_int32),
                ("nsamp", C.c_void_p), ("samp_off", C.c_void_p), ("steps", C.c_void_p), ("samp_ray", C.c_void_p),
                ("cand_pidx", C.c_void_p), ("samp_nvalid", C.c_void_p), ("valid_list", C.c_void_p),
                ("valid_rank", C.c_void_p), ("ray_hit", C.c_void_p), ("ray_rank", C.c_void_p),
                ("scan_tmp", C.c_void_p), ("counters", C.c_void_p), ("raydir", C.c_void_p), ("t", C.c_void_p),
                ("t_ray_stride", C.c_int32), ("campos", C.c_float * 3)]


class ShadeOpts(C.Structure):
    _fields_ = [("campos", C.c_float * 3), ("camrotc2w", C.c_float * 9), ("Rw2c", C.c_float * 9),
                ("vsize_z", C.c_float), ("bg_color", C.c_float * 3), ("raydist_mode_unit", C.c_int32), ("agg_intrp_order", C.c_int32)]


class Mlp(C.Structure):
    _fields_ = [("w", C.c_void_p * 9), ("b", C.c_void_p * 9)]


class Points(C.Structure):
    _fields_ = [("xyz", C.c_void_p), ("emb", C.c_void_p), ("color", C.c_void_p), ("dir", C.c_void_p),
                ("conf", C.c_void_p), ("N", C.c_int32)]


GC = dict(n_occ=0, max_pts=1, overflow_o=2, overflow_p=3, n_inrange=4, slot0_cell=5, first_pt=6,
          box_x0=7, box_y0=8, box_z0=9, box_x1=10, box_y1=11, box_z1=12, sphere_r2=13)
QC = dict(n_cand=0, n_valid=1, n_pairs=2, R1=3, R2=4, overflow=5)

# every symbol include/pnb200.h declares (tests check that the .so exports all of them)
SYMBOLS = ["pnb_version", "pnb_last_error", "pnb_struct_size", "pnb_grid_bytes", "pnb_grid_build", "pnb_query_bytes", "pnb_query",
           "pnb_query_export", "pnb_shade_bytes", "pnb_shade_forward", "pnb_composite_forward",
           "pnb_mlp_pack_bytes", "pnb_mlp_pack", "pnb_point_pre_bytes", "pnb_point_pre", "pnb_shade_tc_bytes", "pnb_shade_forward_tc",
           "pnb_shade_tc_tables", "pnb_backward_bytes", "pnb_shade_backward", "pnb_aux_outputs", "pnb_aux_conf_backward",
           "pnb_probe_maps", "pnb_probe_select_bytes", "pnb_probe_select"]
# test-only library (csrc/selftest/pnb200_selftest.h)
SELFTEST_LIB_PATH = os.path.join(_HERE, "csrc", "libpnb200_selftest.so")
SELFTEST_SYMBOLS = ["pnb_selftest_last_error", "pnb_umma_selftest", "pnb_umma_bench", "pnb_umma_selftest2", "pnb_gemm_tc_test"]
# flags of pnb_shade_forward_tc
TC_PAIRS, TC_COLOR, TC_FROZEN, TC_DBG_NO_WEIGHTS = 1, 2, 4, 64
BWD_FP32_GEMM, BWD_FP32_RECOMPUTE = 1, 4   # flags of pnb_shade_backward

_lib = None
_selftest = None


def load():
    """Load the CUDA library or fail loudly (no CPU path exists in the product)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PnbError("libpnb200.so not found at %s -- run `python -m pointnerf_b200.build` (nvcc, sm_100a). "
                       "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.pnb_version.restype = C.c_int
    lib.pnb_last_error.restype = C.c_char_p
    lib.pnb_struct_size.restype = C.c_size_t
    lib.pnb_struct_size.argtypes = [C.c_int]
    for which, ty in enumerate((Grid, Query, ShadeOpts, Mlp, Points)):
        if lib.pnb_struct_size(which) != C.sizeof(ty):
            raise PnbError("ABI mismatch: struct %s is %d bytes in libpnb200.so, %d in the binding"
                           % (ty.__name__, lib.pnb_struct_size(which), C.sizeof(ty)))
    lib.pnb_grid_bytes.restype = C.c_size_t
    lib.pnb_grid_bytes.argtypes = [C.c_int, C.POINTER(C.c_int32)]
    lib.pnb_grid_build.restype = C.c_int
    lib.pnb_grid_build.argtypes = [C.POINTER(Grid), C.c_void_p, C.c_size_t, C.c_void_p, C.c_int,
                                   C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                   C.POINTER(C.c_int32)]
    lib.pnb_query_bytes.restype = C.c_size_t
    lib.pnb_query_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    lib.pnb_query.restype = C.c_int
    lib.pnb_query.argtypes = [C.POINTER(Query), C.c_void_p, C.c_size_t, C.POINTER(Grid), C.POINTER(C.c_float),
                              C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                              C.POINTER(C.c_int32), C.c_int, C.c_void_p, C.POINTER(C.c_int32)]
    lib.pnb_query_export.restype = C.c_int
    lib.pnb_query_export.argtypes = [C.POINTER(Query), C.POINTER(ShadeOpts), C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pnb_shade_bytes.restype = C.c_size_t
    lib.pnb_shade_bytes.argtypes = [C.c_int]
    lib.pnb_shade_forward.restype = C.c_int
    lib.pnb_shade_forward.argtypes = [C.POINTER(Query), C.POINTER(Points), C.POINTER(Mlp), C.POINTER(ShadeOpts),
                                      C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pnb_composite_forward.restype = C.c_int
    lib.pnb_composite_forward.argtypes = [C.POINTER(Query), C.POINTER(ShadeOpts), C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pnb_aux_outputs.restype = C.c_int
    lib.pnb_aux_outputs.argtypes = [C.POINTER(Query), C.POINTER(Points), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.pnb_aux_conf_backward.restype = C.c_int
    lib.pnb_aux_conf_backward.argtypes = [C.POINTER(Query), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pnb_probe_maps.restype = C.c_int
    lib.pnb_probe_maps.argtypes = [C.POINTER(Query), C.POINTER(Points), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pnb_probe_select_bytes.restype = C.c_size_t
    lib.pnb_probe_select_bytes.argtypes = [C.c_int, C.c_int]
    lib.pnb_probe_select.restype = C.c_int
    lib.pnb_probe_select.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 11 + [C.POINTER(C.c_float), C.c_float, C.c_float, C.c_void_p,
                                                                             C.c_size_t, C.c_int] + [C.c_void_p] * 7
    lib.pnb_mlp_pack_bytes.restype = C.c_size_t
    lib.pnb_mlp_pack_bytes.argtypes = []
    lib.pnb_mlp_pack.restype = C.c_int
    lib.pnb_mlp_pack.argtypes = [C.POINTER(Mlp), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pnb_point_pre_bytes.restype = C.c_size_t
    lib.pnb_point_pre_bytes.argtypes = [C.c_int]
    lib.pnb_point_pre.restype = C.c_int
    lib.pnb_point_pre.argtypes = [C.POINTER(Points), C.POINTER(Mlp), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.pnb_shade_tc_bytes.restype = C.c_size_t
    lib.pnb_shade_tc_bytes.argtypes = [C.c_int]
    lib.pnb_shade_forward_tc.restype = C.c_int
    lib.pnb_shade_forward_tc.argtypes = [C.POINTER(Query), C.POINTER(Points), C.POINTER(Mlp), C.c_void_p, C.c_void_p, C.POINTER(ShadeOpts),
                                         C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.pnb_shade_tc_tables.restype = C.c_int
    lib.pnb_shade_tc_tables.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    lib.pnb_backward_bytes.restype = C.c_size_t
    lib.pnb_backward_bytes.argtypes = [C.c_int, C.c_int]
    lib.pnb_shade_backward.restype = C.c_int
    lib.pnb_shade_backward.argtypes = [C.POINTER(Query), C.POINTER(Points), C.POINTER(Mlp), C.POINTER(ShadeOpts), C.c_void_p,
                                       C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def load_selftest():
    """Test-only library with the tcgen05 self-tests / micro-benchmarks (not part of the product ABI)."""
    global _selftest
    if _selftest is not None:
        return _selftest
    if not os.path.exists(SELFTEST_LIB_PATH):
        raise PnbError("libpnb200_selftest.so not found at %s -- run `python -m pointnerf_b200.build`" % SELFTEST_LIB_PATH)
    lib = C.CDLL(SELFTEST_LIB_PATH)
    lib.pnb_selftest_last_error.restype = C.c_char_p
    lib.pnb_umma_bench.restype = C.c_int
    lib.pnb_umma_bench.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pnb_umma_selftest2.restype = C.c_int
    lib.pnb_umma_selftest2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.pnb_umma_selftest.restype = C.c_int
    lib.pnb_umma_selftest.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.pnb_gemm_tc_test.restype = C.c_int
    lib.pnb_gemm_tc_test.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_void_p, C.c_long, C.c_long, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_int, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    _selftest = lib
    return lib


def check_selftest(rc, what=""):
    if rc != 0:
        raise PnbError("%s failed (status %d): %s" % (what, rc, load_selftest().pnb_selftest_last_error().decode()))


def check(rc, what=""):
    if rc != 0:
        raise PnbError("%s failed (status %d): %s" % (what, rc, load().pnb_last_error().decode()))


def f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def i3(v):
    return (C.c_int32 * 3)(*[int(x) for x in v])
