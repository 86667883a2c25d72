"""Loader of the in-tree CUDA library (topay_b200/libtopay_b200.so) and its C-ABI prototypes.

The library is the product: there is no Python/NumPy fallback. Import works without a GPU (so
that the ABI can be inspected on a CPU box) but every compute entry point returns
TOPAY_ERR_NO_DEVICE there and the wrappers raise.
"""
import ctypes as C
import os
import subprocess

from ._structs import Feasibility, GridDesc, ProbDesc, RogDesc, TrajBatch, OptParams, ProblemBatch, ResultBatch, RobotParams, SolverStats

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("TOPAY_B200_LIB", os.path.join(_HERE, "libtopay_b200.so"))

OK, ERR_INVALID_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_ALLOC, ERR_TOO_LARGE, ERR_NOT_READY = 0, -1, -2, -3, -4, -5, -6


class TopayError(RuntimeError):
    def __init__(self, code, what, detail):
        super().__init__(f"{what}: {detail} (code {code})")
        self.code = code


def build(verbose=False):
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc")]
    out = subprocess.run(cmd, capture_output=not verbose, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libtopay_b200.so failed:\n" + (out.stdout or "") + (out.stderr or ""))
    return SO_PATH


_lib = None
_dp, _ip, _i8p, _fp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int8), C.POINTER(C.c_float)
_i16p, _u8p = C.POINTER(C.c_int16), C.POINTER(C.c_uint8)

# name -> (restype, argtypes); every symbol include/topay_b200.h declares
PROTOTYPES = {
    "topay_strerror": (C.c_char_p, [C.c_int]),
    "topay_last_error": (C.c_char_p, []),
    "topay_version": (C.c_char_p, []),
    "topay_robot_params_default": (None, [C.POINTER(RobotParams)]),
    "topay_opt_params_default": (None, [C.POINTER(OptParams)]),
    "topay_field_create": (C.c_int, [C.POINTER(GridDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "topay_field_destroy": (None, [C.c_void_p]),
    "topay_field_dims": (C.c_int, [C.c_void_p, _ip]),
    "topay_field_set_occupancy": (C.c_int, [C.c_void_p, _i8p, _i8p, _i8p]),
    "topay_field_clear": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_field_rasterize_points": (C.c_int, [C.c_void_p, _fp, C.c_int64]),
    "topay_field_rebuild": (C.c_int, [C.c_void_p]),
    "topay_field_query3d": (C.c_int, [C.c_void_p, _dp, C.c_int64, _dp, _dp]),
    "topay_field_query2d": (C.c_int, [C.c_void_p, _dp, C.c_int64, C.c_int, _dp, _dp]),
    "topay_field_distance3d": (C.c_int, [C.c_void_p, _dp, C.c_int64, _dp]),
    "topay_field_distance2d": (C.c_int, [C.c_void_p, _dp, C.c_int64, _dp]),
    "topay_field_whole_body_collision": (C.c_int, [C.c_void_p, C.POINTER(RobotParams), _dp, C.c_int64, _i8p]),
    "topay_field_is_collision2d": (C.c_int, [C.c_void_p, _dp, C.c_int64, C.c_double, _i8p]),
    "topay_field_is_collision3d": (C.c_int, [C.c_void_p, _dp, C.c_int64, C.c_double, _i8p]),
    "topay_field_is_line_collision_grid2d": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int64, C.c_double, _i8p]),
    "topay_field_dist_coarse2d": (C.c_int, [C.c_void_p, _dp, C.c_int64, C.c_int, _dp]),
    "topay_field_line_visible": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int64, C.c_double, C.c_int, _i8p, _dp]),
    "topay_field_same_topo_paths": (C.c_int, [C.c_void_p, _dp, _ip, C.c_int, _ip, C.c_int, C.c_double, C.c_int, _i8p]),
    "topay_path_length": (C.c_double, [_dp, C.c_int]),
    "topay_discretize_path": (C.c_int, [_dp, C.c_int, C.c_int, _dp]),
    "topay_dense_path": (C.c_int, [_dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _dp,
                                   C.c_int]),
    "topay_field_dist_coarse2i": (C.c_int, [C.c_void_p, _ip, C.c_int64, C.c_int, _dp]),
    "topay_field_query3d_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "topay_field_sync": (C.c_int, [C.c_void_p]),
    "topay_field_download": (C.c_int, [C.c_void_p, C.c_int, _dp]),
    "topay_field_download_sqdist": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip]),
    "topay_field_download_occupancy": (C.c_int, [C.c_void_p, C.c_int, _i8p]),
    "topay_field_set_keep_sqdist": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_field_last_rebuild_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "topay_rogfield_create": (C.c_int, [C.POINTER(RogDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "topay_rogfield_destroy": (None, [C.c_void_p]),
    "topay_rogfield_geometry": (C.c_int, [C.c_void_p, _ip, _ip, _dp, _ip, _ip]),
    "topay_rogfield_slide": (C.c_int, [C.c_void_p, _dp]),
    "topay_rogfield_update_counters": (C.c_int, [C.c_void_p, _dp, _u8p, _u8p, C.c_int64]),
    "topay_rogfield_set_occupied_cnt": (C.c_int, [C.c_void_p, _i16p]),
    "topay_rogfield_download_counters": (C.c_int, [C.c_void_p, _i16p, _i16p]),
    "topay_rogfield_update_esdf": (C.c_int, [C.c_void_p, _dp]),
    "topay_rogfield_query": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_int64, _dp, _dp]),
    "topay_rogfield_is_line_free2d": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int64, C.c_double, _i8p]),
    "topay_rogfield_download": (C.c_int, [C.c_void_p, C.c_int, _dp]),
    "topay_rogfield_last_update_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "topay_probmap_create": (C.c_int, [C.c_void_p, C.POINTER(ProbDesc), C.POINTER(C.c_void_p)]),
    "topay_probmap_destroy": (None, [C.c_void_p]),
    "topay_probmap_update": (C.c_int, [C.c_void_p, _fp, C.c_int64, _dp]),
    "topay_probmap_download": (C.c_int, [C.c_void_p, _fp, _ip]),
    "topay_probmap_set_first_frame": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_traj_check_feasible": (C.c_int, [C.c_void_p, C.POINTER(RobotParams), C.POINTER(TrajBatch),
                                            C.POINTER(Feasibility)]),
    "topay_traj_check_feasible_rog": (C.c_int, [C.c_void_p, C.POINTER(RobotParams), C.POINTER(TrajBatch),
                                                C.POINTER(Feasibility)]),
    "topay_traj_car_seq": (C.c_int, [C.c_int, C.POINTER(TrajBatch), C.c_int, _dp, _ip]),
    "topay_traj_sample": (C.c_int, [C.c_int, C.POINTER(TrajBatch), _dp, C.c_int, _dp, _dp]),
    "topay_select_shortest": (C.c_int, [_ip, _dp, C.c_int]),
    "topay_solver_check_feasible": (C.c_int, [C.c_void_p, C.POINTER(Feasibility), _ip]),
    "topay_solver_select": (C.c_int, [C.c_void_p, C.c_int, _ip, C.c_int, _ip, _ip]),
    "topay_solver_download_candidate": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ResultBatch)]),
    "topay_solver_create": (C.c_int, [C.POINTER(OptParams), C.POINTER(RobotParams), C.c_void_p, C.c_int, C.c_int,
                                      C.POINTER(C.c_void_p)]),
    "topay_solver_create_rog": (C.c_int, [C.POINTER(OptParams), C.POINTER(RobotParams), C.c_void_p, C.c_int, C.c_int,
                                          C.POINTER(C.c_void_p)]),
    "topay_solver_create_pool": (C.c_int, [C.POINTER(OptParams), C.POINTER(RobotParams), C.c_void_p, C.c_int, C.c_int,
                                           C.c_int, C.POINTER(C.c_void_p)]),
    "topay_solver_destroy": (None, [C.c_void_p]),
    "topay_solver_eval": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ProblemBatch), _dp, C.c_int, _dp, _dp, _dp, _dp,
                                    _dp]),
    "topay_prepare_candidate": (C.c_int, [C.POINTER(OptParams), C.POINTER(RobotParams), _dp, C.c_int, _dp, _dp,
                                          C.c_int, _ip, _dp, _dp, _dp, _dp, _dp, _dp, _ip]),
    "topay_solver_solve_batch": (C.c_int, [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp, C.POINTER(ResultBatch), _ip,
                                           _ip]),
    "topay_solver_upload": (C.c_int, [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp]),
    "topay_solver_run": (C.c_int, [C.c_void_p]),
    "topay_solver_assign_fields": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, _ip]),
    "topay_solver_set_plans": (C.c_int, [C.c_void_p, C.c_int, _ip, C.c_int, C.c_int32]),
    "topay_solver_download": (C.c_int, [C.c_void_p, C.POINTER(ResultBatch), _ip, _ip]),
    "topay_solver_set_trace": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_solver_download_trace": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_int, _ip]),
    "topay_solver_debug_download": (C.c_int64, [C.c_void_p, C.c_int, _dp, C.c_int64]),
    "topay_solver_debug_direction": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                               _dp, _ip, _ip]),
    "topay_solver_phase_clocks": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_longlong)]),
    "topay_solver_stream_begin": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_solver_stream_submit": (C.c_int, [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp, C.c_void_p, _ip]),
    "topay_solver_stream_advance": (C.c_int, [C.c_void_p, C.c_int, _ip]),
    "topay_solver_stream_poll": (C.c_int, [C.c_void_p, C.c_int, _ip, _ip, _ip]),
    "topay_solver_stream_take": (C.c_int, [C.c_void_p, C.c_int32, C.c_int, C.POINTER(ResultBatch),
                                           C.POINTER(Feasibility)]),
    "topay_solver_stream_set_grace": (C.c_int, [C.c_void_p, C.c_int32]),
    "topay_solver_stream_stop": (C.c_int, [C.c_void_p, C.c_int32]),
    "topay_solver_stream_set_snapshots": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_solver_stream_end": (C.c_int, [C.c_void_p]),
    "topay_solver_set_timed": (C.c_int, [C.c_void_p, C.c_int]),
    "topay_solver_last_stats": (C.c_int, [C.c_void_p, C.POINTER(SolverStats)]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        _lib = C.CDLL(SO_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(_lib, name)
            fn.restype, fn.argtypes = res, args
    return _lib


def check(code, what):
    if code != OK:
        l = lib()
        raise TopayError(code, what, (l.topay_last_error() or l.topay_strerror(code)).decode())
