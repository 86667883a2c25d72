"""ctypes mirrors of the C structs in include/topay_b200.h (field order must match)."""
import ctypes as C

import numpy as np

DOF, DIM, NSPHERE, NTERMS = 7, 9, 12, 13
TERM_NAMES = ["jerk", "time", "chassis_colli", "moment", "acc", "domega", "mani_colli",
              "self_colli", "mani_pos", "mani_vel", "mani_acc", "mean_time", "endp"]
MAP2D_FLAT, MAP2D_INFLATE, MAP2D_CRITICAL, MAP3D = 0, 1, 2, 3
LBFGSERR_TICK_CAP = -2000      # TOPAY_LBFGSERR_TICK_CAP: stopped by the solver's hard cap on ticks
LBFGSERR_PLAN_GRACE = -2001    # TOPAY_LBFGSERR_PLAN_GRACE: cancelled by its plan's first success + grace


class RobotParams(C.Structure):
    _fields_ = [
        ("chassis_height", C.c_double), ("chassis_colli_radius", C.c_double),
        ("max_v", C.c_double), ("max_a", C.c_double), ("max_w", C.c_double), ("max_dw", C.c_double),
        ("colli_length", C.c_double * (DOF + 1)),
        ("colli_points", C.c_double * (2 * (DOF + 1))),
        ("colli_point_radius", C.c_double * (2 * (DOF + 1))),
        ("joint_pos_limit_max", C.c_double * DOF),
        ("joint_vel_limit", C.c_double * DOF),
        ("joint_acc_limit", C.c_double * DOF),
        ("relative_R", C.c_double * 9),
        ("relative_t", C.c_double * 3),
        ("collision_matrix", C.c_int32 * (NSPHERE * NSPHERE)),
    ]


class LbfgsParams(C.Structure):
    _fields_ = [
        ("mem_size", C.c_int32), ("g_epsilon", C.c_double), ("past", C.c_int32), ("delta", C.c_double),
        ("max_iterations", C.c_int32), ("max_linesearch", C.c_int32),
        ("min_step", C.c_double), ("max_step", C.c_double),
        ("f_dec_coeff", C.c_double), ("s_curv_coeff", C.c_double),
        ("cautious_factor", C.c_double), ("machine_prec", C.c_double),
    ]


class OptParams(C.Structure):
    _fields_ = [
        ("int_K", C.c_int32), ("min_piece_num", C.c_int32), ("relu_mu", C.c_double),
        ("sample_interval", C.c_double), ("energy_weights", C.c_double * DIM),
        ("s1_time_weight", C.c_double), ("s1_moment_weight", C.c_double), ("s1_acc_weight", C.c_double),
        ("s1_domega_weight", C.c_double), ("s1_mean_time_weight", C.c_double),
        ("s1_path_pos_weight", C.c_double),
        ("s1_lbfgs_normal_past", C.c_int32), ("s1_lbfgs_shot_path_past", C.c_int32),
        ("s1_shot_path_horizon", C.c_double), ("s1_lbfgs", LbfgsParams),
        ("s2_time_weight", C.c_double), ("s2_moment_weight", C.c_double), ("s2_acc_weight", C.c_double),
        ("s2_domega_weight", C.c_double), ("s2_collision_weight", C.c_double),
        ("s2_mani_colli_weight", C.c_double), ("s2_self_colli_weight", C.c_double),
        ("s2_mani_pos_weight", C.c_double), ("s2_mani_vel_weight", C.c_double),
        ("s2_mani_acc_weight", C.c_double), ("s2_mean_time_weight", C.c_double),
        ("s2_lbfgs", LbfgsParams),
        ("alm_init_lambda", C.c_double * 2), ("alm_init_rho", C.c_double * 2),
        ("alm_rho_max", C.c_double * 2), ("alm_gamma", C.c_double * 2),
        ("alm_tolerance", C.c_double), ("alm_max_rounds", C.c_int32),
    ]


class GridDesc(C.Structure):
    _fields_ = [("map_size", C.c_double * 3), ("resolution", C.c_double),
                ("chassis_colli_radius", C.c_double), ("chassis_height", C.c_double)]


def grid_desc(map_size=(20.0, 20.0, 1.6), resolution=0.1, chassis_colli_radius=0.4, chassis_height=0.155):
    """Defaults are src/planner/params/grid_map.yaml of the reference."""
    d = GridDesc()
    d.map_size[:] = map_size
    d.resolution = resolution
    d.chassis_colli_radius = chassis_colli_radius
    d.chassis_height = chassis_height
    return d


class RogDesc(C.Structure):
    _fields_ = [("half_prob_map_size_i", C.c_int32 * 3), ("prob_resolution", C.c_double),
                ("esdf_resolution", C.c_double), ("local_update_box", C.c_double * 3),
                ("map_sliding_en", C.c_int32), ("fix_map_origin", C.c_double * 3), ("unk_thresh", C.c_double)]


def rog_desc(half_prob_map_size_i=(400, 400, 40), prob_resolution=0.05, esdf_resolution=0.05,
             local_update_box=(40.0, 40.0, 4.0), map_sliding_en=False, fix_map_origin=(0.0, 0.0, 0.0),
             unk_thresh=0.7):
    """Arguments of ESDFMap::initESDFMap (esdf_map.cpp:28-57); the defaults give the 803x803x83 ring of
    SURVEY.md §8 row a23 (map 40x40x4 m at 0.05 m)."""
    d = RogDesc()
    d.half_prob_map_size_i[:] = half_prob_map_size_i
    d.prob_resolution = prob_resolution
    d.esdf_resolution = esdf_resolution
    d.local_update_box[:] = local_update_box
    d.map_sliding_en = int(map_sliding_en)
    d.fix_map_origin[:] = fix_map_origin
    d.unk_thresh = unk_thresh
    return d


class ProbDesc(C.Structure):
    _fields_ = [("p_hit", C.c_float), ("p_miss", C.c_float), ("p_min", C.c_float), ("p_max", C.c_float),
                ("p_occ", C.c_float), ("p_free", C.c_float), ("raycast_range_min", C.c_double),
                ("raycast_range_max", C.c_double), ("virtual_ceil_height", C.c_double),
                ("virtual_ground_height", C.c_double), ("inflation_resolution", C.c_double),
                ("inflation_step", C.c_int32), ("pad_", C.c_int32), ("local_update_box", C.c_double * 3),
                ("map_sliding_thresh", C.c_double), ("point_filt_num", C.c_int32), ("batch_update_size", C.c_int32),
                ("intensity_thresh", C.c_int32), ("raycasting_en", C.c_int32)]


def prob_desc(p_hit=0.70, p_miss=0.35, p_min=0.12, p_max=0.97, p_occ=0.80, p_free=0.30, ray_range=(0.3, 10.0),
              virtual_ceil_height=3.0, virtual_ground_height=-0.5, local_update_box=(20.0, 20.0, 4.0),
              map_sliding_thresh=0.2, point_filt_num=1, batch_update_size=1, intensity_thresh=-1, raycasting_en=True,
              inflation_resolution=0.05, inflation_step=1):
    """Parameters of rog_map::ProbMap (rog_map_core/config.hpp:160-262); p_* are probabilities, the log-odds are
    logit() in float as config.hpp:229-235."""
    d = ProbDesc()
    d.p_hit, d.p_miss, d.p_min, d.p_max, d.p_occ, d.p_free = p_hit, p_miss, p_min, p_max, p_occ, p_free
    d.raycast_range_min, d.raycast_range_max = ray_range
    d.virtual_ceil_height, d.virtual_ground_height = virtual_ceil_height, virtual_ground_height
    d.inflation_resolution, d.inflation_step = inflation_resolution, inflation_step
    d.local_update_box[:] = local_update_box
    d.map_sliding_thresh = map_sliding_thresh
    d.point_filt_num, d.batch_update_size = point_filt_num, batch_update_size
    d.intensity_thresh, d.raycasting_en = intensity_thresh, int(raycasting_en)
    return d


class ProblemBatch(C.Structure):
    _fields_ = [("n_cand", C.c_int32), ("piece_num", C.POINTER(C.c_int32)),
                ("head_pva", C.POINTER(C.c_double)), ("tail_pva", C.POINTER(C.c_double)),
                ("start_xy", C.POINTER(C.c_double)), ("end_xy", C.POINTER(C.c_double)),
                ("init_inner_xy", C.POINTER(C.c_double)),
                ("alm_lambda", C.POINTER(C.c_double)), ("alm_rho", C.POINTER(C.c_double))]


class ResultBatch(C.Structure):
    _fields_ = [("status", C.POINTER(C.c_int32)), ("lbfgs_code", C.POINTER(C.c_int32)),
                ("piece_num", C.POINTER(C.c_int32)), ("iters", C.POINTER(C.c_int32)),
                ("evals", C.POINTER(C.c_int32)), ("alm_rounds", C.POINTER(C.c_int32)),
                ("cost", C.POINTER(C.c_double)), ("duration", C.POINTER(C.c_double)),
                ("T", C.POINTER(C.c_double)), ("coeff", C.POINTER(C.c_double)),
                ("final_xy_err", C.POINTER(C.c_double)), ("x", C.POINTER(C.c_double))]


class TrajBatch(C.Structure):
    _fields_ = [("n_traj", C.c_int32), ("max_pieces", C.c_int32), ("piece_num", C.POINTER(C.c_int32)),
                ("T", C.POINTER(C.c_double)), ("coeff", C.POINTER(C.c_double)), ("start_se2", C.POINTER(C.c_double))]


FEAS_FIELDS = (("feasible", np.int32, ()), ("feasible_print", np.int32, ()), ("n_samples", np.int32, ()),
               ("max_vel", np.float64, ()), ("max_acc", np.float64, ()), ("max_domega", np.float64, ()),
               ("max_d2omega", np.float64, ()), ("max_q", np.float64, (7,)), ("max_dq", np.float64, (7,)),
               ("max_d2q", np.float64, (7,)), ("min_dist", np.float64, ()), ("min_dist_mani", np.float64, (12,)))


class Feasibility(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_int32 if t is np.int32 else C.c_double)) for n, t, _ in FEAS_FIELDS]


def pack_trajs(trajs):
    """[(durations[N], coeff[6N][9], start_se2[3]), ...] -> (TrajBatch, keep-alive arrays)."""
    n = len(trajs)
    pn = np.array([len(t[0]) for t in trajs], dtype=np.int32)
    NP = int(pn.max()) if n else 1
    T = np.zeros((n, NP))
    cf = np.zeros((n, 6 * NP, 9))
    st = np.zeros((n, 3))
    for i, (d, c, s0) in enumerate(trajs):
        T[i, :pn[i]] = d
        cf[i, :6 * pn[i]] = np.asarray(c).reshape(6 * pn[i], 9)
        st[i] = np.asarray(s0)[:3]
    keep = (pn, T, cf, st)
    tb = TrajBatch(n, NP, pn.ctypes.data_as(C.POINTER(C.c_int32)), T.ctypes.data_as(C.POINTER(C.c_double)),
                   cf.ctypes.data_as(C.POINTER(C.c_double)), st.ctypes.data_as(C.POINTER(C.c_double)))
    return tb, keep


def alloc_feasibility(n, verdicts_only=False):
    """(Feasibility, dict of numpy arrays it points to). verdicts_only: just the two verdicts, every metric
    pointer NULL (the library skips what it is not asked for)."""
    want = [(name, t, shape) for name, t, shape in FEAS_FIELDS
            if not verdicts_only or name in ("feasible", "feasible_print")]
    arrs = {name: np.zeros((n,) + shape, dtype=t) for name, t, shape in want}
    f = Feasibility(*[arrs[name].ctypes.data_as(C.POINTER(C.c_int32 if t is np.int32 else C.c_double))
                      if name in arrs else None for name, t, _ in FEAS_FIELDS])
    return f, arrs


class SolverStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("ticks", C.c_int64), ("evals_total", C.c_int64),
                ("ms_total", C.c_float), ("ms_eval", C.c_float), ("eval_launches", C.c_int64),
                ("eval_nodes", C.c_int64), ("ms_integrate", C.c_float), ("ms_chain", C.c_float), ("ms_cand", C.c_float),
                ("pad_", C.c_float), ("hist_bytes", C.c_int64), ("full_ticks", C.c_int64),
                ("full_hist_bytes", C.c_int64), ("full_ms_cand", C.c_float), ("pad2_", C.c_float),
                ("slot_ticks", C.c_int64), ("ms_adj", C.c_float), ("ms_lbfgs", C.c_float), ("ms_gen", C.c_float),
                ("pad3_", C.c_float)]


def num_vars(piece_num):
    return 10 * piece_num - 8
