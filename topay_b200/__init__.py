"""topay_b200 — B200-native (CUDA sm_100a, fp64) hot path of the TopAY planner.

The product is topay_b200/libtopay_b200.so (kernels in csrc/, C ABI in include/topay_b200.h);
this package is the host-side mirror of the two reference interfaces it replaces:
GridMap (field.py), rog_map::ESDFMap (rog.py) and MomaTrajOpt (optimizer.py).
"""
from ._structs import (LBFGSERR_PLAN_GRACE, LBFGSERR_TICK_CAP, MAP2D_CRITICAL, MAP2D_FLAT, MAP2D_INFLATE, MAP3D, TERM_NAMES, GridDesc, OptParams,
                       RobotParams, RogDesc, grid_desc, num_vars, prob_desc, rog_desc)
from .field import GridMap, robot_params_default
from .rog import ESDFMap, ProbMap
from .optimizer import (MomaTraj, MomaTrajOpt, discretizePath, getDensePath, opt_params_default, pathLength,
                        prepare_candidate)

__all__ = ["GridMap", "ESDFMap", "ProbMap", "prob_desc", "rog_desc", "RogDesc", "MomaTrajOpt", "MomaTraj", "grid_desc", "GridDesc", "OptParams", "RobotParams",
           "robot_params_default", "opt_params_default", "prepare_candidate", "getDensePath", "discretizePath", "pathLength", "num_vars", "TERM_NAMES",
           "MAP2D_FLAT", "MAP2D_INFLATE", "MAP2D_CRITICAL", "MAP3D", "LBFGSERR_TICK_CAP",
           "LBFGSERR_PLAN_GRACE"]
