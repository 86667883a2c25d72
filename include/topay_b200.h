/*
 * topay_b200.h — C ABI of the B200-native hot path of the TopAY planner.
 *
 * Two opaque objects cross this boundary:
 *
 *   topay_field   replaces the distance-field half of the reference:
 *                 GridMap            (src/map/include/map/grid_map.h:77-219,
 *                                     src/map/src/grid_map.cpp:6-87,125-521,716-809)
 *   topay_solver  replaces the NLP-solve half of the reference:
 *                 MomaTrajOpt        (src/planner/include/planner/moma_traj_opt.h:613-675,
 *                                     src/planner/src/moma_traj_opt.cpp:142-498,817-1829)
 *
 * The reference has no FFI layer of its own (SURVEY.md §8b): these entry points
 * are what a maintainer binds from `Planner` (src/planner/src/planner.cpp:873-885)
 * through the C++ shims in shim/ (same class names and members).
 *
 * Conventions: plain pointers and sizes, caller-owned HOST buffers unless the
 * name ends in `_dev`, row-major, fp64 unless stated, int32 status return
 * (TOPAY_OK == 0; negative = error, see topay_strerror), no exceptions cross the
 * boundary, one host thread per handle. There is no CPU fallback: every compute
 * entry point fails with TOPAY_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef TOPAY_B200_H
#define TOPAY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ status */
enum {
    TOPAY_OK = 0,
    TOPAY_ERR_INVALID_ARG = -1,
    TOPAY_ERR_NO_DEVICE = -2,   /* no usable CUDA device: the product path refuses to run */
    TOPAY_ERR_CUDA = -3,        /* a CUDA runtime call failed; see topay_last_error() */
    TOPAY_ERR_ALLOC = -4,
    TOPAY_ERR_TOO_LARGE = -5,   /* n_cand / piece_num / int_K above the solver's capacity */
    TOPAY_ERR_NOT_READY = -6    /* field queried/solved before topay_field_rebuild */
};
const char* topay_strerror(int code);
const char* topay_last_error(void);   /* thread-local detail of the last failure */
const char* topay_version(void);

/* L-BFGS return codes, numerically identical to the reference's enum
 * (src/planner/include/utils/lbfgs.hpp:135-184). */
enum {
    TOPAY_LBFGS_CONVERGENCE = 0,
    TOPAY_LBFGS_STOP = 1,
    TOPAY_LBFGS_CANCELED = 2,
    TOPAY_LBFGSERR_UNKNOWNERROR = -1024,
    TOPAY_LBFGSERR_INVALID_N = -1023,
    TOPAY_LBFGSERR_INVALID_MEMSIZE = -1022,
    TOPAY_LBFGSERR_INVALID_GEPSILON = -1021,
    TOPAY_LBFGSERR_INVALID_TESTPERIOD = -1020,
    TOPAY_LBFGSERR_INVALID_DELTA = -1019,
    TOPAY_LBFGSERR_INVALID_MINSTEP = -1018,
    TOPAY_LBFGSERR_INVALID_MAXSTEP = -1017,
    TOPAY_LBFGSERR_INVALID_FDECCOEFF = -1016,
    TOPAY_LBFGSERR_INVALID_SCURVCOEFF = -1015,
    TOPAY_LBFGSERR_INVALID_MACHINEPREC = -1014,
    TOPAY_LBFGSERR_INVALID_MAXLINESEARCH = -1013,
    TOPAY_LBFGSERR_INVALID_FUNCVAL = -1012,
    TOPAY_LBFGSERR_MINIMUMSTEP = -1011,
    TOPAY_LBFGSERR_MAXIMUMSTEP = -1010,
    TOPAY_LBFGSERR_MAXIMUMLINESEARCH = -1009,
    TOPAY_LBFGSERR_MAXIMUMITERATION = -1008,
    TOPAY_LBFGSERR_WIDTHTOOSMALL = -1007,
    TOPAY_LBFGSERR_INVALIDPARAMETERS = -1006,
    TOPAY_LBFGSERR_INCREASEGRADIENT = -1005,
    /* not a reference code: the device solve stopped this candidate at its hard cap on evaluations
     * (topay_solver_run); the candidate comes back with status 0 */
    TOPAY_LBFGSERR_TICK_CAP = -2000,
    /* not a reference code: the candidate was cancelled because its plan had succeeded more than the grace period
     * earlier (topay_solver_set_plans, topay_solver_stream_set_grace), or its plan was stopped
     * (topay_solver_stream_stop); it comes back with status 0 */
    TOPAY_LBFGSERR_PLAN_GRACE = -2001
};

/* ------------------------------------------------------------------ params */

#define TOPAY_DOF 7          /* arm joints, MomaParam::dof_num (moma_param.h:53) */
#define TOPAY_DIM 9          /* spline dimensions: theta, arc, q1..q7 */
#define TOPAY_NSPHERE 12     /* arm collision spheres (moma_param.h:94-109) */
#define TOPAY_NTERMS 13      /* cost breakdown, order of moma_traj_opt.h:926-938 */

/* Order of the 13 per-evaluation term costs (DebugManager names,
 * src/planner/include/planner/moma_traj_opt.h:926-938). */
enum {
    TOPAY_TERM_JERK = 0, TOPAY_TERM_TIME, TOPAY_TERM_CHASSIS_COLLI, TOPAY_TERM_MOMENT,
    TOPAY_TERM_ACC, TOPAY_TERM_DOMEGA, TOPAY_TERM_MANI_COLLI, TOPAY_TERM_SELF_COLLI,
    TOPAY_TERM_MANI_POS, TOPAY_TERM_MANI_VEL, TOPAY_TERM_MANI_ACC, TOPAY_TERM_MEAN_TIME,
    TOPAY_TERM_ENDP   /* stage 2: ALM end-point term; stage 1: path-point tracking term */
};

/* Robot constants — mirrors struct MomaParam
 * (src/simulator/fake_moma/include/fake_moma/moma_param.h:33-144). */
typedef struct topay_robot_params {
    double chassis_height;            /* 0.155 */
    double chassis_colli_radius;      /* 0.4   */
    double max_v, max_a, max_w, max_dw;
    double colli_length[TOPAY_DOF + 1];
    double colli_points[2 * (TOPAY_DOF + 1)];        /* 0.0 entries are skipped */
    double colli_point_radius[2 * (TOPAY_DOF + 1)];
    double joint_pos_limit_max[TOPAY_DOF];           /* symmetric limits */
    double joint_vel_limit[TOPAY_DOF];
    double joint_acc_limit[TOPAY_DOF];
    double relative_R[9];                            /* row-major */
    double relative_t[3];
    int32_t collision_matrix[TOPAY_NSPHERE * TOPAY_NSPHERE]; /* -1 => pair is checked */
} topay_robot_params;

/* Fills the defaults exactly as MomaParam::MomaParam() does (moma_param.h:72-144),
 * including the zero-pose derivation of collision_matrix. Pure host code. */
void topay_robot_params_default(topay_robot_params* out);

/* lbfgs::lbfgs_parameter_t (src/planner/include/utils/lbfgs.hpp:13-129). */
typedef struct topay_lbfgs_params {
    int32_t mem_size;
    double  g_epsilon;
    int32_t past;
    double  delta;
    int32_t max_iterations;
    int32_t max_linesearch;
    double  min_step, max_step;
    double  f_dec_coeff, s_curv_coeff, cautious_factor, machine_prec;
} topay_lbfgs_params;

/* MomaTrajOptParam (moma_traj_opt.h:432-564) with the values of
 * src/planner/params/optimizer.yaml as defaults. */
typedef struct topay_opt_params {
    int32_t int_K;
    int32_t min_piece_num;
    double  relu_mu;
    double  sample_interval;
    double  energy_weights[TOPAY_DIM];
    /* first stage */
    double  s1_time_weight, s1_moment_weight, s1_acc_weight, s1_domega_weight;
    double  s1_mean_time_weight, s1_path_pos_weight;
    int32_t s1_lbfgs_normal_past, s1_lbfgs_shot_path_past;
    double  s1_shot_path_horizon;
    topay_lbfgs_params s1_lbfgs;
    /* second stage */
    double  s2_time_weight, s2_moment_weight, s2_acc_weight, s2_domega_weight;
    double  s2_collision_weight, s2_mani_colli_weight, s2_self_colli_weight;
    double  s2_mani_pos_weight, s2_mani_vel_weight, s2_mani_acc_weight, s2_mean_time_weight;
    topay_lbfgs_params s2_lbfgs;
    double  alm_init_lambda[2], alm_init_rho[2], alm_rho_max[2], alm_gamma[2];
    double  alm_tolerance;
    /* The reference bounds the ALM loop by 1.0 s of wall clock
     * (moma_traj_opt.cpp:403). A deterministic cap replaces it on both the
     * device path and the oracle: at most this many inner solves. */
    int32_t alm_max_rounds;
} topay_opt_params;

void topay_opt_params_default(topay_opt_params* out);

/* Dense GridMap geometry — the rosparams of src/planner/params/grid_map.yaml;
 * everything else is derived exactly as GridMap::init does (grid_map.cpp:33-54). */
typedef struct topay_grid_desc {
    double map_size[3];
    double resolution;
    double chassis_colli_radius;   /* threshold of the inflated 2-D maps (grid_map.cpp:288,360) */
    double chassis_height;         /* rasterisation threshold of occ_2d (grid_map.cpp:740) */
} topay_grid_desc;

typedef struct topay_field  topay_field;
typedef struct topay_solver topay_solver;

/* which 2-D map a query reads (GridMap::getDisWithGradI2d flags, grid_map.h:364-429) */
enum { TOPAY_MAP2D_FLAT = 0, TOPAY_MAP2D_INFLATE = 1, TOPAY_MAP2D_CRITICAL = 2, TOPAY_MAP3D = 3 };

/* ------------------------------------------------------------------- field */

/* GridMap::init (grid_map.cpp:6-65): allocates occupancy + ESDF buffers in HBM. */
int topay_field_create(const topay_grid_desc* desc, int device, topay_field** out);
void topay_field_destroy(topay_field* f);
/* voxel_num as GridMap::getVoxelNum (grid_map.h:179). */
int topay_field_dims(const topay_field* f, int32_t dims[3]);

/* GridMap::loadMap (grid_map.cpp:800-809) semantics when occ2d_critical == NULL:
 * occ_2d and occ_3d are replaced, the critical occupancy is left as it is.
 * A NULL occ3d / occ2d leaves that buffer unchanged. Values are 0/1, layout
 * x*Ny*Nz + y*Nz + z (grid_map.h:808-816) and x*Ny + y (grid_map.h:798-806). */
int topay_field_set_occupancy(topay_field* f, const int8_t* occ3d, const int8_t* occ2d,
                              const int8_t* occ2d_critical);
/* The reset GridMap::regenerateMap / regenerateDesk perform before rasterising
 * (grid_map.cpp:719-722): occ_2d and occ_3d are zeroed; occ_2d_critical is
 * kept unless clear_critical != 0 (reference quirk, SURVEY.md §8a quirk 6). */
int topay_field_clear(topay_field* f, int clear_critical);
/* Point-cloud ingest of regenerateMap / cloudCallback (grid_map.cpp:733-747,
 * 554-568): float32 xyz triples, promoted to double before indexing. */
int topay_field_rasterize_points(topay_field* f, const float* xyz, int64_t n_points);
/* GridMap::updateESDF (grid_map.cpp:125-521): four signed 2-D maps + the signed 3-D map. */
int topay_field_rebuild(topay_field* f);

/* GridMap::getDisWithGradI3d (grid_map.h:443-509); grad may be NULL. pos is n x 3. */
int topay_field_query3d(topay_field* f, const double* pos, int64_t n, double* dist, double* grad);
/* GridMap::getDisWithGradI2d (grid_map.h:364-441); pos is n x 2, grad n x 2 or NULL. */
int topay_field_query2d(topay_field* f, const double* pos, int64_t n, int which, double* dist,
                        double* grad);
/* GridMap::getDistance3d / getDistance2d (grid_map.h:256-362): value only, 1e10 outside. */
int topay_field_distance3d(topay_field* f, const double* pos, int64_t n, double* dist);
int topay_field_distance2d(topay_field* f, const double* pos, int64_t n, double* dist);
/* GridMap::isWholeBodyCollision (grid_map.h:613-650); states are n x 10; out 0/1. */
int topay_field_whole_body_collision(topay_field* f, const topay_robot_params* robot,
                                     const double* states, int64_t n, int8_t* out);
/* GridMap::isCollision2d / isCollision3d (grid_map.h:511-536, 695-724): distance below
 * threshold, or outside the map. pos is n x 2 / n x 3, out[i] in {0,1}. */
int topay_field_is_collision2d(topay_field* f, const double* pos, int64_t n, double threshold, int8_t* out);
int topay_field_is_collision3d(topay_field* f, const double* pos, int64_t n, double threshold, int8_t* out);
/* GridMap::isLineCollisionGrid2d (grid_map.h:565-611): Bresenham walk over the flat map between
 * the cells of p1 and p2 (both n x 2), both end cells tested. */
int topay_field_is_line_collision_grid2d(topay_field* f, const double* p1, const double* p2, int64_t n,
                                         double threshold, int8_t* out);
/* GridMap::getDistCoarse2d / getDistCoarse2i (grid_map.h:887-940): nearest cell (clamped to the
 * grid) of the critical map, else of the inflated map. idx is n x 2 int32. */
int topay_field_dist_coarse2d(topay_field* f, const double* pos, int64_t n, int critical, double* out);
int topay_field_dist_coarse2i(topay_field* f, const int32_t* idx, int64_t n, int critical, double* out);
/* TopologyPRM::lineVisib (src/planner/src/topo_prm.cpp:278-315) on n segments p1 -> p2 (both n x 3, z is
 * carried through the ray walk as in the reference): the planner's RayCaster (src/planner/src/utils/raycast.cpp:
 * 253-346) steps through the cells from p1 / res to p2 / res, every cell but the end cell is looked up through
 * getDistCoarse2i in the inflated (use_critical = 0) or critical map; visible[i] = 0 when a cell at or below `thresh`
 * blocks the ray, and pc[i] (n x 3, in/out) then holds the midpoint of that cell's centre and the previous
 * cell's, z = 0; pc of a visible segment is left as passed in. Front-end row N2 of SURVEY.md §8f. */
int topay_field_line_visible(topay_field* f, const double* p1, const double* p2, int64_t n, double thresh,
                             int use_critical, int8_t* visible, double* pc);
/* TopologyPRM::sameTopoPath (topo_prm.cpp:424-448) for n_pairs pairs of paths in one launch (the PRM's
 * pruneEquivalent compares every path with every kept one): path p is the polyline pts[offsets[p] .. offsets[p+1])
 * (rows of 3), pairs is n_pairs x 2 path indices; same[k] = 1 when every pair of the ceil(max length / resolution)
 * equally spaced points (discretizePath) of the two paths sees each other (lineVisib with `thresh`). Paths must be
 * longer than one cell. */
int topay_field_same_topo_paths(topay_field* f, const double* pts, const int32_t* offsets, int n_paths,
                                const int32_t* pairs, int n_pairs, double thresh, int use_critical, int8_t* same);
/* Same queries with DEVICE pointers (inputs and outputs already in HBM), asynchronous
 * on the field's stream; used by the resident benchmark and by the solver. The launch goes to
 * the field's own non-blocking stream and is not ordered after any work the caller queued on
 * its streams: the caller must synchronise the stream that wrote pos_dev (or the device)
 * before the call, and call topay_field_sync before it reads dist_dev / grad_dev. */
int topay_field_query3d_dev(topay_field* f, const double* pos_dev, int64_t n, double* dist_dev,
                            double* grad_dev);
int topay_field_sync(topay_field* f);

/* getESDFBuffer2d/3d (grid_map.h:216-217) and the other two 2-D maps; `which` as above. */
int topay_field_download(topay_field* f, int which, double* esdf_out);
/* The integer squared distances (in cells^2) behind a map: pos_sq to the nearest
 * occupied cell, neg_sq to the nearest free cell; INT32_MAX where the reference
 * carries DBL_MAX (no source cell on the whole grid). Either pointer may be NULL. */
int topay_field_download_sqdist(topay_field* f, int which, int32_t* pos_sq, int32_t* neg_sq);
int topay_field_download_occupancy(topay_field* f, int which, int8_t* occ_out);
/* Whether topay_field_rebuild also stores the integer grids (default 1). Turning it off
 * removes 8 B/voxel of writes from the last pass; download_sqdist then fails. */
int topay_field_set_keep_sqdist(topay_field* f, int keep);
/* Device time of the last topay_field_rebuild, measured with CUDA events on the
 * field's stream; ms_3d is the 3-D part alone. */
int topay_field_last_rebuild_ms(topay_field* f, float* ms_total, float* ms_3d);

/* ---------------------------------------------------------- ROG-Map field */

/* The sliding ring-buffer distance field the reference uses when
 * grid_map/use_rog is true: rog_map::ESDFMap (src/rog_map/include/rog_map/
 * esdf_map.h) on top of CounterMap and SlidingMap, ORIGIN_AT_CORNER
 * discretisation (src/rog_map/CMakeLists.txt:14). The arguments are those of
 * ESDFMap::initESDFMap (esdf_map.cpp:28-57) as ProbMap passes them
 * (prob_map.cpp:48-58). */
typedef struct topay_rog_desc {
    int32_t half_prob_map_size_i[3];   /* cfg_.half_map_size_i (config.hpp:336-382) */
    double  prob_resolution;           /* cfg_.resolution */
    double  esdf_resolution;           /* cfg_.esdf_resolution */
    double  local_update_box[3];       /* cfg_.esdf_local_update_box, metres */
    int32_t map_sliding_en;
    double  fix_map_origin[3];         /* origin when map_sliding_en == 0 */
    double  unk_thresh;                /* ratio in [0,1] (counter_map.cpp:83-85) */
} topay_rog_desc;

typedef struct topay_rogfield topay_rogfield;

/* rog_map::GridType (include/utils/common_lib.hpp:74-81) */
enum { TOPAY_ROG_UNDEFINED = 0, TOPAY_ROG_UNKNOWN = 1, TOPAY_ROG_OUT_OF_MAP = 2, TOPAY_ROG_OCCUPIED = 3,
       TOPAY_ROG_KNOWN_FREE = 4 };

/* which quantity topay_rogfield_query evaluates */
enum {
    TOPAY_ROG_Q_EDT = 0,            /* evaluateEDT + evaluateFirstGrad = getValueGrad (esdf_map.cpp:951-1003) */
    TOPAY_ROG_Q_FLAT = 1,           /* getValueGrad2d        (esdf_map.cpp:1053-1097) */
    TOPAY_ROG_Q_CRITICAL = 2,       /* getCriticalValueGrad  (esdf_map.cpp:1005-1051) */
    TOPAY_ROG_Q_CELL = 3,           /* getDistance(pos)         nearest cell, grad untouched (esdf_map.cpp:78-80) */
    TOPAY_ROG_Q_CELL_FLAT = 4,      /* getDistance2d(pos)       (esdf_map.cpp:104-111) */
    TOPAY_ROG_Q_CELL_CRITICAL = 5   /* getCriticalDistance(pos) (esdf_map.cpp:86-93) */
};
/* buffers topay_rogfield_download returns */
enum { TOPAY_ROG_BUF_DIST3 = 0, TOPAY_ROG_BUF_NEG3 = 1, TOPAY_ROG_BUF_CRITICAL = 2, TOPAY_ROG_BUF_FLAT = 3 };

/* rog_map::ProbMap — the probabilistic occupancy layer that drives the ESDF counter map from point clouds
 * (src/rog_map/src/rog_map/prob_map.cpp; parameters of rog_map_core/config.hpp:160-262). The probability grid
 * shares half_prob_map_size_i / prob_resolution / map_sliding_en / fix_map_origin with the ESDF ring it feeds. */
typedef struct topay_prob_desc {
    float   p_hit, p_miss, p_min, p_max, p_occ, p_free;   /* raycasting/p_*; the log-odds are logit() in float */
    double  raycast_range_min, raycast_range_max;          /* raycasting/ray_range */
    double  virtual_ceil_height, virtual_ground_height;    /* as configured: InfMap's constructor pulls them in by
                                                            * inflation_step cells first (inf_map.cpp:81-89), then
                                                            * initProbMap snaps them to the grid (prob_map.cpp:66-71) */
    double  inflation_resolution;                          /* rounded up to a multiple of the resolution (config.hpp:338-349) */
    int32_t inflation_step;
    int32_t pad_;
    double  local_update_box[3];                           /* raycasting/local_update_box, metres */
    double  map_sliding_thresh;
    int32_t point_filt_num;                                /* keep every point_filt_num-th point */
    int32_t batch_update_size;                             /* clouds per probabilistic update */
    int32_t intensity_thresh;                              /* <= 0: off */
    int32_t raycasting_en;
} topay_prob_desc;
typedef struct topay_probmap topay_probmap;

/* initESDFMap: sizes derived as CounterMap::initCounterMap does (counter_map.cpp:31-91,
 * inflation_step 0), buffers in HBM, counters reset (esdf_map.cpp:72-76). */
int topay_rogfield_create(const topay_rog_desc* desc, int device, topay_rogfield** out);
void topay_rogfield_destroy(topay_rogfield* f);
/* half_map_size_i, map_size_i (= 2*half+1), resolution, local origin index, half update box. */
int topay_rogfield_geometry(const topay_rogfield* f, int32_t half[3], int32_t size[3], double* resolution,
                            int32_t origin_i[3], int32_t half_box_i[3]);
/* SlidingMap::mapSliding (sliding_map.cpp:113-166): moves the local origin to the cell of
 * odom and clears the slabs that left the map (both counters, counter_map.h:127-131). */
int topay_rogfield_slide(topay_rogfield* f, const double odom[3]);
/* CounterMap::updateGridCounter (counter_map.cpp:94-151) for n positions (n x 3), applied
 * in order; from_type / to_type are GridType values, one byte each. */
int topay_rogfield_update_counters(topay_rogfield* f, const double* pos, const uint8_t* from_type,
                                   const uint8_t* to_type, int64_t n);
/* Whole-buffer access to md_.occupied_cnt (ring-memory layout x*Sy*Sz + y*Sz + z). */
int topay_rogfield_set_occupied_cnt(topay_rogfield* f, const int16_t* cnt);
int topay_rogfield_download_counters(topay_rogfield* f, int16_t* occupied_cnt, int16_t* unknown_cnt);
/* ESDFMap::updateESDF3D (esdf_map.cpp:154-500): signed EDT of the local update box around
 * cur_odom with the ring wrap, then the critical and flat 2-D maps. */
int topay_rogfield_update_esdf(topay_rogfield* f, const double cur_odom[3]);
/* Batched queries; pos is n x 3 (z is ignored by the 2-D kinds except for the ring index of
 * the taps, as in the reference). dist: n; grad: n x 3 or NULL. */
int topay_rogfield_query(topay_rogfield* f, int kind, const double* pos, int64_t n, double* dist, double* grad);
/* ESDFMap::isLineFree2d (esdf_map.cpp:122-152): start/end are n x 2, out[i] = 1 when free. */
int topay_rogfield_is_line_free2d(topay_rogfield* f, const double* start, const double* end, int64_t n,
                                  double threshold, int8_t* out);
int topay_rogfield_download(topay_rogfield* f, int which, double* out);
int topay_rogfield_last_update_ms(topay_rogfield* f, float* ms_total, float* ms_3d);

/* ProbMap over an ESDF ring (borrowed; must outlive the prob map): initProbMap (prob_map.cpp:25-88). */
int topay_probmap_create(topay_rogfield* esdf, const topay_prob_desc* desc, topay_probmap** out);
void topay_probmap_destroy(topay_probmap* m);
/* ProbMap::updateProbMap(cloud, pose) (prob_map.cpp:302-373): slides the maps when the robot left them, clips
 * and filters the points, walks the rays, applies the cached hits / misses to the log-odds, forwards every
 * UNKNOWN / OCCUPIED / KNOWN_FREE transition to the ESDF counter map and runs updateESDF3D(pos). cloud: n x
 * (x, y, z, intensity) float32, host memory. */
int topay_probmap_update(topay_probmap* m, const float* cloud_xyzi, int64_t n, const double pos[3]);
/* occupancy_buffer_ (log-odds, ring memory, (2h+1)^3 floats) and the map origin in cells. */
int topay_probmap_download(topay_probmap* m, float* occupancy, int32_t origin_i[3]);
/* the first-frame sphere clearing of updateProbMap is a function-level static in the reference (once per
 * process); this re-arms (1) or disarms (0) it for this map */
int topay_probmap_set_first_frame(topay_probmap* m, int armed);

/* -------------------------------------- result post-processing + success gate */

/* n MomaTraj inputs (moma_traj_opt.h:26-68): what MinJerkOpt<9>::getTraj hands over
 * (minco.hpp:908-921) plus the SE(2) start. coeff rows are in the solver's layout —
 * row 6i+k = coefficient of t^k of piece i — the reference stores the same numbers in
 * descending order. Host pointers. */
typedef struct topay_traj_batch {
    int32_t n_traj;
    int32_t max_pieces;          /* row pitch of T and coeff */
    const int32_t* piece_num;    /* [n] */
    const double*  T;            /* [n][max_pieces] */
    const double*  coeff;        /* [n][6*max_pieces][9] */
    const double*  start_se2;    /* [n][3] x, y, yaw */
} topay_traj_batch;

/* What checkFeasible / printConstraintsSituations accumulate (moma_traj_opt.h:948-1210)
 * over samples at t = 0, 0.01, ... < duration. The max_* entries are the signed value of the
 * first sample that attains the largest magnitude, as the reference's running update keeps
 * it. Host pointers; any may be NULL except feasible. */
typedef struct topay_feasibility {
    int32_t* feasible;         /* [n] checkFeasible */
    int32_t* feasible_print;   /* [n] printConstraintsSituations: manipulator clearance reported, not enforced (:1199) */
    int32_t* n_samples;        /* [n] */
    double*  max_vel;          /* [n] */
    double*  max_acc;
    double*  max_domega;
    double*  max_d2omega;
    double*  max_q;            /* [n][7] */
    double*  max_dq;
    double*  max_d2q;
    double*  min_dist;         /* [n] chassis clearance (getDistance2d) */
    double*  min_dist_mani;    /* [n][12] sphere-centre clearance (getDistance3d) */
} topay_feasibility;

/* MomaTrajOpt::checkFeasible for n trajectories at once: one thread block per trajectory. */
int topay_traj_check_feasible(topay_field* f, const topay_robot_params* robot, const topay_traj_batch* trajs,
                              topay_feasibility* out);
/* The same check against a ROG-Map ring (GridMap's use_rog branches, as the solver-resident gate of a ROG solver reads
 * it): is a trajectory still feasible on the map as it is now? Runs on the ring's stream, after every update queued
 * there. A ring never updated (topay_rogfield_update_esdf): TOPAY_ERR_NOT_READY. */
int topay_traj_check_feasible_rog(topay_rogfield* f, const topay_robot_params* robot, const topay_traj_batch* trajs,
                                  topay_feasibility* out);
/* MomaTraj::car_seq (moma_traj_opt.h:38-68): entries (x, y, yaw, t); len[i] entries of
 * trajectory i are written to car_seq[i*cap*4 ...] (TOPAY_ERR_TOO_LARGE if one needs more than cap). */
int topay_traj_car_seq(int device, const topay_traj_batch* trajs, int cap, double* car_seq, int32_t* len);
/* MomaTraj::getState / getDState (moma_traj_opt.h:121-160) at m times per trajectory:
 * t [n][m] -> state [n][m][10] (x, y, yaw, q1..q7), dstate [n][m][10] (v, omega, 0, dq); either output may be NULL. */
int topay_traj_sample(int device, const topay_traj_batch* trajs, const double* t, int m, double* state,
                      double* dstate);
/* The planner's pick (planner.cpp:999-1010): first success, replaced by any later strictly
 * shorter trajectory; -1 when nothing succeeded. Pure host code. */
int topay_select_shortest(const int32_t* success, const double* duration, int n);

/* ------------------------------------------------------------------ solver */

/* One solver = the device-side state for up to max_cand candidates of up to
 * max_pieces pieces each (what the reference keeps in <= 8 MomaTrajOpt
 * instances, planner.cpp:59-66). The field is borrowed, read-only. */
int topay_solver_create(const topay_opt_params* opt, const topay_robot_params* robot,
                        topay_field* field, int max_cand, int max_pieces, topay_solver** out);
/* The same solver reading the ROG-Map ring instead of the dense field: GridMap's use_rog
 * branches of getDisWithGradI2d / getDisWithGradI3d / getDistance2d / getDistance3d
 * (grid_map.h:256-267, 307-322, 364-392, 443-461). */
int topay_solver_create_rog(const topay_opt_params* opt, const topay_robot_params* robot,
                            topay_rogfield* rog, int max_cand, int max_pieces, topay_solver** out);
/* Continuous batching: an upload may hold up to max_cand candidates (several plans back to back) while only
 * n_slots of them are in flight on the device; the moment a candidate reaches a terminal state its slot takes
 * the next waiting one, on the device, so every tick runs over live candidates only. This is the worker pool
 * of planner.cpp:921-952 (a fixed number of workers, each taking the next candidate when it is done) with the
 * queue on the GPU. topay_solver_create(max_cand) == topay_solver_create_pool(max_cand, n_slots = max_cand).
 * Device memory: n_slots x 2 x mem_size x (10 max_pieces - 8) x 8 B of L-BFGS history (2.6 MB per slot at
 * 64 pieces) + 30 KB of results per stored candidate. */
int topay_solver_create_pool(const topay_opt_params* opt, const topay_robot_params* robot,
                             topay_field* field, int max_cand, int n_slots, int max_pieces,
                             topay_solver** out);
void topay_solver_destroy(topay_solver* s);

/* The fixed data of each candidate's NLP, i.e. what optimizeTraj derives before it
 * packs x (moma_traj_opt.cpp:281-304). Host pointers. */
typedef struct topay_problem_batch {
    int32_t        n_cand;
    const int32_t* piece_num;      /* [n_cand] */
    const double*  head_pva;       /* [n_cand][9][3]  minco_start_state */
    const double*  tail_pva;       /* [n_cand][9][3]  minco_end_state; [1][0] is overwritten by x */
    const double*  start_xy;       /* [n_cand][2]     start_state.head(2) */
    const double*  end_xy;         /* [n_cand][2]     end_state.head(2) */
    const double*  init_inner_xy;  /* [n_cand][max_pieces][2] stage-1 targets, first piece_num rows used */
    const double*  alm_lambda;     /* [n_cand][2]  stage 2 only (may be NULL for stage 1) */
    const double*  alm_rho;        /* [n_cand][2] */
} topay_problem_batch;

/* One cost+gradient evaluation per candidate: firstStageCostCallback (stage == 1,
 * moma_traj_opt.cpp:817-883) or secondStageCostCallback (stage == 2, :885-955).
 * x and grad are [n_cand][x_stride] with the layout of moma_traj_opt.cpp:324-344
 * (tau(N) | theta(N-1) | arc(N) | vq(7 x (N-1), column-major)); cost is [n_cand];
 * term_costs is [n_cand][TOPAY_NTERMS] or NULL; coeff_out is
 * [n_cand][6*max_pieces][9] or NULL; final_xy_out [n_cand][2] or NULL. */
int topay_solver_eval(topay_solver* s, int stage, const topay_problem_batch* prob,
                      const double* x, int x_stride, double* cost, double* grad,
                      double* term_costs, double* coeff_out, double* final_xy_out);

/* Number of optimisation variables of an N-piece candidate: 9(N-1)+N+1. */
static inline int topay_num_vars(int piece_num) { return 10 * piece_num - 8; }

/* GraphSearch::getDensePath (src/planner/src/graph_search.cpp:119-176; called by every planning worker right
 * before the sampler and the solve, planner.cpp:858): raw 2-D waypoints (n x 2) -> rows (x, y, theta, dt): every
 * segment cut into ceil(len / step_size) steps, a turn-in-place row before and after every move, yaw unwrapped
 * against the previous row, rows shorter than 1e-3 s dropped. Host arithmetic. Writes at most `cap` rows to out
 * (cap x 4) and returns the number of rows the path has (> cap: call again), or a negative TOPAY_ERR_*. */
int topay_dense_path(const double* raw_xy, int n, double step_size, double start_yaw, double end_yaw, double v_max,
                     double w_max, double* out, int cap);

/* TopologyPRM::pathLength / discretizePath (src/planner/src/topo_prm.cpp:462-506): length of a 3-D polyline (n rows
 * of 3) and pt_num >= 2 points at equal arc-length spacing along it (out: pt_num x 3). Host arithmetic. */
double topay_path_length(const double* path, int n);
int topay_discretize_path(const double* path, int n, int pt_num, double* out);

/* MomaTrajOpt::optimizeTraj pre-processing (moma_traj_opt.cpp:146-344): waypoints ->
 * problem data + initial x. Host-side helper of solve_batch, exported for parity
 * tests. init_path is path_len x 10 (x,y,yaw,q1..q7); bvel/bacc are 10 x 2
 * row-major (planner.cpp:873-875). Outputs sized for max_pieces; returns the
 * piece count in *piece_num or TOPAY_ERR_TOO_LARGE. */
int topay_prepare_candidate(const topay_opt_params* opt, const topay_robot_params* robot,
                            const double* init_path, int path_len, const double* bvel,
                            const double* bacc, int max_pieces, int32_t* piece_num,
                            double* head_pva /*27*/, double* tail_pva /*27*/,
                            double* start_xy /*2*/, double* end_xy /*2*/,
                            double* init_inner_xy /*max_pieces x 2*/, double* x0 /*10*max_pieces-8*/,
                            int32_t* s1_past);

/* Results of a batched solve; host pointers, any may be NULL except status. */
typedef struct topay_result_batch {
    int32_t* status;        /* [n] 1 = optimizeTraj returned true, 0 = false */
    int32_t* lbfgs_code;    /* [n] return code of the last lbfgs_optimize call */
    int32_t* piece_num;     /* [n] */
    int32_t* iters;         /* [n] L-BFGS iterations, both stages */
    int32_t* evals;         /* [n] cost/gradient evaluations, both stages */
    int32_t* alm_rounds;    /* [n] */
    double*  cost;          /* [n] traj_cost (moma_traj_opt.cpp:495) */
    double*  duration;      /* [n] sum of piece durations of the returned trajectory */
    double*  T;             /* [n][max_pieces], zero past piece_num */
    double*  coeff;         /* [n][6*max_pieces][9] minco coefficients of the last evaluation, rows past
                               6*piece_num zero */
    double*  final_xy_err;  /* [n][2] */
    double*  x;             /* [n][10*max_pieces-8] final variables */
} topay_result_batch;

/* The batched replacement of n_cand concurrent MomaTrajOpt::optimizeTraj calls
 * (planner.cpp:878): pre-processing on the host, then stage 1, then the stage-2
 * ALM loop entirely on the device. init_paths holds the candidates' waypoint
 * lists back to back (sum(path_len) x 10). best_by_duration follows the
 * reference's selection rule (planner.cpp:999-1010), best_by_cost is the
 * north-star's argmin over successful candidates; -1 when none succeeded. */
int topay_solver_solve_batch(topay_solver* s, int n_cand, const int32_t* path_len,
                             const double* init_paths, const double* bvel, const double* bacc,
                             topay_result_batch* out, int32_t* best_by_duration,
                             int32_t* best_by_cost);

/* Split form for resident benchmarking: upload + pre-process once, then run the
 * device solve any number of times from the same initial state. */
int topay_solver_upload(topay_solver* s, int n_cand, const int32_t* path_len,
                        const double* init_paths, const double* bvel, const double* bacc);
int topay_solver_run(topay_solver* s);          /* device solve of the uploaded batch, blocking */
/* Scenario sweeps (BASELINE configs[4]: thousands of independent scenarios, each with its own 200 x 200 x 16 field and
 * a handful of candidates; the reference plans them one after the other, planner.cpp:494-548 + :847-1010): the
 * candidates of ONE upload may belong to different scenarios. field_of[c] (one entry per uploaded candidate) indexes
 * `fields` (dense fields on the solver's device, rebuilt before the run); the solve, the success gate
 * (topay_solver_check_feasible) and the selection then read every candidate against its own field, so that a whole
 * group of scenarios shares the launches of one solve. The assignment holds for uploads of the same size until it is
 * changed; n_fields <= 1 returns to the solver's own field. Call after topay_solver_upload. Rebuild the fields first;
 * in a streaming session, a plan's field must stay as it is until the plan has finished (topay_solver_stream_submit). */
int topay_solver_assign_fields(topay_solver* s, topay_field* const* fields, int n_fields, const int32_t* field_of);
/* First success + grace of the planner's worker pool (planner.cpp:931-952), with the grace counted in evaluations
 * instead of the reference's 100 ms of wall-clock time, so that the outcome does not depend on scheduling. The upload
 * is read as n_plans plans, plan p = candidates plan_offset[p] .. plan_offset[p+1]-1 (n_plans + 1 entries, starting
 * at 0, non-decreasing, ending at the uploaded n_cand). All candidates of a plan count as started together.
 *   A candidate succeeds when it ends with status 1 and, with use_gate != 0, printConstraintsSituations passes
 *   (feasible_print, planner.cpp:877-880). S_p = the fewest evaluations (result `evals`) among the candidates of plan p
 *   that succeed when nothing is cancelled; no success: S_p = infinity.
 *   A candidate with evals <= S_p + grace_evals in that unbounded run is KEPT: its results, trace and gate metrics
 *   are bit-identical to the unbounded run. Every other candidate of the plan is CANCELLED: status 0, lbfgs_code
 *   TOPAY_LBFGSERR_PLAN_GRACE, piece_num kept, iters, evals, alm_rounds, cost, duration, T, coeff, final_xy_err and x
 *   zero, an empty trace, both gate verdicts, n_samples and every gate metric zero.
 * So a plan has a winner if and only if it has one unbounded (its earliest success is never cancelled), and the
 * result depends on each candidate's own evaluation count only: not on slots, lanes, timed mode or queue order.
 * Cancelled candidates free their slots at once. The setting holds for uploads of the same size until it is changed
 * (topay_solver_run refuses an upload of another size with TOPAY_ERR_NOT_READY); n_plans == 0 turns it off. Call after
 * topay_solver_upload. Malformed offsets, grace_evals < 0 or n_plans > n_cand: TOPAY_ERR_INVALID_ARG. */
int topay_solver_set_plans(topay_solver* s, int n_plans, const int32_t* plan_offset, int use_gate, int32_t grace_evals);
int topay_solver_download(topay_solver* s, topay_result_batch* out, int32_t* best_by_duration,
                          int32_t* best_by_cost);

/* Device-side counters of the last run: kernel launches issued, lock-step ticks,
 * device ms spent in the evaluation kernels and in the whole solve (CUDA events). */
typedef struct topay_solver_stats {
    int64_t kernel_launches;
    int64_t ticks;
    int64_t evals_total;       /* sum over candidates */
    float   ms_total;
    float   ms_eval;           /* penalty-node kernel only */
    int64_t eval_launches;     /* launches of the penalty-node kernel */
    int64_t eval_nodes;        /* penalty nodes processed by them (active candidates only) */
    float   ms_integrate;      /* timed mode only: device ms in k_integrate, k_chain, k_cand */
    float   ms_chain;
    float   ms_cand;
    float   pad_;
    int64_t hist_bytes;        /* algorithmic bytes of L-BFGS history the two-loop recursions walked:
                                * 2 loops x bound rows x (s_j, y_j) x n x 8 B, summed over candidates */
    /* timed mode only: the same k_cand figures restricted to the tick batches in which every
     * candidate was still solving (full activity) */
    int64_t full_ticks;
    int64_t full_hist_bytes;
    float   full_ms_cand;
    float   pad2_;
    int64_t slot_ticks;        /* live slots summed over the ticks: the evaluations the launches were sized for;
                                * evals_total / slot_ticks = slot utilisation */
    float   ms_adj, ms_lbfgs, ms_gen;   /* timed mode only: the three per-candidate launches that make up ms_cand;
                                         * full_ms_cand is the L-BFGS launch alone */
    float   pad3_;
} topay_solver_stats;
int topay_solver_last_stats(topay_solver* s, topay_solver_stats* out);
/* The worker's success gate on the device, straight from the solver's result buffers
 * (planner.cpp:877-880): checkFeasible of every candidate of the last run. best_success is
 * the shortest-duration candidate among those with status && feasible_print (the gate the
 * planner applies), -1 if none. */
int topay_solver_check_feasible(topay_solver* s, topay_feasibility* out, int32_t* best_success);
/* The planner's pick among the candidates of the last run, ON THE DEVICE (planner.cpp:999-1010: the first success,
 * replaced only by a strictly shorter duration; the same rule on the cost): the upload is read as n_plans plans,
 * plan i = candidates plan_offset[i] .. plan_offset[i+1]-1 (plan_offset has n_plans + 1 entries). A candidate
 * counts when optimizeTraj succeeded and, with use_gate != 0, printConstraintsSituations passed
 * (planner.cpp:877-880; topay_solver_check_feasible must have run on this solve). Writes, per plan, the index
 * INSIDE the plan of the winner by duration / by cost (-1: none); either output may be NULL. Two ints per plan
 * cross the bus. */
int topay_solver_select(topay_solver* s, int n_plans, const int32_t* plan_offset, int use_gate,
                        int32_t* best_by_duration, int32_t* best_by_cost);
/* Results of ONE candidate of the last run (e.g. the winner): `out`'s arrays have length 1 (T: max_pieces,
 * coeff: 6 max_pieces x 9, x: topay_num_vars(max_pieces)). 28 KB at 64 pieces instead of the whole batch. */
int topay_solver_download_candidate(topay_solver* s, int cand, topay_result_batch* out);

/* Streaming session: plans are submitted while the solve runs, and each plan's winners come back as soon as that plan's
 * last candidate has finished — the worker pool of planner.cpp:921-952 with plans arriving while it works. Every
 * streamed plan is bit-identical to the same plan solved alone through the batch API on a fresh upload (results, gate
 * metrics and winners): a candidate's result depends on its own inputs only, not on slots, lanes, timed mode or when
 * its plan arrived. One host thread per solver, as for every other call.
 *   stream_begin starts a session on an empty pool; it drops the uploaded batch and its set_plans setting, so a
 *     session starts with first success + grace off (stream_set_grace turns it on). Both stages need bounded max_iterations (else TOPAY_ERR_INVALID_ARG), so every candidate ends; TOPAY_MAX_TICKS
 *     does not apply. use_gate != 0: a candidate counts for its plan's winners only if printConstraintsSituations
 *     passes (as topay_solver_select with use_gate). Two lanes when n_slots reaches the batch run's threshold.
 *   stream_submit prepares every candidate on the host (a failure changes nothing), writes them into free store rows
 *     and queues them; *plan_id names the plan until it is taken. Not enough free rows: TOPAY_ERR_TOO_LARGE, nothing
 *     changed. `field` (NULL: the solver's own) is a built dense field on the solver's device; every candidate of the
 *     plan is solved and gated against it. A ROG solver takes NULL only.
 *   stream_advance runs up to max_batches batches of 16 ticks (graph replays, or plain launches in timed mode); idle
 *     slots take the newly queued candidates first. *n_live (may be NULL) = candidates in the slots afterwards; 0 means
 *     every submitted candidate has finished. Returns at once when nothing is live.
 *   stream_poll writes up to cap finished plans, each reported once, with their winners by duration and by cost (index
 *     inside the plan, -1: none; planner.cpp:999-1010, ties to the earliest candidate); returns the number written.
 *   stream_take downloads the results of candidate `cand` of a finished plan (-1: all of them, in submission order;
 *     topay_result_batch layout, entries past piece_num zero) and, if gate is not NULL, their gate metrics; then the
 *     plan's rows and its id are free. An unknown, unfinished or already taken plan: TOPAY_ERR_INVALID_ARG.
 *   stream_set_grace applies first success + grace (topay_solver_set_plans) to every plan streamed from then on:
 *     grace_evals >= 0 turns it on, -1 turns it off, any other value is TOPAY_ERR_INVALID_ARG. A success follows the
 *     session's use_gate. Every plan streamed with grace G is bit-identical (results, gate metrics from stream_take,
 *     winners) to the same plan solved alone on a fresh upload with set_plans(1, {0, n}, use_gate, G), whatever the
 *     slots, lanes, timed mode, arrival schedule or store rows. G is part of each live plan's contract: while a
 *     submitted plan has not finished, the call returns TOPAY_ERR_NOT_READY (finished plans not taken yet are fine).
 *   stream_stop stops a live plan, as the reference's interrupt_all (planner.cpp:952) does for its workers: a candidate
 *     in a slot is cancelled at its next L-BFGS step; a queued one still takes a slot for one tick, its first
 *     evaluation, and is cancelled right after it. The plan then finishes through stream_advance and stream_poll as
 *     usual, reported once. Its candidates that finished before the stop keep their results under the plan's grace
 *     contract, with S_p taken over them (with grace off, all of them are kept); every other candidate comes back
 *     cancelled (status 0, TOPAY_LBFGSERR_PLAN_GRACE, the values of topay_solver_set_plans). Which candidates finish
 *     before a stop depends on timing, so a stopped plan's outcome is not deterministic. What holds: each of its
 *     candidates is either bit-identical to its result without grace or cancelled; a candidate that finished before
 *     the stop and is kept by the grace contract is kept; other plans are unaffected bit for bit. A plan's field must
 *     still stay as it is until the plan is reported. A finished plan not taken yet: TOPAY_OK, nothing changes. An
 *     unknown or taken plan: TOPAY_ERR_INVALID_ARG. The first stop of a session without grace has candidates read their
 *     plan's bound for the rest of the session (until stream_set_grace(-1) with no plan live), which replaces the
 *     captured graphs once.
 *   stream_set_snapshots (ROG solver) pins each plan to the ring as it was at its submit, so that the map keeps
 *     updating while plans solve. n_snapshots >= 1 allocates that many copies of the ring's distance_buffer and its
 *     critical and flat 2-D maps (at the reference's 803 x 803 x 83 ring: 428 MB + 2 x 5.2 MB = 438 MB each); 0 frees
 *     them, and plans read the live ring again, with the launches of a session that never had snapshots. From then on
 *     every stream_submit solves and gates its plan against the ring as it is at the submit: the caller may slide,
 *     update counters, run topay_rogfield_update_esdf or topay_probmap_update between any two calls on the solver
 *     (from the solver's host thread, or serialised with its calls: a submit reads the ring's state and queues its
 *     copy on the ring's stream, so it must not overlap a ring update), and each plan is
 *     bit-identical (results, gate metrics from stream_take, winners) to the same plan solved alone through the batch
 *     API by a ROG solver on the ring as it was then (with grace, set_plans(1, {0, n}, use_gate, G)). Plans submitted
 *     while the ring has not changed share one snapshot; a submit after a change copies the ring (on the ring's
 *     stream) into a snapshot no plan holds, and when every snapshot is held it returns TOPAY_ERR_TOO_LARGE with
 *     nothing changed, as for store rows. A plan holds its snapshot until stream_take, which runs the gate again.
 *     While a submitted plan has not been taken: TOPAY_ERR_NOT_READY; a dense solver or n_snapshots < 0:
 *     TOPAY_ERR_INVALID_ARG. stream_begin starts with snapshots off; stream_end frees them.
 *   stream_end ends the session and drops every plan not taken; the next upload / run gives what a fresh solver gives.
 * Inside a session upload, run, solve_batch, eval, the download calls, select, check_feasible, assign_fields, set_plans,
 * set_timed, set_trace and debug_direction return TOPAY_ERR_NOT_READY, and so do stream calls (stream_set_grace,
 * stream_stop and stream_set_snapshots included) outside one.
 * topay_solver_last_stats counts the session since stream_begin (evals_total: the candidates taken so far).
 * Fields and the ring: in a session of a ROG solver with snapshots on, the library guarantees each plan the ring as it
 * was at its submit. Otherwise a field a live plan reads (the ring of a ROG solver without snapshots, a dense plan's
 * field) must not be rebuilt, slid or updated until that plan has been taken, since stream_take gates it again; the
 * library does not check this. */
int topay_solver_stream_begin(topay_solver* s, int use_gate);
int topay_solver_stream_submit(topay_solver* s, int n_cand, const int32_t* path_len, const double* init_paths,
                               const double* bvel, const double* bacc, topay_field* field, int32_t* plan_id);
int topay_solver_stream_advance(topay_solver* s, int max_batches, int32_t* n_live);
int topay_solver_stream_poll(topay_solver* s, int cap, int32_t* plan_id, int32_t* best_by_duration,
                             int32_t* best_by_cost);
int topay_solver_stream_take(topay_solver* s, int32_t plan_id, int cand, topay_result_batch* out,
                             topay_feasibility* gate);
int topay_solver_stream_set_grace(topay_solver* s, int32_t grace_evals);
int topay_solver_stream_stop(topay_solver* s, int32_t plan_id);
int topay_solver_stream_set_snapshots(topay_solver* s, int n_snapshots);
int topay_solver_stream_end(topay_solver* s);

/* timed != 0: every k_penalty launch is bracketed by CUDA events (stats.ms_eval) and the ticks are
 * plain launches; timed == 0 (default): a batch of 16 ticks is replayed as one CUDA graph, which
 * removes the per-launch host cost that dominates small plans; stats.ms_eval is then 0. */
int topay_solver_set_timed(topay_solver* s, int timed);

/* Optional L-BFGS iterate trace (parity / debugging): when cap > 0 every accepted iteration of
 * every candidate records (f, step, k, line-search evaluations) — the arguments the reference
 * passes to its progress callback (lbfgs.hpp:585-592). cap = 0 turns it off. */
int topay_solver_set_trace(topay_solver* s, int cap);
int topay_solver_download_trace(topay_solver* s, int cand, double* out /*cap x 4*/, int cap, int32_t* len);

/* Developer profiling: accumulated SM clock cycles of the per-candidate kernel's phases
 * (candidate 0) since the last call; enable != 0 switches the counters on. out16 may be NULL. */
int topay_solver_phase_clocks(topay_solver* s, int enable, long long* out16);
/* Developer aid: raw copy of an intermediate device array of the last topay_solver_eval (bit-level A/B
 * runs). which: 0 gnode, 1 gsum, 2 gdC, 3 gdT, 4 tot, 5 Ixy, 6 g. Returns the doubles written or a status. */
int64_t topay_solver_debug_download(topay_solver* s, int which, double* out, int64_t cap);

/* Parity hook for the L-BFGS direction update (lbfgs.hpp:657-710): loads a history into the first slot and runs
 * ONE launch of the L-BFGS kernel in which the line search is accepted, the pair (s, y) = (x - xp, g - gp) enters
 * the ring at slot `end`, and the two-loop recursion over min(bound + 1, m) pairs produces the next search
 * direction d_out[n_vars]. S_rows / Y_rows are [m][n_vars] (row j = pair j of the ring, m = the stage-2 mem_size),
 * ys is [m]; bound pairs are valid, the newest at (end - 1) mod m. Every y_j . s_j must be positive. */
int topay_solver_debug_direction(topay_solver* s, int n_vars, int bound, int end, const double* S_rows,
                                 const double* Y_rows, const double* ys, const double* x, const double* xp,
                                 const double* g, const double* gp, double* d_out, int32_t* bound_out,
                                 int32_t* end_out);

#ifdef __cplusplus
}
#endif
#endif /* TOPAY_B200_H */
