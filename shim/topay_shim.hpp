// Reference-facing C++ shims over the C ABI: the same class names, member names and argument
// meaning as the reference's GridMap (src/map/include/map/grid_map.h:77-219) and MomaTrajOpt
// (src/planner/include/planner/moma_traj_opt.h:613-675), so that Planner's worker
// (src/planner/src/planner.cpp:847-918) compiles against them unchanged apart from the include.
//
// The reference passes Eigen types; Eigen is not available in this build environment, so the shims
// are templates over "anything with size() and operator[] / operator()(r, c)". With Eigen present,
// Eigen::VectorXd / Eigen::MatrixXd / Eigen::Vector3d satisfy these directly.
#pragma once
#include <cmath>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <array>
#include <vector>

#include "../include/topay_b200.h"

namespace rog_map {
class ESDFMap;   // below: MomaTrajOpt can be built over the ROG-Map ring
}

namespace nmoma_planner {

inline void topay_check(int rc, const char* what) {
    if (rc != TOPAY_OK) throw std::runtime_error(std::string(what) + ": " + topay_last_error());
}

// MomaTraj (moma_traj_opt.h:26-247): durations + MINCO coefficients of one optimised trajectory; the
// pose table and the state samplers are evaluated on the device.
struct MomaTraj {
    bool is_init = false;
    std::vector<double> durations;          // N
    std::vector<double> coeff;              // 6N x 9, row 6i+k = coefficient of t^k of piece i
    double start_se2[3] = {0, 0, 0};
    int device = 0;
    double getTotalDuration() const {
        double s = 0;
        for (double d : durations) s += d;
        return s;
    }
    int getPieceNum() const { return (int)durations.size(); }
    topay_traj_batch view(int32_t* piece_num) const {
        *piece_num = getPieceNum();
        topay_traj_batch b;
        b.n_traj = 1; b.max_pieces = getPieceNum(); b.piece_num = piece_num;
        b.T = durations.data(); b.coeff = coeff.data(); b.start_se2 = start_se2;
        return b;
    }
    // std::vector<Eigen::Vector4d> car_seq (moma_traj_opt.h:36, 38-68): rows x, y, yaw, t
    std::vector<double> car_seq() const {
        int32_t pn, len = 0;
        topay_traj_batch b = view(&pn);
        const int cap = (int)(getTotalDuration() / 0.1) + 4;
        std::vector<double> out((size_t)cap * 4);
        topay_check(topay_traj_car_seq(device, &b, cap, out.data(), &len), "topay_traj_car_seq");
        out.resize((size_t)len * 4);
        return out;
    }
    // Eigen::VectorXd getState(double t) const (moma_traj_opt.h:121): x, y, yaw, q1..q7
    std::vector<double> getState(double t) const {
        int32_t pn;
        topay_traj_batch b = view(&pn);
        std::vector<double> st(10);
        topay_check(topay_traj_sample(device, &b, &t, 1, st.data(), nullptr), "topay_traj_sample");
        return st;
    }
    // Eigen::VectorXd getDState(double t) const (moma_traj_opt.h:151): v, omega, 0, dq1..dq7
    std::vector<double> getDState(double t) const {
        int32_t pn;
        topay_traj_batch b = view(&pn);
        std::vector<double> ds(10);
        topay_check(topay_traj_sample(device, &b, &t, 1, nullptr, ds.data()), "topay_traj_sample");
        return ds;
    }
    // many times in one launch: states is m x 10
    void getStateBatch(const double* t, int m, double* states) const {
        int32_t pn;
        topay_traj_batch b = view(&pn);
        topay_check(topay_traj_sample(device, &b, t, m, states, nullptr), "topay_traj_sample");
    }
};

class GridMap {
public:
    typedef std::shared_ptr<GridMap> Ptr;
    double resolution = 0, resolution_inv = 0;
    int voxel_num[3] = {0, 0, 0};
    bool use_rog = false;

    // GridMap::init (grid_map.cpp:6-87) with the rosparams passed explicitly.
    void init(double map_size_x, double map_size_y, double map_size_z, double res, int device = 0) {
        topay_grid_desc d = {};
        d.map_size[0] = map_size_x; d.map_size[1] = map_size_y; d.map_size[2] = map_size_z;
        d.resolution = res; d.chassis_colli_radius = 0.4; d.chassis_height = 0.155;
        topay_check(topay_field_create(&d, device, &f_), "topay_field_create");
        int32_t dims[3];
        topay_field_dims(f_, dims);
        for (int i = 0; i < 3; i++) voxel_num[i] = dims[i];
        resolution = res; resolution_inv = 1.0 / res;
        map_origin[0] = -map_size_x / 2.0; map_origin[1] = -map_size_y / 2.0; map_origin[2] = 0.0;   // grid_map.cpp:41-47
    }
    GridMap() = default;
    GridMap(const GridMap&) = delete;               // owns the device field
    GridMap& operator=(const GridMap&) = delete;
    ~GridMap() { topay_field_destroy(f_); }

    void loadMap(const std::vector<char>& occ_2d, const std::vector<char>& occ_3d) {      // grid_map.cpp:800
        topay_check(topay_field_set_occupancy(f_, (const int8_t*)occ_3d.data(), (const int8_t*)occ_2d.data(), nullptr),
                    "topay_field_set_occupancy");
        updateESDF();
    }
    // ingest half of regenerateMap / cloudCallback (grid_map.cpp:716-750, 543-578)
    void regenerateMap(const float* xyz, int64_t n_points) {
        topay_check(topay_field_clear(f_, 0), "topay_field_clear");
        topay_check(topay_field_rasterize_points(f_, xyz, n_points), "topay_field_rasterize_points");
        updateESDF();
    }
    void updateESDF() { topay_check(topay_field_rebuild(f_), "topay_field_rebuild"); map_ready_ = true; }
    bool mapReady() const { return map_ready_; }

    template <class V3> void getDisWithGradI3d(const V3& pos, double& distance, V3& grad) {   // grid_map.h:443
        double p[3] = {pos[0], pos[1], pos[2]}, g[3];
        topay_check(topay_field_query3d(f_, p, 1, &distance, g), "topay_field_query3d");
        grad[0] = g[0]; grad[1] = g[1]; grad[2] = g[2];
    }
    template <class V2> void getDisWithGradI2d(const V2& pos, double& distance, V2& grad, bool inflate = false,
                                               bool critical = false) {                      // grid_map.h:364
        double p[2] = {pos[0], pos[1]}, g[2];
        const int which = critical ? TOPAY_MAP2D_CRITICAL : (inflate ? TOPAY_MAP2D_INFLATE : TOPAY_MAP2D_FLAT);
        topay_check(topay_field_query2d(f_, p, 1, which, &distance, g), "topay_field_query2d");
        grad[0] = g[0]; grad[1] = g[1];
    }
    template <class V3> void getDistance3d(const V3& pos, double& distance) {                   // grid_map.h:307
        double p[3] = {pos[0], pos[1], pos[2]};
        topay_check(topay_field_distance3d(f_, p, 1, &distance), "topay_field_distance3d");
    }
    template <class V2> void getDistance2d(const V2& pos, double& distance) {                   // grid_map.h:256
        double p[2] = {pos[0], pos[1]};
        topay_check(topay_field_distance2d(f_, p, 1, &distance), "topay_field_distance2d");
    }
    template <class V> bool isWholeBodyCollision(const V& state) {                               // grid_map.h:613
        double s[10];
        for (int i = 0; i < 10; i++) s[i] = state[i];
        topay_robot_params rp;
        topay_robot_params_default(&rp);
        int8_t out = 1;
        topay_check(topay_field_whole_body_collision(f_, &rp, s, 1, &out), "topay_field_whole_body_collision");
        return out != 0;
    }
    template <class V2> bool isCollision2d(const V2& pos, double threshold) {                    // grid_map.h:511
        double p[2] = {pos[0], pos[1]};
        int8_t out = 1;
        topay_check(topay_field_is_collision2d(f_, p, 1, threshold, &out), "topay_field_is_collision2d");
        return out != 0;
    }
    template <class V3> bool isCollision3d(const V3& pos, double threshold) {                    // grid_map.h:695
        double p[3] = {pos[0], pos[1], pos[2]};
        int8_t out = 1;
        topay_check(topay_field_is_collision3d(f_, p, 1, threshold, &out), "topay_field_is_collision3d");
        return out != 0;
    }
    template <class V2> bool isLineCollisionGrid2d(const V2& p1, const V2& p2, double threshold = 0.0) {   // grid_map.h:565
        double a[2] = {p1[0], p1[1]}, b[2] = {p2[0], p2[1]};
        int8_t out = 1;
        topay_check(topay_field_is_line_collision_grid2d(f_, a, b, 1, threshold, &out), "is_line_collision_grid2d");
        return out != 0;
    }
    template <class V2> double getDistCoarse2d(const V2& pos, bool critical = false) {           // grid_map.h:887
        double p[2] = {pos[0], pos[1]}, d = 0;
        topay_check(topay_field_dist_coarse2d(f_, p, 1, critical, &d), "topay_field_dist_coarse2d");
        return d;
    }
    template <class V2i> double getDistCoarse2i(const V2i& id, bool critical = false) {          // grid_map.h:914
        int32_t i2[2] = {(int32_t)id[0], (int32_t)id[1]};
        double d = 0;
        topay_check(topay_field_dist_coarse2i(f_, i2, 1, critical, &d), "topay_field_dist_coarse2i");
        return d;
    }
    // TopologyPRM::lineVisib (topo_prm.cpp:278-315; the PRM's guard / connection / shortcut visibility test) on this
    // field: single segment, and the batched form (one launch for all rays of a roadmap pass)
    template <class V3> bool lineVisib(const V3& p1, const V3& p2, double thresh, V3& pc, bool use_critical = false) {
        double a[3] = {p1[0], p1[1], p1[2]}, b[3] = {p2[0], p2[1], p2[2]}, c[3] = {pc[0], pc[1], pc[2]};
        int8_t vis = 0;
        topay_check(topay_field_line_visible(f_, a, b, 1, thresh, use_critical, &vis, c), "topay_field_line_visible");
        pc[0] = c[0]; pc[1] = c[1]; pc[2] = c[2];
        return vis != 0;
    }
    void lineVisibBatch(const double* p1, const double* p2, int64_t n, double thresh, bool use_critical, int8_t* visible,
                        double* pc) {
        topay_check(topay_field_line_visible(f_, p1, p2, n, thresh, use_critical, visible, pc), "topay_field_line_visible");
    }
    // TopologyPRM::sameTopoPath (topo_prm.cpp:424-448) for many pairs in one launch (pruneEquivalent)
    void sameTopoPaths(const double* pts, const int32_t* offsets, int n_paths, const int32_t* pairs, int n_pairs,
                       double thresh, bool use_critical, int8_t* same) {
        topay_check(topay_field_same_topo_paths(f_, pts, offsets, n_paths, pairs, n_pairs, thresh, use_critical, same),
                    "topay_field_same_topo_paths");
    }
    // batched forms for the front-end (one launch for many samples)
    void isWholeBodyCollisionBatch(const double* states, int64_t n, int8_t* out) {
        topay_robot_params rp;
        topay_robot_params_default(&rp);
        topay_check(topay_field_whole_body_collision(f_, &rp, states, n, out), "topay_field_whole_body_collision");
    }
    void getDisWithGradI3dBatch(const double* pos, int64_t n, double* dist, double* grad) {
        topay_check(topay_field_query3d(f_, pos, n, dist, grad), "topay_field_query3d");
    }
    std::vector<double> getESDFBuffer3d() {                                                      // grid_map.h:217
        std::vector<double> b((size_t)voxel_num[0] * voxel_num[1] * voxel_num[2]);
        topay_check(topay_field_download(f_, TOPAY_MAP3D, b.data()), "topay_field_download");
        return b;
    }
    std::vector<double> getESDFBuffer2d() {                                                      // grid_map.h:216
        std::vector<double> b((size_t)voxel_num[0] * voxel_num[1]);
        topay_check(topay_field_download(f_, TOPAY_MAP2D_FLAT, b.data()), "topay_field_download");
        return b;
    }
    // index helpers, pure host arithmetic (grid_map.h:727-885, dense branch)
    template <class V3, class V3i> void posToIndex3d(const V3& pos, V3i& id) const {
        for (int i = 0; i < 3; i++) id[i] = (int)std::floor((pos[i] - map_origin[i]) * resolution_inv);
    }
    template <class V2, class V2i> void posToIndex2d(const V2& pos, V2i& id) const {
        for (int i = 0; i < 2; i++) id[i] = (int)std::floor((pos[i] - map_origin[i]) * resolution_inv);
    }
    template <class V3i, class V3> void indexToPos3d(const V3i& id, V3& pos) const {
        for (int i = 0; i < 3; i++) pos[i] = (id[i] + 0.5) * resolution + map_origin[i];
    }
    template <class V2i, class V2> void indexToPos2d(const V2i& id, V2& pos) const {
        for (int i = 0; i < 2; i++) pos[i] = (id[i] + 0.5) * resolution + map_origin[i];
    }
    template <class V3i> void boundIndex3d(V3i& id) const {
        for (int i = 0; i < 3; i++) id[i] = id[i] < 0 ? 0 : (id[i] > voxel_num[i] - 1 ? voxel_num[i] - 1 : id[i]);
    }
    template <class V2i> void boundIndex2d(V2i& id) const {
        for (int i = 0; i < 2; i++) id[i] = id[i] < 0 ? 0 : (id[i] > voxel_num[i] - 1 ? voxel_num[i] - 1 : id[i]);
    }
    double map_origin[3] = {0, 0, 0};
    topay_field* handle() const { return f_; }

private:
    topay_field* f_ = nullptr;
    bool map_ready_ = false;
};

// JPS::GraphSearch::getDensePath (graph_search.cpp:119-176): rows (x, y, theta, dt) as std::array<double, 4>.
namespace JPS {
struct GraphSearch {
    template <class V2>
    static std::vector<std::array<double, 4>> getDensePath(const std::vector<V2>& raw_path, double step_size,
                                                           double start_yaw, double end_yaw, double v_max,
                                                           double w_max) {
        std::vector<double> raw;
        for (const auto& p : raw_path) {
            raw.push_back(p[0]);
            raw.push_back(p[1]);
        }
        std::vector<std::array<double, 4>> out(64);
        for (;;) {
            const int n = topay_dense_path(raw.data(), (int)raw_path.size(), step_size, start_yaw, end_yaw, v_max, w_max,
                                           &out[0][0], (int)out.size());
            if (n < 0) topay_check(n, "topay_dense_path");
            const bool fits = n <= (int)out.size();
            out.resize(n);
            if (fits) return out;
        }
    }
};
}  // namespace JPS


class MomaTrajOpt {
public:
    typedef std::shared_ptr<MomaTrajOpt> Ptr;
    topay_opt_params opt_param;          // MomaTrajOptParam (moma_traj_opt.h:553-564)
    double traj_cost = 0.0;

    // max_cand > 1 turns the instance into the batched optimizer that replaces the <= 8
    // per-thread instances of planner.cpp:59-66.
    explicit MomaTrajOpt(GridMap::Ptr grid_map_, int max_cand = 1, int max_pieces = 32)
        : grid_map(grid_map_), max_cand_(max_cand), max_pieces_(max_pieces) {
        topay_opt_params_default(&opt_param);
        topay_robot_params_default(&moma_param);
    }
    // GridMap with use_rog (grid_map.h:90): the solve and the gate read the ROG-Map ring
    explicit MomaTrajOpt(std::shared_ptr<rog_map::ESDFMap> esdf_map, int max_cand = 1, int max_pieces = 32)
        : esdf_map_(esdf_map), max_cand_(max_cand), max_pieces_(max_pieces) {
        topay_opt_params_default(&opt_param);
        topay_robot_params_default(&moma_param);
    }
    MomaTrajOpt(const MomaTrajOpt&) = delete;       // owns the device solver
    MomaTrajOpt& operator=(const MomaTrajOpt&) = delete;
    ~MomaTrajOpt() { topay_solver_destroy(s_); }

    // void init(ros::NodeHandle&) reads the rosparams into opt_param (moma_traj_opt.h:845-941); here the
    // caller fills opt_param (defaults = params/optimizer.yaml) and then calls init().
    void init() {
        if (esdf_map_)
            topay_check(topay_solver_create_rog(&opt_param, &moma_param, ring(), max_cand_, max_pieces_, &s_),
                        "topay_solver_create_rog");
        else
            topay_check(topay_solver_create(&opt_param, &moma_param, grid_map->handle(), max_cand_, max_pieces_, &s_),
                        "topay_solver_create");
    }
    bool useRog() const { return esdf_map_ != nullptr; }

    // bool optimizeTraj(std::vector<Eigen::VectorXd> init_path, const Eigen::MatrixXd& boundary_vel,
    //                   const Eigen::MatrixXd& boundary_acc)          (moma_traj_opt.cpp:142)
    template <class Path, class Mat>
    bool optimizeTraj(const Path& init_path, const Mat& boundary_vel, const Mat& boundary_acc) {
        std::vector<std::vector<double>> flat(1);
        for (const auto& wp : init_path)
            for (int d = 0; d < 10; d++) flat[0].push_back(wp[d]);
        double bv[20], ba[20];
        for (int r = 0; r < 10; r++)
            for (int c = 0; c < 2; c++) { bv[r * 2 + c] = boundary_vel(r, c); ba[r * 2 + c] = boundary_acc(r, c); }
        std::vector<int> ok = optimizeTrajBatch(flat, bv, ba);
        return ok[0] != 0;
    }
    // All candidates of a plan at once: paths[c] is a flattened (len x 10) waypoint list; bvel / bacc are
    // n x 10 x 2 row-major. Returns the per-candidate success flags; best index by the reference's
    // shortest-duration rule (planner.cpp:999-1010) in best_by_duration.
    std::vector<int> optimizeTrajBatch(const std::vector<std::vector<double>>& paths, const double* bvel,
                                       const double* bacc) {
        const int n = (int)paths.size();
        std::vector<int32_t> len(n);
        std::vector<double> all;
        for (int c = 0; c < n; c++) {
            len[c] = (int32_t)(paths[c].size() / 10);
            all.insert(all.end(), paths[c].begin(), paths[c].end());
        }
        status_.assign(n, 0); pieces_.assign(n, 0); cost_.assign(n, 0.0);
        T_.assign((size_t)n * max_pieces_, 0.0);
        coeff_.assign((size_t)n * 6 * max_pieces_ * 9, 0.0);
        starts_.assign((size_t)n * 3, 0.0);
        for (int c = 0; c < n; c++)
            for (int d = 0; d < 3; d++) starts_[c * 3 + d] = paths[c][d];
        topay_result_batch out = {};
        out.status = status_.data(); out.piece_num = pieces_.data(); out.cost = cost_.data();
        out.T = T_.data(); out.coeff = coeff_.data();
        if (grace_evals_ < 0) {
            topay_check(topay_solver_solve_batch(s_, n, len.data(), all.data(), bvel, bacc, &out, &best_by_duration,
                                                 &best_by_cost), "topay_solver_solve_batch");
        } else {   // the batch is one plan: its first success + grace under the planner's success test
            topay_check(topay_solver_upload(s_, n, len.data(), all.data(), bvel, bacc), "topay_solver_upload");
            const int32_t off[2] = {0, n};
            topay_check(topay_solver_set_plans(s_, 1, off, 1, grace_evals_), "topay_solver_set_plans");
            topay_check(topay_solver_run(s_), "topay_solver_run");
            topay_check(topay_solver_download(s_, &out, &best_by_duration, &best_by_cost), "topay_solver_download");
        }
        traj_cost = cost_[0];
        return std::vector<int>(status_.begin(), status_.end());
    }
    // First success + grace of the planner's worker pool (planner.cpp:931-952), counted in evaluations: from the next
    // optimizeTrajBatch on, once a candidate passes optimizeTraj && printConstraintsSituations, the candidates that
    // need more than `evals` evaluations beyond it are cancelled (status 0, TOPAY_LBFGSERR_PLAN_GRACE), and
    // selectFeasible sees them as failed. evals < 0 turns it off (the default).
    void setGrace(int evals) {
        if (evals < 0 && grace_evals_ >= 0) topay_check(topay_solver_set_plans(s_, 0, nullptr, 0, 0), "topay_solver_set_plans");
        grace_evals_ = evals < 0 ? -1 : evals;
    }
    // MomaTraj getTraj() const (moma_traj_opt.h:943-946)
    MomaTraj getTraj(int idx = 0) const {
        MomaTraj t;
        const int N = pieces_[idx];
        t.durations.assign(T_.begin() + (size_t)idx * max_pieces_, T_.begin() + (size_t)idx * max_pieces_ + N);
        const size_t o = (size_t)idx * 6 * max_pieces_ * 9;
        t.coeff.assign(coeff_.begin() + o, coeff_.begin() + o + (size_t)6 * N * 9);
        for (int d = 0; d < 3; d++) t.start_se2[d] = starts_[idx * 3 + d];
        t.is_init = true;
        return t;
    }
    // bool checkFeasible(MomaTraj traj) (moma_traj_opt.h:948-1045)
    bool checkFeasible(const MomaTraj& traj) { return gate(traj, false); }
    // bool printConstraintsSituations(MomaTraj traj) (moma_traj_opt.h:1047-1210); the accumulated
    // metrics of the last call stay in `constraints`
    bool printConstraintsSituations(const MomaTraj& traj) { return gate(traj, true); }
    struct Constraints {
        double max_vel, max_acc, max_domega, max_d2omega, max_q[7], max_dq[7], max_d2q[7], min_dist, min_dist_mani[12];
        int32_t n_samples;
    } constraints;
    // The worker's gate for every candidate of the last optimizeTrajBatch, on the device:
    // optimizeTraj && printConstraintsSituations (planner.cpp:877-880), then the shortest duration
    // (planner.cpp:999-1010). Returns the winner or -1; success[c] is the gate per candidate.
    int selectFeasible(std::vector<int>* success = nullptr) {
        const int n = (int)status_.size();
        std::vector<int32_t> f(n), fp(n);
        topay_feasibility out = {};
        out.feasible = f.data(); out.feasible_print = fp.data();
        int32_t best = -1;
        topay_check(topay_solver_check_feasible(s_, &out, &best), "topay_solver_check_feasible");
        if (success) {
            success->resize(n);
            for (int c = 0; c < n; c++) (*success)[c] = status_[c] == 1 && fp[c];
        }
        return best;
    }
    int32_t best_by_duration = -1, best_by_cost = -1;

    // scenario sweeps: candidate c of the uploaded batch is solved and gated against fields[field_of[c]]
    void assignFields(const std::vector<GridMap*>& fields, const std::vector<int32_t>& field_of) {
        std::vector<topay_field*> h;
        for (GridMap* g : fields) h.push_back(g->handle());
        topay_check(topay_solver_assign_fields(s_, h.data(), (int)h.size(), field_of.data()), "topay_solver_assign_fields");
    }

    // Streaming session (topay_solver_stream_*): plans are submitted while the solve runs, and each plan's winners
    // come back as soon as that plan is done — the worker pool of planner.cpp:921-952 with plans arriving while it
    // works. The batch calls above are refused between streamBegin and streamEnd.
    struct StreamDone { int32_t plan_id, best_by_duration, best_by_cost; };
    // grace_evals >= 0: first success + grace for every plan of the session (setGrace's rule; -1: off).
    // snapshots >= 1 (ROG solver): streamSetSnapshots.
    void streamBegin(bool use_gate = true, int grace_evals = -1, int snapshots = 0) {
        topay_check(topay_solver_stream_begin(s_, use_gate ? 1 : 0), "topay_solver_stream_begin");
        stream_starts_.clear();
        if (grace_evals >= 0) topay_check(topay_solver_stream_set_grace(s_, grace_evals), "topay_solver_stream_set_grace");
        if (snapshots > 0) streamSetSnapshots(snapshots);
    }
    // ROG solver: every plan submitted from now on is solved and gated against the ring as it is at the submit, so
    // the ProbMap may keep updating it; up to n ring states are held by untaken plans at once (0: the live ring).
    void streamSetSnapshots(int n) {
        topay_check(topay_solver_stream_set_snapshots(s_, n), "topay_solver_stream_set_snapshots");
    }
    // Cancels a live plan's remaining candidates (planner.cpp:952's interrupt_all); streamPoll reports it as usual.
    void streamStop(int32_t plan_id) { topay_check(topay_solver_stream_stop(s_, plan_id), "topay_solver_stream_stop"); }
    // One plan (paths, bvel and bacc as in optimizeTrajBatch); `field` (nullptr: the solver's own) must stay as it is
    // until the plan is taken (a ROG solver with snapshots: the ring may change). Returns the plan id.
    int32_t streamSubmit(const std::vector<std::vector<double>>& paths, const double* bvel, const double* bacc,
                         GridMap* field = nullptr) {
        const int n = (int)paths.size();
        std::vector<int32_t> len(n);
        std::vector<double> all, starts;
        for (int c = 0; c < n; c++) {
            len[c] = (int32_t)(paths[c].size() / 10);
            all.insert(all.end(), paths[c].begin(), paths[c].end());
            starts.insert(starts.end(), paths[c].begin(), paths[c].begin() + 3);
        }
        int32_t id = -1;
        topay_check(topay_solver_stream_submit(s_, n, len.data(), all.data(), bvel, bacc,
                                               field ? field->handle() : nullptr, &id), "topay_solver_stream_submit");
        stream_starts_[id] = starts;
        return id;
    }
    // Runs up to max_batches batches of 16 ticks; returns the candidates still in the slots (0: every plan is done).
    int streamAdvance(int max_batches = 1) {
        int32_t live = 0;
        topay_check(topay_solver_stream_advance(s_, max_batches, &live), "topay_solver_stream_advance");
        return live;
    }
    // The plans that finished since the last call, with their winners (index inside the plan, -1: none).
    std::vector<StreamDone> streamPoll() {
        std::vector<int32_t> id(max_cand_), bd(max_cand_), bc(max_cand_);
        const int k = topay_solver_stream_poll(s_, max_cand_, id.data(), bd.data(), bc.data());
        if (k < 0) topay_check(k, "topay_solver_stream_poll");
        std::vector<StreamDone> out;
        for (int i = 0; i < k; i++) out.push_back(StreamDone{id[i], bd[i], bc[i]});
        return out;
    }
    // Takes a finished plan's candidates (all of them, or only `cand`): getTraj(i) then returns the i-th one taken.
    // The plan's id is free afterwards.
    void streamTake(int32_t plan_id, int cand = -1) {
        auto it = stream_starts_.find(plan_id);
        if (it == stream_starts_.end()) topay_check(TOPAY_ERR_INVALID_ARG, "topay_solver_stream_take");
        const int n = cand < 0 ? (int)it->second.size() / 3 : 1;
        status_.assign(n, 0); pieces_.assign(n, 0); cost_.assign(n, 0.0);
        T_.assign((size_t)n * max_pieces_, 0.0);
        coeff_.assign((size_t)n * 6 * max_pieces_ * 9, 0.0);
        topay_result_batch out = {};
        out.status = status_.data(); out.piece_num = pieces_.data(); out.cost = cost_.data();
        out.T = T_.data(); out.coeff = coeff_.data();
        topay_check(topay_solver_stream_take(s_, plan_id, cand, &out, nullptr), "topay_solver_stream_take");
        starts_.assign(it->second.begin() + (cand < 0 ? 0 : 3 * cand),
                       it->second.begin() + (cand < 0 ? it->second.size() : 3 * cand + 3));
        stream_starts_.erase(it);
        traj_cost = cost_[0];
    }
    void streamEnd() {
        topay_check(topay_solver_stream_end(s_), "topay_solver_stream_end");
        stream_starts_.clear();
    }
private:
    bool gate(const MomaTraj& traj, bool print_rule) {
        int32_t pn, f = 0, fp = 0;
        topay_traj_batch b = traj.view(&pn);
        topay_feasibility out = {};
        out.feasible = &f; out.feasible_print = &fp; out.n_samples = &constraints.n_samples;
        out.max_vel = &constraints.max_vel; out.max_acc = &constraints.max_acc;
        out.max_domega = &constraints.max_domega; out.max_d2omega = &constraints.max_d2omega;
        out.max_q = constraints.max_q; out.max_dq = constraints.max_dq; out.max_d2q = constraints.max_d2q;
        out.min_dist = &constraints.min_dist; out.min_dist_mani = constraints.min_dist_mani;
        if (esdf_map_)
            topay_check(topay_traj_check_feasible_rog(ring(), &moma_param, &b, &out), "topay_traj_check_feasible_rog");
        else
            topay_check(topay_traj_check_feasible(grid_map->handle(), &moma_param, &b, &out), "topay_traj_check_feasible");
        return (print_rule ? fp : f) != 0;
    }
    topay_rogfield* ring() const;   // esdf_map_'s handle (defined after rog_map::ESDFMap)
    topay_robot_params moma_param;
    GridMap::Ptr grid_map;
    std::shared_ptr<rog_map::ESDFMap> esdf_map_;   // set instead of grid_map: GridMap's use_rog
    topay_solver* s_ = nullptr;
    int max_cand_, max_pieces_;
    int grace_evals_ = -1;
    std::vector<int32_t> status_, pieces_;
    std::vector<double> cost_, T_, coeff_, starts_;
    std::map<int32_t, std::vector<double>> stream_starts_;   // start poses of the submitted plans, by plan id
};

}  // namespace nmoma_planner

namespace rog_map {

// rog_map::ESDFMap (src/rog_map/include/rog_map/esdf_map.h:34-93) with the SlidingMap / CounterMap members
// the planner side uses; positions are "anything with operator[]".
class ESDFMap {
public:
    typedef std::shared_ptr<ESDFMap> Ptr;
    ESDFMap() = default;
    ESDFMap(const ESDFMap&) = delete;               // owns the device ring
    ESDFMap& operator=(const ESDFMap&) = delete;
    ~ESDFMap() { topay_rogfield_destroy(f_); }
    // initESDFMap (esdf_map.cpp:28-57); sliding_thresh is the caller's business (prob_map.cpp:292-298)
    template <class V3i, class V3>
    void initESDFMap(const V3i& half_prob_map_size_i, double prob_map_resolution, double temp_counter_map_resolution,
                     const V3& local_update_box, bool map_sliding_en, double /*sliding_thresh*/,
                     const V3& fix_map_origin, double unk_thresh, int device = 0) {
        topay_rog_desc d = {};
        for (int i = 0; i < 3; i++) {
            d.half_prob_map_size_i[i] = half_prob_map_size_i[i];
            d.local_update_box[i] = local_update_box[i];
            d.fix_map_origin[i] = fix_map_origin[i];
        }
        d.prob_resolution = prob_map_resolution; d.esdf_resolution = temp_counter_map_resolution;
        d.map_sliding_en = map_sliding_en; d.unk_thresh = unk_thresh;
        nmoma_planner::topay_check(topay_rogfield_create(&d, device, &f_), "topay_rogfield_create");
    }
    template <class V3> void mapSliding(const V3& odom) {                                   // sliding_map.cpp:113
        double o[3] = {odom[0], odom[1], odom[2]};
        nmoma_planner::topay_check(topay_rogfield_slide(f_, o), "topay_rogfield_slide");
    }
    template <class V3> void updateGridCounter(const V3& pos, int from_type, int to_type) {  // counter_map.cpp:94
        double p[3] = {pos[0], pos[1], pos[2]};
        uint8_t a = (uint8_t)from_type, b = (uint8_t)to_type;
        nmoma_planner::topay_check(topay_rogfield_update_counters(f_, p, &a, &b, 1), "topay_rogfield_update_counters");
    }
    void updateGridCounterBatch(const double* pos, const uint8_t* from_type, const uint8_t* to_type, int64_t n) {
        nmoma_planner::topay_check(topay_rogfield_update_counters(f_, pos, from_type, to_type, n), "update_counters");
    }
    template <class V3> void updateESDF3D(const V3& cur_odom) {                             // esdf_map.cpp:154
        double o[3] = {cur_odom[0], cur_odom[1], cur_odom[2]};
        nmoma_planner::topay_check(topay_rogfield_update_esdf(f_, o), "topay_rogfield_update_esdf");
    }
    template <class V3> void evaluateEDT(const V3& pos, double& dist) { q(TOPAY_ROG_Q_EDT, pos, dist, (V3*)nullptr); }
    template <class V3> void evaluateFirstGrad(const V3& pos, V3& grad) { double d; q(TOPAY_ROG_Q_EDT, pos, d, &grad); }
    template <class V3> void getValueGrad(const V3& pos, double& dist, V3& grad) { q(TOPAY_ROG_Q_EDT, pos, dist, &grad); }
    template <class V3> void getValueGrad2d(const V3& pos, double& dist, V3& grad) { q(TOPAY_ROG_Q_FLAT, pos, dist, &grad); }
    template <class V3> void getCriticalValueGrad(const V3& pos, double& dist, V3& grad) { q(TOPAY_ROG_Q_CRITICAL, pos, dist, &grad); }
    template <class V3> double getDistance(const V3& pos) { double d; q(TOPAY_ROG_Q_CELL, pos, d, (V3*)nullptr); return d; }
    template <class V3> double getDistance2d(const V3& pos) { double d; q(TOPAY_ROG_Q_CELL_FLAT, pos, d, (V3*)nullptr); return d; }
    template <class V3> double getCriticalDistance(const V3& pos) { double d; q(TOPAY_ROG_Q_CELL_CRITICAL, pos, d, (V3*)nullptr); return d; }
    template <class V2> bool isLineFree2d(const V2& start, const V2& end, double threshold = 0.0) {   // esdf_map.cpp:122
        double a[2] = {start[0], start[1]}, b[2] = {end[0], end[1]};
        int8_t out = 0;
        nmoma_planner::topay_check(topay_rogfield_is_line_free2d(f_, a, b, 1, threshold, &out), "is_line_free2d");
        return out != 0;
    }
    topay_rogfield* handle() const { return f_; }

private:
    template <class V3> void q(int kind, const V3& pos, double& dist, V3* grad) {
        double p[3] = {pos[0], pos[1], pos[2]}, g[3] = {0, 0, 0};
        nmoma_planner::topay_check(topay_rogfield_query(f_, kind, p, 1, &dist, grad ? g : nullptr), "topay_rogfield_query");
        if (grad) { (*grad)[0] = g[0]; (*grad)[1] = g[1]; (*grad)[2] = g[2]; }
    }
    topay_rogfield* f_ = nullptr;
};

// rog_map::ProbMap (src/rog_map/include/rog_map/prob_map.h:34-160): the probabilistic occupancy layer over an
// ESDFMap. cfg is filled by the caller as Config's constructor would from the rosparams (config.hpp:160-262).
class ProbMap {
public:
    typedef std::shared_ptr<ProbMap> Ptr;
    topay_prob_desc cfg_ = {};
    ESDFMap::Ptr esdf_map_;
    ProbMap() = default;
    ProbMap(const ProbMap&) = delete;               // owns the device ring
    ProbMap& operator=(const ProbMap&) = delete;
    ~ProbMap() { topay_probmap_destroy(m_); }
    // initProbMap (prob_map.cpp:25-88): the grid geometry is the ESDFMap's descriptor
    void initProbMap(ESDFMap::Ptr esdf_map) {
        esdf_map_ = esdf_map;
        nmoma_planner::topay_check(topay_probmap_create(esdf_map->handle(), &cfg_, &m_), "topay_probmap_create");
    }
    // updateProbMap(cloud, pose) (prob_map.cpp:302-373); cloud_xyzi: n x (x, y, z, intensity) float32
    template <class V3> void updateProbMap(const float* cloud_xyzi, int64_t n, const V3& pose_pos) {
        double p[3] = {pose_pos[0], pose_pos[1], pose_pos[2]};
        nmoma_planner::topay_check(topay_probmap_update(m_, cloud_xyzi, n, p), "topay_probmap_update");
    }
    topay_probmap* handle() const { return m_; }

private:
    topay_probmap* m_ = nullptr;
};

}  // namespace rog_map

inline topay_rogfield* nmoma_planner::MomaTrajOpt::ring() const { return esdf_map_->handle(); }
