"""The C++ shim's ROG path compiles with the host compiler alone: a MomaTrajOpt built over a rog_map::ESDFMap fed by a
ProbMap, streaming with ring snapshots and gating a trajectory on the ring (GridMap's use_rog, grid_map.h:90)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r"""
#include <array>
#include <memory>
#include <vector>

#include "topay_shim.hpp"

using namespace nmoma_planner;

// A replanning loop: the ProbMap keeps updating the ring while plans solve, each plan pinned to the ring of its
// submit; the trajectory being executed is checked against the ring as it is now.
int replan(std::shared_ptr<rog_map::ESDFMap> esdf, rog_map::ProbMap& prob, const float* cloud, int64_t n_points,
           const std::vector<std::vector<double>>& paths, const double* bvel, const double* bacc) {
    MomaTrajOpt opt(esdf, /*max_cand=*/16, /*max_pieces=*/16);
    opt.init();
    if (!opt.useRog()) return -1;
    opt.streamBegin(/*use_gate=*/true, /*grace_evals=*/8, /*snapshots=*/2);
    const int32_t a = opt.streamSubmit(paths, bvel, bacc);
    const std::array<double, 3> pose = {0.0, 0.0, 0.4};
    prob.updateProbMap(cloud, n_points, pose);
    const int32_t b = opt.streamSubmit(paths, bvel, bacc);
    int winner = -1, taken = 0;
    for (int k = 0; k < 1000 && taken < 2; k++) {
        opt.streamAdvance(1);
        for (const MomaTrajOpt::StreamDone& d : opt.streamPoll()) {
            opt.streamTake(d.plan_id);
            taken++;
            if (d.plan_id == a || d.plan_id == b) winner = d.best_by_duration;
        }
    }
    opt.streamEnd();
    opt.streamBegin(true);
    opt.streamSetSnapshots(0);
    opt.streamEnd();
    if (winner < 0) return -1;
    const MomaTraj traj = opt.getTraj(winner);
    return opt.checkFeasible(traj) && opt.printConstraintsSituations(traj) ? winner : -1;
}
"""


def test_rog_shim_streams_with_snapshots_and_compiles(tmp_path):
    src = tmp_path / "rog_worker.cpp"
    src.write_text(WORKER)
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "shim"), str(src)])
