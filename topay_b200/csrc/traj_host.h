// Host-side handle of the trajectory post-processing kernels (traj.cu), shared with solver.cu
// (topay_solver_check_feasible runs them straight on the solver's device buffers).
#pragma once
#include <vector>

#include "common_host.h"

#define TP_NMAXABS 25     // vel, acc, domega, d2omega, q[7], dq[7], d2q[7]
#define TP_NMIN 13        // chassis + 12 spheres

struct TpTrajMeta {
    double total;
    int32_t n_samples, seq_num, n_seq, seq_off;
};

struct TpFeasOut {
    double maxabs[TP_NMAXABS];
    double mins[TP_NMIN];
    int32_t feasible, feasible_print, n_samples, pad;
};

// Device view of n trajectories (all pointers device memory).
struct TpTrajView {
    int n, max_pieces;
    const int32_t* piece_num;   // [n]
    const double* T;            // [n][max_pieces]
    const double* coeff;        // [n][6*max_pieces][9]
    const double* start;        // [n][3]
    const int32_t* idx;         // null, or [n]: trajectory i of the check is entry idx[i] of the arrays above
};

struct TpTrajChecker {
    int device = 0;
    cudaStream_t stream = nullptr;
    double* ttab = nullptr;     // the accumulated 0.01 s sample clock
    int ttab_len = 0;
    TpTrajMeta* meta = nullptr;
    TpFeasOut* feas = nullptr;
    double* car_seq = nullptr;  // pose tables back to back, 4 doubles per entry
    int cap_n = 0;
    size_t cap_seq = 0;
    std::vector<TpTrajMeta> h_meta;
    int checked_n = 0;          // trajectories of the last successful check() (their verdicts are still in `feas`)

    TpTrajChecker() = default;
    TpTrajChecker(const TpTrajChecker&) = delete;
    ~TpTrajChecker();
    int init(int device, cudaStream_t stream);
    // durations, sample counts and the pose tables of the batch (one host round trip for the sizes)
    int prepare(const TpTrajView& V);
    int check(const TpTrajView& V, const TpParams& P, const TpGrid& g, topay_feasibility* out,
              const TpGrid* grids = nullptr, const int32_t* field_of = nullptr);   // per-trajectory fields (sweeps)
    // check() in two steps: the verdicts of V into `feas` on the device (field_of is indexed like V's arrays) ...
    int run(const TpTrajView& V, const TpParams& P, const TpGrid& g, const TpGrid* grids, const int32_t* field_of);
    // ... and the first n of them to the host
    int fetch(int n, topay_feasibility* out);
};
