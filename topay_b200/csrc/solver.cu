// Host side of topay_solver: allocation, candidate upload, the tick loop and downloads.
// Replaces the per-thread MomaTrajOpt instances of the reference
// (src/planner/src/planner.cpp:59-66, 847-918) with one batched device solve.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <ctime>
#include <map>
#include <string>
#include <vector>

#include "common_host.h"
#include "solver_kernels.cuh"
#include "traj_host.h"

#include <atomic>

// solves in flight in this process (plans driven by concurrent host threads)
static std::atomic<int> g_solves_running{0};
struct TpRunningGuard {
    int concurrent;
    TpRunningGuard() : concurrent(++g_solves_running) {}
    ~TpRunningGuard() { --g_solves_running; }
};

#define TP_EV 7   // CUDA events per tick in timed mode: start, after integrate / penalty / chain / adjoint / L-BFGS / generate

// Live slots up to which a tick runs k_cand as one fused launch: one wave of candidate blocks (3 blocks x 148 SMs).
constexpr int TP_FUSE_MAX_SLOTS = 444;

// One lane of a run: the live lists and counts its kernels read and write, the stream it is enqueued on, and its
// live-slot count, which returns from the device through a pinned word after every batch.
struct TpLane {
    int32_t* list;          // [TP_TICKS + 1][n_slots] live lists
    int32_t* count;         // [TP_TICKS + 1] live counts
    cudaStream_t stream;
    int32_t* h_live;        // pinned
    int live;
};

// Launches of an enqueue, counted where they are enqueued.
struct TpLaunches {
    int64_t kernels = 0, evals = 0;
    void add_to(topay_solver_stats& st) const {
        st.kernel_launches += kernels;
        st.eval_launches += evals;
    }
};

// A captured batch of ticks and the launches one replay of it makes.
struct TpBatchGraph {
    cudaGraphExec_t exec;
    TpLaunches launches;
};

struct topay_solver {
    TpSolverDev dev;
    TpParams params;
    topay_field* field;          // dense GridMap field, or
    topay_rogfield* rog;         // the ROG-Map ring (GridMap's use_rog branches); exactly one is set
    int device;
    cudaStream_t stream;
    int n_cand;          // candidates of the uploaded batch
    int max_N;           // largest piece count in the batch
    // pinned host staging (one cudaMallocHost block sized for max_cand): initial per-candidate state and x,
    // and the packed problem data on their way to the device
    char* h_pin;
    TpCandState* h_state;
    double *p_head, *p_tail, *p_sxy, *p_exy, *p_ixy;
    std::vector<void*> allocs;
    int32_t* h_active;   // pinned: [0] lane A's live slots after the batch, [1..3] queue state, [4] lane B's live slots
    unsigned long long* h_nodes;  // pinned
    int n_slots_used;    // slots seeded by the last run (min(n_slots, n_cand))
    std::vector<cudaEvent_t> ev;  // event pool for the penalty kernel timing
    cudaEvent_t ev_begin, ev_end;
    cudaEvent_t ev_batch;   // blocking-sync event: the host thread sleeps while a batch of ticks runs
                            // (P plans in flight x N ranks would otherwise spin on as many cores)
    topay_solver_stats stats;
    size_t smem_cand;    // dynamic shared memory of the adjoint / generate launches (banded system)
    size_t smem_lbfgs;   // ... of the L-BFGS launch (TMA ring + tables)
    // initial state kept on the host for repeated runs
    double* h_x0;
    size_t h_x0_count;
    // one batch of `slots` ticks as a CUDA graph (launch-bound small plans); rebuilt when the
    // launch geometry or a captured pointer changes
    bool timed;                 // per-launch CUDA events around k_penalty (plain launches, no graph)
    // one CUDA graph per launch-grid bucket (live slots rounded up), rebuilt when max_N or a captured pointer changes
    std::map<int, TpBatchGraph> graphs;
    int graph_max_N;
    // Two LANES (large pools only): the slots are split into two halves with their own live lists, and a batch runs
    // the halves' tick chains as two parallel branches of one CUDA graph (lane B's branch on its own stream). The
    // kernels of a tick are bound by different things (k_penalty: FP64 issue; the two-loop: HBM; the banded LU: one
    // warp's latency chain), so one half's k_penalty overlaps the other half's k_cand. Store, queue and results are
    // shared: which lane solves a candidate does not change its result.
    TpLane lane[2];             // lane A: dev.list / dev.count on `stream`; lane B: its own lists on a second stream
    int lanes;                  // lanes of the run in progress (1 or 2)
    int lane_min_slots;         // two lanes from this many seeded slots on (TOPAY_LANE_MIN_SLOTS; 0 = never)
    cudaEvent_t ev_fork, ev_join;
    // scenario sweeps: candidates of one upload may belong to different fields (topay_solver_assign_fields)
    std::vector<topay_field*> fields;
    TpGrid* d_grids;            // [max_cand] (a field per candidate at most), allocated on first use
    int32_t* d_field_of;        // [max_cand]
    int fields_n_cand;          // the upload size the assignment was made for
    // success gate (topay_solver_check_feasible): built on first use
    TpTrajChecker* checker;
    int32_t* d_pn;
    double* d_start;
};

namespace {

void solver_grid(const topay_solver* s, TpGrid* G) {
    if (s->rog) tp_rogfield_grid(s->rog, G);
    else tp_field_grid(s->field, G);
}
bool solver_field_ready(const topay_solver* s) {
    if (s->dev.n_fields > 1) {
        for (const topay_field* f : s->fields)
            if (!tp_field_ready(f)) return false;
        return true;
    }
    return s->rog ? tp_rogfield_ready(s->rog) : tp_field_ready(s->field);
}

template <typename T>
int dev_alloc(topay_solver* s, T** p, size_t count) {
    const int rc = tp_dev_malloc(p, count);
    if (rc != TOPAY_OK) return rc;
    cudaMemsetAsync(*p, 0, std::max<size_t>(count, 1) * sizeof(T), s->stream);
    s->allocs.push_back(*p);
    return TOPAY_OK;
}

int kpad_of(int K) {
    int p = 4;
    while (p < K) p <<= 1;
    return p;
}

size_t penalty_smem(int kpad) {   // two sphere stores per thread + the coefficient blocks of the warp's 32 / kpad pieces
    return (size_t)(72 * TP_PEN_WARPS * 32 + TP_PEN_WARPS * (32 / kpad) * 54) * sizeof(double);
}

// grid.y / grid.x of a tick: the live-slot count rounded up to a bucket (1..8, then 12, 16, 24, 32, 48, ...),
// so that a handful of graphs covers a run; blocks beyond the live count exit at once
int grid_bucket(int n) {
    if (n <= 8) return n < 1 ? 1 : n;
    for (int p = 8;; p *= 2) {
        if (n <= p) return p;
        if (n <= p + p / 2) return p + p / 2;
    }
}

// k_penalty<Kpad, MULTI>, [log2(Kpad) - 2][MULTI]
using PenaltyKernel = decltype(&k_penalty<4>);
const PenaltyKernel k_penalty_of[4][2] = {{k_penalty<4>, k_penalty<4, true>},
                                          {k_penalty<8>, k_penalty<8, true>},
                                          {k_penalty<16>, k_penalty<16, true>},
                                          {k_penalty<32>, k_penalty<32, true>}};
int kpad_index(int kpad) { return kpad == 4 ? 0 : kpad == 8 ? 1 : kpad == 16 ? 2 : 3; }

// k_cand<MODE> of a launch mode, and its dynamic shared memory: the banded system (adjoint, generate), the L-BFGS
// ring (advance), or the larger of the two (all three halves fused)
constexpr int TP_MODE_ALL = TP_MODE_ADJ | TP_MODE_ADVANCE | TP_MODE_GEN;
constexpr int TP_CAND_MODES[4] = {TP_MODE_ADJ, TP_MODE_ADVANCE, TP_MODE_GEN, TP_MODE_ALL};
using CandKernel = decltype(&k_cand<TP_MODE_ALL>);
CandKernel cand_kernel(int mode) {
    switch (mode) {
        case TP_MODE_ADJ: return k_cand<TP_MODE_ADJ>;
        case TP_MODE_ADVANCE: return k_cand<TP_MODE_ADVANCE>;
        case TP_MODE_GEN: return k_cand<TP_MODE_GEN>;
        default: return k_cand<TP_MODE_ALL>;
    }
}
size_t cand_smem(const topay_solver* s, int mode) {
    if (mode == TP_MODE_ADVANCE) return s->smem_lbfgs;
    if (mode == TP_MODE_ALL) return std::max(s->smem_cand, s->smem_lbfgs);
    return s->smem_cand;
}

// What a kernel of lane L reads: the solver's device view with the lane's live lists.
TpSolverDev lane_dev(const topay_solver* s, const TpLane& L) {
    TpSolverDev D = s->dev;
    D.list = L.list;
    D.count = L.count;
    return D;
}

void launch_eval(topay_solver* s, const TpLane& L, bool timed, int tick, int ny, TpLaunches& n) {
    const TpSolverDev D = lane_dev(s, L);
    const int groups = (s->max_N + D.ppw - 1) / D.ppw;
    const int end_warps = D.end_tasks ? (s->max_N + 31) / 32 : 0;
    dim3 blk(TP_WARPS_PER_BLOCK * 32);
    dim3 g1((groups + TP_WARPS_PER_BLOCK - 1) / TP_WARPS_PER_BLOCK, ny);
    dim3 blk2(TP_PEN_WARPS * 32);
    dim3 g2((groups + end_warps + TP_PEN_WARPS - 1) / TP_PEN_WARPS, ny);
    const size_t sm_int = (size_t)TP_WARPS_PER_BLOCK * D.ppw * 3 * (2 * D.K + 1) * sizeof(double);
    const size_t sm_pen = penalty_smem(D.Kpad);
    TpGrid G;
    solver_grid(s, &G);
    cudaStream_t q = L.stream;
    const int te = tick % TP_TICKS;
    if (timed) cudaEventRecord(s->ev[TP_EV * te], q);
    k_integrate<<<g1, blk, sm_int, q>>>(D, tick);
    if (timed) cudaEventRecord(s->ev[TP_EV * te + 1], q);
    k_penalty_of[kpad_index(D.Kpad)][D.n_fields > 1]<<<g2, blk2, sm_pen, q>>>(D, s->params, G, groups, tick);
    if (timed) cudaEventRecord(s->ev[TP_EV * te + 2], q);
    k_chain<<<g1, blk, 0, q>>>(D, s->params, tick);
    if (timed) cudaEventRecord(s->ev[TP_EV * te + 3], q);
    n.kernels += 3;
    n.evals += 1;
}

void launch_cand(topay_solver* s, const TpLane& L, int mode, int tick_in, int tick_out, int nx, TpLaunches& n) {
    const size_t sm = cand_smem(s, mode);
    cand_kernel(mode)<<<nx, TP_CAND_THREADS, sm, L.stream>>>(lane_dev(s, L), s->params, (int)(sm / sizeof(double)),
                                                            tick_in, tick_out);
    n.kernels += 1;
}

void drop_graphs(topay_solver* s) {
    for (auto& kv : s->graphs) cudaGraphExecDestroy(kv.second.exec);
    s->graphs.clear();
}

}  // namespace

static int solver_create(const topay_opt_params* opt, const topay_robot_params* robot, topay_field* field,
                         topay_rogfield* rog, int max_cand, int n_slots, int max_pieces, topay_solver** out);
extern "C" int topay_solver_assign_fields(topay_solver* s, topay_field* const* fields, int n_fields, const int32_t* field_of);

extern "C" int topay_solver_create(const topay_opt_params* opt, const topay_robot_params* robot,
                                   topay_field* field, int max_cand, int max_pieces, topay_solver** out) {
    if (!field) return TOPAY_ERR_INVALID_ARG;
    return solver_create(opt, robot, field, nullptr, max_cand, max_cand, max_pieces, out);
}

extern "C" int topay_solver_create_rog(const topay_opt_params* opt, const topay_robot_params* robot,
                                       topay_rogfield* rog, int max_cand, int max_pieces, topay_solver** out) {
    if (!rog) return TOPAY_ERR_INVALID_ARG;
    return solver_create(opt, robot, nullptr, rog, max_cand, max_cand, max_pieces, out);
}

extern "C" int topay_solver_create_pool(const topay_opt_params* opt, const topay_robot_params* robot,
                                        topay_field* field, int max_cand, int n_slots, int max_pieces,
                                        topay_solver** out) {
    if (!field) return TOPAY_ERR_INVALID_ARG;
    return solver_create(opt, robot, field, nullptr, max_cand, n_slots, max_pieces, out);
}

static int solver_create(const topay_opt_params* opt, const topay_robot_params* robot, topay_field* field,
                         topay_rogfield* rog, int max_cand, int n_slots, int max_pieces, topay_solver** out) {
    if (!opt || !robot || !out || max_cand < 1 || max_pieces < 1 || n_slots < 1) return TOPAY_ERR_INVALID_ARG;
    if (n_slots > max_cand) n_slots = max_cand;
    if (opt->int_K < 1 || opt->int_K > TP_MAX_K) {
        tp_set_error("int_K must be in [1, 32]");
        return TOPAY_ERR_TOO_LARGE;
    }
    if (opt->s1_lbfgs_normal_past > TP_LBFGS_MAX_PAST || opt->s1_lbfgs_shot_path_past > TP_LBFGS_MAX_PAST ||
        opt->s2_lbfgs.past > TP_LBFGS_MAX_PAST) {
        tp_set_error("lbfgs past above the supported ring size");
        return TOPAY_ERR_TOO_LARGE;
    }
    if (topay_num_vars(max_pieces) > TP_EPT * TP_CAND_THREADS || max_pieces > 64 ||
        std::max(opt->s1_lbfgs.mem_size, opt->s2_lbfgs.mem_size) > 256) {
        tp_set_error("max_pieces above 64 or lbfgs mem_size above 256 is not supported");
        return TOPAY_ERR_TOO_LARGE;
    }
    const int dev = rog ? tp_rogfield_device(rog) : tp_field_device(field);
    int rc = tp_require_device(dev);
    if (rc != TOPAY_OK) return rc;
    topay_solver* s = new topay_solver();
    s->field = field;
    s->rog = rog;
    s->device = dev;
    s->n_cand = 0;
    s->max_N = 0;
    s->n_slots_used = 0;
    s->timed = false;
    s->graph_max_N = -1;
    s->checker = nullptr;
    s->d_pn = nullptr;
    s->d_start = nullptr;
    memset(&s->stats, 0, sizeof(s->stats));
    cudaSetDevice(s->device);
    tp_pool_keep(s->device);
    TP_CUDA_OK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking), { delete s; });
    memset(&s->params, 0, sizeof(s->params));
    s->params.robot = *robot;
    s->params.opt = *opt;
    tp_derive_params(s->params);
    TpSolverDev& D = s->dev;
    memset(&D, 0, sizeof(D));
    D.max_cand = max_cand;
    D.n_slots = n_slots;
    D.max_pieces = max_pieces;
    D.K = opt->int_K;
    D.Kpad = kpad_of(D.K);
    D.ppw = 32 / D.Kpad;
    D.end_tasks = D.K == D.Kpad ? 1 : 0;
    D.xs = (topay_num_vars(max_pieces) + 3) & ~3;
    D.mem = std::max(1, std::max(opt->s1_lbfgs.mem_size, opt->s2_lbfgs.mem_size));
    const size_t G = max_cand, C = n_slots, NP = max_pieces, K = D.K;
#define ALLOC(ptr, count)                                    \
    if ((rc = dev_alloc(s, &(ptr), (count))) != TOPAY_OK) {  \
        topay_solver_destroy(s);                             \
        return rc;                                           \
    }
    // store
    ALLOC(D.head_pva, G * 27);
    ALLOC(D.tail_pva, G * 27);
    ALLOC(D.start_xy, G * 2);
    ALLOC(D.end_xy, G * 2);
    ALLOC(D.init_inner_xy, G * NP * 2);
    ALLOC(D.x0, G * D.xs);
    ALLOC(D.st0, G);
    ALLOC(D.res_st, G);
    ALLOC(D.res_T, G * NP);
    ALLOC(D.res_coeff, G * 6 * NP * 9);
    ALLOC(D.res_x, G * D.xs);
    // scheduling
    ALLOC(D.slot_gid, C);
    ALLOC(D.list, (size_t)(TP_TICKS + 1) * C);
    ALLOC(D.count, (size_t)TP_TICKS + 1);
    ALLOC(s->lane[1].list, (size_t)(TP_TICKS + 1) * C);
    ALLOC(s->lane[1].count, (size_t)TP_TICKS + 1);
    ALLOC(D.queue, 4);
    // slots
    ALLOC(D.st, C);
    ALLOC(D.x, C * D.xs);
    ALLOC(D.g, C * D.xs);
    ALLOC(D.xp, C * D.xs);
    ALLOC(D.gp, C * D.xs);
    ALLOC(D.d, C * D.xs);
    ALLOC(D.lm_s, C * D.mem * D.xs);
    ALLOC(D.lm_y, C * D.mem * D.xs);
    ALLOC(D.lm_ys, C * D.mem);
    ALLOC(D.lm_alpha, C * D.mem);
    ALLOC(D.T, C * NP);
    ALLOC(D.coeff, C * 6 * NP * 9);
    ALLOC(D.lu, C * 6 * NP * TP_BAND);
    ALLOC(D.Ixy, C * NP * K * 2);
    ALLOC(D.tot, C * NP * 2);
    ALLOC(D.gnode, C * NP * (K + 1) * 2);
    ALLOC(D.gsum, C * NP * 2);
    ALLOC(D.gdC, C * 6 * NP * 9);
    ALLOC(D.gdC_end, C * NP * 54);
    ALLOC(D.gdT, C * NP);
    ALLOC(D.gdT_end, C * NP);
    ALLOC(D.terms, C * NP * TOPAY_NTERMS);
    ALLOC(D.terms_end, C * NP * TOPAY_NTERMS);
    ALLOC(D.f, C);
    ALLOC(D.term_out, C * TOPAY_NTERMS);
    ALLOC(D.node_count, 2);
#undef ALLOC
    {
        const size_t b_state = ((G * sizeof(TpCandState) + 15) / 16) * 16;
        const size_t n_dbl = G * D.xs + G * (27 + 27 + 2 + 2) + G * NP * 2;
        TP_CUDA_OK(cudaMallocHost(&s->h_pin, b_state + n_dbl * sizeof(double)), { topay_solver_destroy(s); });
        s->h_state = reinterpret_cast<TpCandState*>(s->h_pin);
        double* dp = reinterpret_cast<double*>(s->h_pin + b_state);
        s->h_x0 = dp;            dp += G * D.xs;
        s->p_head = dp;          dp += G * 27;
        s->p_tail = dp;          dp += G * 27;
        s->p_sxy = dp;           dp += G * 2;
        s->p_exy = dp;           dp += G * 2;
        s->p_ixy = dp;
        s->h_x0_count = 0;
    }
    TP_CUDA_OK(cudaMallocHost(&s->h_active, 8 * sizeof(int32_t)), { topay_solver_destroy(s); });
    TP_CUDA_OK(cudaMallocHost(&s->h_nodes, 2 * sizeof(unsigned long long)), { topay_solver_destroy(s); });
    s->ev.resize(TP_EV * TP_TICKS);
    for (auto& e : s->ev) cudaEventCreate(&e);
    cudaEventCreate(&s->ev_begin);
    cudaEventCreate(&s->ev_end);
    cudaEventCreateWithFlags(&s->ev_batch, cudaEventBlockingSync | cudaEventDisableTiming);
    s->lane[0].list = D.list;
    s->lane[0].count = D.count;
    s->lane[0].stream = s->stream;
    s->lane[0].h_live = s->h_active;
    cudaStreamCreateWithFlags(&s->lane[1].stream, cudaStreamNonBlocking);
    s->lane[1].h_live = s->h_active + 4;
    cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming);
    s->lanes = 1;
    s->lane_min_slots = getenv("TOPAY_LANE_MIN_SLOTS") ? atoi(getenv("TOPAY_LANE_MIN_SLOTS")) : 512;
    // LU band + one right-hand-side matrix, or the two-loop's TMA ring + its two 256-entry tables + one
    // vector of scratch (single-warp variant)
    // at least six full-width stages; small solvers still get 64 KB so that short rows ride a deep ring
    s->smem_cand = std::max(std::max((size_t)6 * NP * (TP_BAND + 9), (size_t)6 * 2 * D.xs + 512 + D.xs) * sizeof(double),
                            (size_t)64 * 1024);
    D.smem_doubles = (int32_t)(s->smem_cand / sizeof(double));
    // L-BFGS launch: four full-width stages of (s_j, y_j) + the alpha / 1/ys tables + one vector of scratch; short rows
    // (small plans run the recursion on one warp) still get up to 64 KB so that they ride a deep ring
    {
        const size_t rowd = (size_t)((topay_num_vars(max_pieces) + 1) & ~1);
        const size_t tail = (size_t)512 + D.xs;
        const size_t four = (4 * 2 * rowd + tail) * sizeof(double);
        const size_t deep = std::min((size_t)64 * 1024, (TP_RING_MAX * 2 * rowd + tail) * sizeof(double));
        s->smem_lbfgs = std::max(four, deep);
    }
    if (s->smem_cand > 227 * 1024) {
        tp_set_error("max_pieces too large for the per-candidate shared-memory working set");
        topay_solver_destroy(s);
        return TOPAY_ERR_TOO_LARGE;
    }
    for (int mode : TP_CAND_MODES)
        TP_CUDA_OK(tp_grow_dyn_smem((const void*)cand_kernel(mode), cand_smem(s, mode)), { topay_solver_destroy(s); });
    const size_t sm_int = (size_t)TP_WARPS_PER_BLOCK * D.ppw * 3 * (2 * D.K + 1) * sizeof(double);
    TP_CUDA_OK(tp_grow_dyn_smem((const void*)k_integrate, sm_int), { topay_solver_destroy(s); });
    for (int k = 0; k < 4; k++)
        for (PenaltyKernel kern : k_penalty_of[k])
            TP_CUDA_OK(tp_grow_dyn_smem((const void*)kern, penalty_smem(4 << k)), { topay_solver_destroy(s); });
    TP_CUDA_OK(cudaStreamSynchronize(s->stream), { topay_solver_destroy(s); });
    *out = s;
    return TOPAY_OK;
}

extern "C" void topay_solver_destroy(topay_solver* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    drop_graphs(s);
    delete s->checker;
    for (void* p : s->allocs) cudaFree(p);
    if (s->dev.trace) cudaFree(s->dev.trace);
    if (s->dev.trace_len) cudaFree(s->dev.trace_len);
    if (s->dev.prof) cudaFree(s->dev.prof);
    if (s->h_pin) cudaFreeHost(s->h_pin);
    if (s->h_active) cudaFreeHost(s->h_active);
    if (s->h_nodes) cudaFreeHost(s->h_nodes);
    for (auto& e : s->ev) cudaEventDestroy(e);
    if (s->ev_begin) cudaEventDestroy(s->ev_begin);
    if (s->ev_end) cudaEventDestroy(s->ev_end);
    if (s->ev_batch) cudaEventDestroy(s->ev_batch);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    if (s->lane[1].stream) cudaStreamDestroy(s->lane[1].stream);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// Uploads problem data + x of n_cand candidates into the store and their initial per-candidate state.
static int upload_problem(topay_solver* s, int n_cand, const int32_t* piece_num, const double* head,
                          const double* tail, const double* sxy, const double* exy, const double* inner_xy,
                          const double* x, int x_stride, const int32_t* s1_past, int phase, const double* lambda,
                          const double* rho) {
    TpSolverDev& D = s->dev;
    if (n_cand < 1 || n_cand > D.max_cand) {
        tp_set_error("n_cand above the solver capacity");
        return TOPAY_ERR_TOO_LARGE;
    }
    int maxN = 0;
    for (int c = 0; c < n_cand; c++) {
        if (piece_num[c] < 1 || piece_num[c] > D.max_pieces) {
            tp_set_error("piece_num above the solver capacity");
            return TOPAY_ERR_TOO_LARGE;
        }
        maxN = std::max(maxN, piece_num[c]);
    }
    cudaSetDevice(s->device);
    s->n_cand = n_cand;
    s->max_N = maxN;
    double* xs = s->h_x0;
    memset(xs, 0, (size_t)n_cand * D.xs * sizeof(double));
    s->h_x0_count = (size_t)n_cand * D.xs;
    for (int c = 0; c < n_cand; c++) {
        TpCandState& st = s->h_state[c];
        memset(&st, 0, sizeof(st));
        st.phase = phase;
        st.N = piece_num[c];
        st.n = topay_num_vars(piece_num[c]);
        st.ls_init = 1;
        st.s1_past = s1_past ? s1_past[c] : s->params.opt.s1_lbfgs.past;
        st.lambda[0] = lambda ? lambda[2 * c] : s->params.opt.alm_init_lambda[0];
        st.lambda[1] = lambda ? lambda[2 * c + 1] : s->params.opt.alm_init_lambda[1];
        st.rho[0] = rho ? rho[2 * c] : s->params.opt.alm_init_rho[0];
        st.rho[1] = rho ? rho[2 * c + 1] : s->params.opt.alm_init_rho[1];
        memcpy(&xs[(size_t)c * D.xs], x + (size_t)c * x_stride, st.n * sizeof(double));
    }
    // the packed problem goes through the pinned staging block
    memcpy(s->p_head, head, (size_t)n_cand * 27 * 8);
    memcpy(s->p_tail, tail, (size_t)n_cand * 27 * 8);
    memcpy(s->p_sxy, sxy, (size_t)n_cand * 2 * 8);
    memcpy(s->p_exy, exy, (size_t)n_cand * 2 * 8);
    memcpy(s->p_ixy, inner_xy, (size_t)n_cand * D.max_pieces * 2 * 8);
    cudaStream_t q = s->stream;
    TP_CUDA_OK(cudaMemcpyAsync(D.st0, s->h_state, n_cand * sizeof(TpCandState), cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.head_pva, s->p_head, (size_t)n_cand * 27 * 8, cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.tail_pva, s->p_tail, (size_t)n_cand * 27 * 8, cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.start_xy, s->p_sxy, (size_t)n_cand * 2 * 8, cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.end_xy, s->p_exy, (size_t)n_cand * 2 * 8, cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.init_inner_xy, s->p_ixy, (size_t)n_cand * D.max_pieces * 2 * 8,
                               cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaMemcpyAsync(D.x0, xs, s->h_x0_count * 8, cudaMemcpyHostToDevice, q), {});
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    return TOPAY_OK;
}

// Seeds the slots with the first candidates of the store; the live list is list TP_TICKS.
static int seed_slots(topay_solver* s) {
    const TpSolverDev& D = s->dev;
    const int n0 = std::min(D.n_slots, s->n_cand);
    s->n_slots_used = n0;
    k_slot_init<<<n0, 128, 0, s->stream>>>(D, n0, s->n_cand);
    return n0;
}

// Two lanes: slots [0, na) stay on lane A's list, slots [na, n0) move to lane B's.
__global__ void k_lane_split(const __grid_constant__ TpSolverDev S, int32_t* list_b, int32_t* count_b, int na, int n0) {
    for (int i = threadIdx.x; i < n0 - na; i += blockDim.x) list_b[(size_t)TP_TICKS * S.n_slots + i] = na + i;
    if (threadIdx.x == 0) {
        for (int t = 0; t < TP_TICKS; t++) count_b[t] = 0;
        count_b[TP_TICKS] = n0 - na;
        S.count[TP_TICKS] = na;
    }
}

extern "C" int topay_solver_eval(topay_solver* s, int stage, const topay_problem_batch* prob, const double* x,
                                 int x_stride, double* cost, double* grad, double* term_costs, double* coeff_out,
                                 double* final_xy_out) {
    if (!s || !prob || !x || !cost || !grad || (stage != 1 && stage != 2)) return TOPAY_ERR_INVALID_ARG;
    if (!solver_field_ready(s)) {
        tp_set_error("field not built: call topay_field_rebuild first");
        return TOPAY_ERR_NOT_READY;
    }
    if (prob->n_cand > s->dev.n_slots) {
        tp_set_error("topay_solver_eval evaluates at most n_slots candidates at a time");
        return TOPAY_ERR_TOO_LARGE;
    }
    if (s->dev.n_fields > 1) topay_solver_assign_fields(s, nullptr, 0, nullptr);   // evaluations read the solver's own field
    int rc = upload_problem(s, prob->n_cand, prob->piece_num, prob->head_pva, prob->tail_pva, prob->start_xy,
                            prob->end_xy, prob->init_inner_xy, x, x_stride, nullptr, stage, prob->alm_lambda,
                            prob->alm_rho);
    if (rc != TOPAY_OK) return rc;
    const TpSolverDev& D = s->dev;
    const int n = prob->n_cand;
    seed_slots(s);   // slot i <- candidate i
    TpLaunches launches;
    launch_cand(s, s->lane[0], TP_MODE_GEN, TP_TICKS, -1, n, launches);
    launch_eval(s, s->lane[0], false, TP_TICKS, n, launches);
    launch_cand(s, s->lane[0], TP_MODE_ADJ, TP_TICKS, -1, n, launches);
    launches.add_to(s->stats);
    TP_CUDA_OK(cudaStreamSynchronize(s->stream), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    s->n_cand = 0;   // the uploaded problem carried the evaluation's phase / multipliers: not a solvable upload
    std::vector<double> g((size_t)n * D.xs);
    TP_CUDA_OK(cudaMemcpy(cost, D.f, n * 8, cudaMemcpyDeviceToHost), {});
    TP_CUDA_OK(cudaMemcpy(g.data(), D.g, g.size() * 8, cudaMemcpyDeviceToHost), {});
    for (int c = 0; c < n; c++)
        memcpy(grad + (size_t)c * x_stride, &g[(size_t)c * D.xs], topay_num_vars(prob->piece_num[c]) * 8);
    if (term_costs) TP_CUDA_OK(cudaMemcpy(term_costs, D.term_out, (size_t)n * TOPAY_NTERMS * 8, cudaMemcpyDeviceToHost), {});
    if (coeff_out)
        TP_CUDA_OK(cudaMemcpy(coeff_out, D.coeff, (size_t)n * 6 * D.max_pieces * 9 * 8, cudaMemcpyDeviceToHost), {});
    if (final_xy_out) {
        std::vector<TpCandState> st(n);
        TP_CUDA_OK(cudaMemcpy(st.data(), D.st, n * sizeof(TpCandState), cudaMemcpyDeviceToHost), {});
        for (int c = 0; c < n; c++) {
            final_xy_out[2 * c] = st[c].final_xy[0];
            final_xy_out[2 * c + 1] = st[c].final_xy[1];
        }
    }
    return TOPAY_OK;
}

// Scenario sweeps (BASELINE configs[4]): the candidates of ONE upload may belong to different scenarios, each with its
// own field. field_of[c] (n_cand entries, the uploaded batch) indexes `fields`; all fields live on the solver's device
// and are dense GridMap fields. The assignment holds for uploads of the same size until it is changed; n_fields <= 1
// returns to the solver's own field. Call after topay_solver_upload, before topay_solver_run; rebuild the fields first.
extern "C" int topay_solver_assign_fields(topay_solver* s, topay_field* const* fields, int n_fields,
                                          const int32_t* field_of) {
    if (!s) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    TpSolverDev& D = s->dev;
    if (n_fields <= 1) {
        if (D.n_fields > 1) drop_graphs(s);     // the captured kernel arguments change
        D.n_fields = 0;
        s->fields.clear();
        return TOPAY_OK;
    }
    if (!fields || !field_of || s->rog || s->n_cand < 1 || n_fields > D.max_cand) return TOPAY_ERR_INVALID_ARG;
    std::vector<TpGrid> hg(n_fields);
    for (int i = 0; i < n_fields; i++) {
        if (!fields[i] || tp_field_device(fields[i]) != s->device) return TOPAY_ERR_INVALID_ARG;
        tp_field_grid(fields[i], &hg[i]);
    }
    for (int c = 0; c < s->n_cand; c++)
        if (field_of[c] < 0 || field_of[c] >= n_fields) return TOPAY_ERR_INVALID_ARG;
    int rc;
    if (!s->d_grids) {
        if ((rc = dev_alloc(s, &s->d_grids, (size_t)D.max_cand)) != TOPAY_OK) return rc;
        if ((rc = dev_alloc(s, &s->d_field_of, (size_t)D.max_cand)) != TOPAY_OK) return rc;
    }
    TP_CUDA_OK(cudaMemcpyAsync(s->d_grids, hg.data(), (size_t)n_fields * sizeof(TpGrid), cudaMemcpyHostToDevice, s->stream), {});
    TP_CUDA_OK(cudaMemcpyAsync(s->d_field_of, field_of, (size_t)s->n_cand * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(s->stream), {});
    if (D.n_fields <= 1) drop_graphs(s);
    D.grids = s->d_grids;
    D.field_of = s->d_field_of;
    D.n_fields = 2;             // "one field per candidate" (the kernels only test > 1)
    s->fields.assign(fields, fields + n_fields);
    s->fields_n_cand = s->n_cand;
    return TOPAY_OK;
}

extern "C" int topay_solver_upload(topay_solver* s, int n_cand, const int32_t* path_len, const double* init_paths,
                                   const double* bvel, const double* bacc) {
    if (!s || !path_len || !init_paths || !bvel || !bacc) return TOPAY_ERR_INVALID_ARG;
    const TpSolverDev& D = s->dev;
    if (n_cand < 1 || n_cand > D.max_cand) {
        tp_set_error("n_cand above the solver capacity");
        return TOPAY_ERR_TOO_LARGE;
    }
    const int NP = D.max_pieces, xstride = topay_num_vars(NP);
    std::vector<int32_t> pn(n_cand), past(n_cand);
    std::vector<double> head((size_t)n_cand * 27), tail((size_t)n_cand * 27), sxy((size_t)n_cand * 2),
        exy((size_t)n_cand * 2), ixy((size_t)n_cand * NP * 2), x((size_t)n_cand * xstride, 0.0);
    size_t off = 0;
    for (int c = 0; c < n_cand; c++) {
        int rc = topay_prepare_candidate(&s->params.opt, &s->params.robot, init_paths + off * 10, path_len[c],
                                         bvel + (size_t)c * 20, bacc + (size_t)c * 20, NP, &pn[c], &head[c * 27],
                                         &tail[c * 27], &sxy[c * 2], &exy[c * 2], &ixy[(size_t)c * NP * 2],
                                         &x[(size_t)c * xstride], &past[c]);
        if (rc != TOPAY_OK) {
            tp_set_error("candidate needs more pieces than max_pieces");
            return rc;
        }
        off += path_len[c];
    }
    return upload_problem(s, n_cand, pn.data(), head.data(), tail.data(), sxy.data(), exy.data(), ixy.data(),
                          x.data(), xstride, past.data(), 1, nullptr, nullptr);
}

// One batch of TP_TICKS ticks of lane L over at most `ny` live slots: roll the list, then per tick the three
// evaluation kernels and k_cand; the lane's live count after the batch returns through its pinned word.
static void enqueue_lane(topay_solver* s, const TpLane& L, int ny, bool timed, TpLaunches& n) {
    cudaStream_t q = L.stream;
    k_list_roll<<<1, 1024, 0, q>>>(lane_dev(s, L));
    n.kernels += 1;
    // Up to one wave of candidate blocks the three halves of k_cand run as ONE launch (the banded system stays in
    // shared memory from the adjoint solve to the next factorisation, two launch boundaries less on the dependent
    // chain of a small plan); above that they are separate launches, each at its own occupancy.
    const bool fused = !timed && ny <= TP_FUSE_MAX_SLOTS;
    for (int t = 0; t < TP_TICKS; t++) {
        launch_eval(s, L, timed, t, ny, n);
        if (fused) {
            launch_cand(s, L, TP_MODE_ALL, t, t + 1, ny, n);
            continue;
        }
        launch_cand(s, L, TP_MODE_ADJ, t, -1, ny, n);
        if (timed) cudaEventRecord(s->ev[TP_EV * t + 4], q);
        launch_cand(s, L, TP_MODE_ADVANCE, t, -1, ny, n);
        if (timed) cudaEventRecord(s->ev[TP_EV * t + 5], q);
        launch_cand(s, L, TP_MODE_GEN, t, t + 1, ny, n);
        if (timed) cudaEventRecord(s->ev[TP_EV * t + 6], q);
    }
    cudaMemcpyAsync(L.h_live, L.count + TP_TICKS, sizeof(int32_t), cudaMemcpyDeviceToHost, q);
}

// One batch of both lanes (ny, ny_b: their launch grids); returns the launches it enqueued.
static TpLaunches enqueue_batch(topay_solver* s, int ny, int ny_b, bool timed) {
    TpLaunches n;
    cudaStream_t q = s->stream;
    if (s->lanes == 2) {
        // fork: lane B's chain is a second branch of the captured graph
        cudaEventRecord(s->ev_fork, q);
        cudaStreamWaitEvent(s->lane[1].stream, s->ev_fork, 0);
        enqueue_lane(s, s->lane[1], ny_b, timed, n);
        cudaEventRecord(s->ev_join, s->lane[1].stream);
    }
    enqueue_lane(s, s->lane[0], ny, timed, n);
    if (s->lanes == 2) cudaStreamWaitEvent(q, s->ev_join, 0);
    cudaMemcpyAsync(s->h_active + 1, s->dev.queue, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, q);
    return n;
}

// Marks every candidate that is still live (or was never started) as stopped by the tick cap.
__global__ void k_mark_tick_cap(const __grid_constant__ TpSolverDev S, int n_store) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S.count[TP_TICKS]) {
        const int slot = S.list[(size_t)TP_TICKS * S.n_slots + i];
        TpCandState st = S.st[slot];
        if (st.phase != 0) {
            st.phase = 0;
            st.status = 0;
            st.last_code = TOPAY_LBFGSERR_TICK_CAP;
            S.st[slot] = st;
            S.res_st[S.slot_gid[slot]] = st;
        }
    }
    if (i >= S.queue[0] && i < n_store) {   // never handed to a slot
        TpCandState st = S.st0[i];
        st.phase = 0;
        st.status = 0;
        st.last_code = TOPAY_LBFGSERR_TICK_CAP;
        S.res_st[i] = st;
    }
}

// Tick cap: marks lane L's live candidates and, with n_store > 0, the candidates of the store never handed to a slot.
// Runs after the last batch, when both lanes have joined the solver's stream.
static void mark_tick_cap(topay_solver* s, const TpLane& L, int n_store) {
    k_mark_tick_cap<<<(std::max(n_store, s->dev.n_slots) + 127) / 128, 128, 0, s->stream>>>(lane_dev(s, L), n_store);
}

extern "C" int topay_solver_run(topay_solver* s) {
    if (!s || s->n_cand < 1) return TOPAY_ERR_INVALID_ARG;
    if (!solver_field_ready(s)) {
        tp_set_error("field not built: call topay_field_rebuild first");
        return TOPAY_ERR_NOT_READY;
    }
    if (s->dev.n_fields > 1 && s->fields_n_cand != s->n_cand) {
        tp_set_error("the field assignment was made for an upload of another size: call topay_solver_assign_fields again");
        return TOPAY_ERR_NOT_READY;
    }
    cudaSetDevice(s->device);
    TpSolverDev& D = s->dev;
    cudaStream_t q = s->stream;
    TpRunningGuard running;
    memset(&s->stats, 0, sizeof(s->stats));
    cudaMemsetAsync(D.node_count, 0, 2 * sizeof(unsigned long long), q);
    if (D.trace) cudaMemsetAsync(D.trace_len, 0, (size_t)D.max_cand * sizeof(int32_t), q);
    cudaEventRecord(s->ev_begin, q);
    // the store holds the uploaded initial state, so repeated runs do identical work
    TpLane &A = s->lane[0], &B = s->lane[1];
    A.live = seed_slots(s);
    B.live = 0;
    TpLaunches first;
    launch_cand(s, A, TP_MODE_GEN, TP_TICKS, -1, A.live, first);
    first.kernels += 1;   // seed_slots' k_slot_init
    first.add_to(s->stats);
    s->lanes = (!s->timed && s->lane_min_slots > 0 && A.live >= s->lane_min_slots) ? 2 : 1;
    if (s->lanes == 2) {
        const int na = (A.live + 1) / 2;
        k_lane_split<<<1, 1024, 0, q>>>(D, B.list, B.count, na, A.live);
        B.live = A.live - na;
        A.live = na;
    }
    double ms_eval = 0.0, ms_k[3] = {0.0, 0.0, 0.0}, ms_c[3] = {0.0, 0.0, 0.0}, full_ms_cand = 0.0;
    unsigned long long hist_prev = 0, full_hist = 0;
    long long full_ticks = 0;
    // Hard cap on ticks: no candidate does more evaluations than this (max_iterations == 0 means unbounded in
    // lbfgs.hpp; the cap then only guards against a runaway loop), times the number of refills of a slot.
    const topay_opt_params& op = s->params.opt;
    auto evals_of = [](const topay_lbfgs_params& lp) -> double {
        const double it = lp.max_iterations > 0 ? lp.max_iterations + 2.0 : 1e7;
        return it * (lp.max_linesearch + 1.0);
    };
    const double per_cand = evals_of(op.s1_lbfgs) + (op.alm_max_rounds + 1.0) * evals_of(op.s2_lbfgs);
    const double waves = std::ceil((double)s->n_cand / std::max(1, s->n_slots_used));
    long long max_ticks = (long long)std::min(per_cand * waves, 4e15);
    if (const char* e = getenv("TOPAY_MAX_TICKS")) max_ticks = std::max(1LL, atoll(e));   // tests: force the cap
    long long ticks = 0;
    long long slot_ticks = 0;      // live slots summed over the batches (upper bound of the evaluations done)
    bool done = false;
    const bool use_graph = !s->timed;
    if (s->graph_max_N != s->max_N) {
        drop_graphs(s);
        s->graph_max_N = s->max_N;
    }
    while (!done && ticks < max_ticks) {
        const int ny = grid_bucket(A.live), ny_b = s->lanes == 2 ? grid_bucket(B.live) : 0;
        const int key = ny | (ny_b << 16);
        if (use_graph) {
            auto it = s->graphs.find(key);
            if (it == s->graphs.end()) {
                cudaGraph_t g = nullptr;
                cudaGraphExec_t ge = nullptr;
                TP_CUDA_OK(cudaStreamBeginCapture(q, cudaStreamCaptureModeThreadLocal), {});
                const TpLaunches launches = enqueue_batch(s, ny, ny_b, false);
                TP_CUDA_OK(cudaStreamEndCapture(q, &g), {});
                TP_CUDA_OK(cudaGraphInstantiate(&ge, g, 0), { cudaGraphDestroy(g); });
                cudaGraphDestroy(g);
                it = s->graphs.emplace(key, TpBatchGraph{ge, launches}).first;
            }
            TP_CUDA_OK(cudaGraphLaunch(it->second.exec, q), {});
            it->second.launches.add_to(s->stats);
        } else {
            enqueue_batch(s, ny, 0, true).add_to(s->stats);
            cudaMemcpyAsync(s->h_nodes, D.node_count, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, q);
        }
        ticks += TP_TICKS;
        slot_ticks += (long long)(A.live + B.live) * TP_TICKS;
        // spin while at most two solves run in this process (lowest latency, one busy core per plan), else sleep
        if (g_solves_running.load(std::memory_order_relaxed) <= 2) {
            TP_CUDA_OK(cudaStreamSynchronize(q), {});
        } else {
            cudaEventRecord(s->ev_batch, q);
            TP_CUDA_OK(cudaEventSynchronize(s->ev_batch), {});
        }
        const int live_after = *A.h_live;
        if (!use_graph) {
            // batches in which every slot was still solving: the full-activity figures
            const bool full = live_after == A.live;
            const unsigned long long hist_now = s->h_nodes[1];
            double cand_batch = 0.0, lbfgs_batch = 0.0;
            for (int t = 0; t < TP_TICKS; t++) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, s->ev[TP_EV * t + 1], s->ev[TP_EV * t + 2]);
                ms_eval += ms;
                cudaEventElapsedTime(&ms, s->ev[TP_EV * t], s->ev[TP_EV * t + 1]);
                ms_k[0] += ms;
                cudaEventElapsedTime(&ms, s->ev[TP_EV * t + 2], s->ev[TP_EV * t + 3]);
                ms_k[1] += ms;
                cudaEventElapsedTime(&ms, s->ev[TP_EV * t + 3], s->ev[TP_EV * t + 6]);
                ms_k[2] += ms;
                cand_batch += ms;
                for (int k = 0; k < 3; k++) {
                    cudaEventElapsedTime(&ms, s->ev[TP_EV * t + 3 + k], s->ev[TP_EV * t + 4 + k]);
                    ms_c[k] += ms;
                    if (k == 1) lbfgs_batch += ms;
                }
            }
            if (full) {
                full_ms_cand += lbfgs_batch;
                full_hist += hist_now - hist_prev;
                full_ticks += TP_TICKS;
            }
            hist_prev = hist_now;
        }
        A.live = live_after;
        if (s->lanes == 2) B.live = *B.h_live;
        done = A.live + B.live == 0;
    }
    if (!done) {
        if (s->lanes == 2) mark_tick_cap(s, B, 0);
        mark_tick_cap(s, A, s->n_cand);
        tp_set_error("tick cap reached: unfinished candidates carry TOPAY_LBFGSERR_TICK_CAP");
    }
    cudaEventRecord(s->ev_end, q);
    cudaMemcpyAsync(s->h_nodes, D.node_count, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, q);
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    cudaEventElapsedTime(&s->stats.ms_total, s->ev_begin, s->ev_end);
    s->stats.ms_eval = (float)ms_eval;
    s->stats.ms_integrate = (float)ms_k[0];
    s->stats.ms_chain = (float)ms_k[1];
    s->stats.ms_cand = (float)ms_k[2];
    s->stats.ms_adj = (float)ms_c[0];
    s->stats.ms_lbfgs = (float)ms_c[1];
    s->stats.ms_gen = (float)ms_c[2];
    s->stats.ticks = ticks;
    s->stats.slot_ticks = slot_ticks;
    s->stats.eval_nodes = (int64_t)s->h_nodes[0];
    s->stats.hist_bytes = (int64_t)s->h_nodes[1] * 16;
    s->stats.full_ticks = full_ticks;
    s->stats.full_hist_bytes = (int64_t)full_hist * 16;
    s->stats.full_ms_cand = (float)full_ms_cand;   // one s_j and one y_j element per row element
    return TOPAY_OK;
}

// Entry c of `out` from a candidate's final state and its piece durations T[0..N); returns the trajectory's duration
// (summed in piece order).
static double fill_result(topay_result_batch* out, int c, const TpCandState& st, const double* T) {
    double dur = 0.0;
    for (int i = 0; i < st.N; i++) dur += T[i];
    out->status[c] = st.status;
    if (out->lbfgs_code) out->lbfgs_code[c] = st.last_code;
    if (out->piece_num) out->piece_num[c] = st.N;
    if (out->iters) out->iters[c] = st.iters_total;
    if (out->evals) out->evals[c] = st.evals_total;
    if (out->alm_rounds) out->alm_rounds[c] = st.alm_round;
    if (out->cost) out->cost[c] = st.cost;
    if (out->duration) out->duration[c] = dur;
    if (out->final_xy_err) {
        out->final_xy_err[2 * c] = st.final_xy[0];
        out->final_xy_err[2 * c + 1] = st.final_xy[1];
    }
    return dur;
}

// A store row holds its candidate's N pieces; the entries past them are whatever an earlier upload's candidate of that
// row left there. They leave the library as zeros, so that a candidate's result does not depend on what the solver
// ran before.
static void clear_tail(topay_result_batch* out, int c, int N, int NP) {
    if (out->T) std::fill(out->T + (size_t)c * NP + N, out->T + (size_t)(c + 1) * NP, 0.0);
    if (out->coeff)
        std::fill(out->coeff + ((size_t)c * 6 * NP + 6 * N) * 9, out->coeff + (size_t)(c + 1) * 6 * NP * 9, 0.0);
}

extern "C" int topay_solver_download(topay_solver* s, topay_result_batch* out, int32_t* best_by_duration,
                                     int32_t* best_by_cost) {
    if (!s || !out || !out->status || s->n_cand < 1) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    const TpSolverDev& D = s->dev;
    const int n = s->n_cand, NP = D.max_pieces;
    std::vector<TpCandState> st(n);
    TP_CUDA_OK(cudaMemcpy(st.data(), D.res_st, n * sizeof(TpCandState), cudaMemcpyDeviceToHost), {});
    std::vector<double> T((size_t)n * NP);
    TP_CUDA_OK(cudaMemcpy(T.data(), D.res_T, T.size() * 8, cudaMemcpyDeviceToHost), {});
    int bd = -1, bc = -1;
    double bdv = 0, bcv = 0;
    int64_t evals = 0;
    for (int c = 0; c < n; c++) {
        const double dur = fill_result(out, c, st[c], &T[(size_t)c * NP]);
        evals += st[c].evals_total;
        if (st[c].status == 1) {
            // planner.cpp:999-1010: first success, replaced only by a strictly shorter duration
            if (bd < 0 || dur < bdv) {
                bd = c;
                bdv = dur;
            }
            if (bc < 0 || st[c].cost < bcv) {
                bc = c;
                bcv = st[c].cost;
            }
        }
    }
    s->stats.evals_total = evals;
    if (out->T) memcpy(out->T, T.data(), T.size() * 8);
    if (out->coeff) TP_CUDA_OK(cudaMemcpy(out->coeff, D.res_coeff, (size_t)n * 6 * NP * 9 * 8, cudaMemcpyDeviceToHost), {});
    if (out->x) {
        std::vector<double> xs((size_t)n * D.xs);
        TP_CUDA_OK(cudaMemcpy(xs.data(), D.res_x, xs.size() * 8, cudaMemcpyDeviceToHost), {});
        const int xstride = topay_num_vars(NP);
        for (int c = 0; c < n; c++) memcpy(out->x + (size_t)c * xstride, &xs[(size_t)c * D.xs], st[c].n * 8);
    }
    for (int c = 0; c < n; c++) clear_tail(out, c, st[c].N, NP);
    if (best_by_duration) *best_by_duration = bd;
    if (best_by_cost) *best_by_cost = bc;
    return TOPAY_OK;
}

extern "C" int topay_solver_solve_batch(topay_solver* s, int n_cand, const int32_t* path_len,
                                        const double* init_paths, const double* bvel, const double* bacc,
                                        topay_result_batch* out, int32_t* best_by_duration, int32_t* best_by_cost) {
    int rc = topay_solver_upload(s, n_cand, path_len, init_paths, bvel, bacc);
    if (rc != TOPAY_OK) return rc;
    rc = topay_solver_run(s);
    if (rc != TOPAY_OK) return rc;
    return topay_solver_download(s, out, best_by_duration, best_by_cost);
}

// Piece counts live in the per-candidate state and the start pose is split over start_xy and the
// yaw slot of head_pva; gather both into the layout the trajectory kernels read.
__global__ void k_solver_traj_view(const TpCandState* __restrict__ st, const double* __restrict__ start_xy,
                                   const double* __restrict__ head_pva, int n, int32_t* pn, double* start) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    pn[c] = st[c].N;
    start[3 * c] = start_xy[2 * c];
    start[3 * c + 1] = start_xy[2 * c + 1];
    start[3 * c + 2] = head_pva[(size_t)c * 27];
}

extern "C" int topay_solver_check_feasible(topay_solver* s, topay_feasibility* out, int32_t* best_success) {
    if (!s || !out || !out->feasible || s->n_cand < 1) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    TpSolverDev& D = s->dev;
    const int n = s->n_cand, NP = D.max_pieces;
    int rc;
    if (!s->checker) {
        if ((rc = dev_alloc(s, &s->d_pn, (size_t)D.max_cand)) != TOPAY_OK) return rc;
        if ((rc = dev_alloc(s, &s->d_start, (size_t)D.max_cand * 3)) != TOPAY_OK) return rc;
        s->checker = new TpTrajChecker();
        if ((rc = s->checker->init(s->device, s->stream)) != TOPAY_OK) return rc;
    }
    k_solver_traj_view<<<(n + 127) / 128, 128, 0, s->stream>>>(D.res_st, D.start_xy, D.head_pva, n, s->d_pn, s->d_start);
    TpTrajView V{n, NP, s->d_pn, D.res_T, D.res_coeff, s->d_start};
    TpGrid G;
    solver_grid(s, &G);
    std::vector<int32_t> fp;
    int32_t* keep_fp = out->feasible_print;
    if (!keep_fp) {   // the gate below needs it
        fp.resize(n);
        out->feasible_print = fp.data();
    }
    rc = s->checker->check(V, s->params, G, out, D.n_fields > 1 ? D.grids : nullptr, D.field_of);
    s->checker->checked_n = rc == TOPAY_OK ? n : 0;
    out->feasible_print = keep_fp;
    if (rc == TOPAY_OK && best_success) {
        // planner.cpp:877-880 + :999-1010: optimizeTraj && printConstraintsSituations, shortest duration — on the device
        const int32_t off[2] = {0, n};
        rc = topay_solver_select(s, 1, off, 1, best_success, nullptr);
    }
    return rc;
}

// Selection on the device (planner.cpp:999-1010: the first success, replaced only by a strictly shorter duration;
// the same rule on the cost): one block per plan walks its candidates, `ok` = optimizeTraj's status and, when the
// gate ran, printConstraintsSituations' verdict (planner.cpp:877-880). Durations are summed in piece order like the
// host loop of topay_solver_download, ties go to the lowest index.
__global__ void __launch_bounds__(128)
k_select(const TpCandState* __restrict__ st, const double* __restrict__ T, int max_pieces,
         const TpFeasOut* __restrict__ feas, const int32_t* __restrict__ plan_off, int32_t* __restrict__ out) {
    const int plan = blockIdx.x, c0 = plan_off[plan], c1 = plan_off[plan + 1];
    int bd = INT32_MAX, bc = INT32_MAX;
    double bdv = 0.0, bcv = 0.0;
    for (int c = c0 + threadIdx.x; c < c1; c += blockDim.x) {
        const bool ok = st[c].status == 1 && (!feas || feas[c].feasible_print != 0);
        if (!ok) continue;
        double dur = 0.0;
        for (int i = 0; i < st[c].N; i++) dur += T[(size_t)c * max_pieces + i];
        if (bd == INT32_MAX || dur < bdv) {
            bd = c;
            bdv = dur;
        }
        if (bc == INT32_MAX || st[c].cost < bcv) {
            bc = c;
            bcv = st[c].cost;
        }
    }
    __shared__ double s_v[2][128];
    __shared__ int s_i[2][128];
    s_v[0][threadIdx.x] = bdv; s_i[0][threadIdx.x] = bd;
    s_v[1][threadIdx.x] = bcv; s_i[1][threadIdx.x] = bc;
    __syncthreads();
    for (int w = 64; w > 0; w >>= 1) {
        if (threadIdx.x < w)
            for (int k = 0; k < 2; k++) {
                const int ia = s_i[k][threadIdx.x], ib = s_i[k][threadIdx.x + w];
                const double va = s_v[k][threadIdx.x], vb = s_v[k][threadIdx.x + w];
                // smaller value wins; equal values: the lower index (= the first in the reference's scan)
                if (ib != INT32_MAX && (ia == INT32_MAX || vb < va || (vb == va && ib < ia))) {
                    s_i[k][threadIdx.x] = ib;
                    s_v[k][threadIdx.x] = vb;
                }
            }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[2 * plan] = s_i[0][0] == INT32_MAX ? -1 : s_i[0][0] - c0;
        out[2 * plan + 1] = s_i[1][0] == INT32_MAX ? -1 : s_i[1][0] - c0;
    }
}

extern "C" int topay_solver_select(topay_solver* s, int n_plans, const int32_t* plan_offset, int use_gate,
                                   int32_t* best_by_duration, int32_t* best_by_cost) {
    if (!s || s->n_cand < 1 || n_plans < 1 || !plan_offset || (!best_by_duration && !best_by_cost))
        return TOPAY_ERR_INVALID_ARG;
    for (int i = 0; i < n_plans; i++)
        if (plan_offset[i] < 0 || plan_offset[i] > plan_offset[i + 1] || plan_offset[i + 1] > s->n_cand)
            return TOPAY_ERR_INVALID_ARG;
    if (use_gate && (!s->checker || s->checker->checked_n != s->n_cand)) {
        tp_set_error("topay_solver_select(use_gate): run topay_solver_check_feasible on this solve first");
        return TOPAY_ERR_NOT_READY;
    }
    cudaSetDevice(s->device);
    const TpSolverDev& D = s->dev;
    int32_t* d = nullptr;
    TP_CUDA_OK(cudaMallocAsync(&d, (size_t)(3 * n_plans + 1) * sizeof(int32_t), s->stream), {});
    int32_t* d_off = d + 2 * n_plans;
    TP_CUDA_OK(cudaMemcpyAsync(d_off, plan_offset, (size_t)(n_plans + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream),
               { cudaFreeAsync(d, s->stream); });
    k_select<<<n_plans, 128, 0, s->stream>>>(D.res_st, D.res_T, D.max_pieces, use_gate ? s->checker->feas : nullptr, d_off, d);
    std::vector<int32_t> h((size_t)2 * n_plans);
    TP_CUDA_OK(cudaMemcpyAsync(h.data(), d, h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, s->stream),
               { cudaFreeAsync(d, s->stream); });
    cudaFreeAsync(d, s->stream);
    TP_CUDA_OK(cudaStreamSynchronize(s->stream), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    for (int i = 0; i < n_plans; i++) {
        if (best_by_duration) best_by_duration[i] = h[2 * i];
        if (best_by_cost) best_by_cost[i] = h[2 * i + 1];
    }
    return TOPAY_OK;
}

// Results of ONE candidate of the last run (the winner): the arrays of `out` have length 1 (T: max_pieces,
// coeff: 6 max_pieces x 9, x: num_vars(max_pieces)).
extern "C" int topay_solver_download_candidate(topay_solver* s, int cand, topay_result_batch* out) {
    if (!s || !out || !out->status || cand < 0 || cand >= s->n_cand) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    const TpSolverDev& D = s->dev;
    const int NP = D.max_pieces;
    TpCandState st;
    TP_CUDA_OK(cudaMemcpyAsync(&st, D.res_st + cand, sizeof(st), cudaMemcpyDeviceToHost, s->stream), {});
    std::vector<double> T(NP);
    TP_CUDA_OK(cudaMemcpyAsync(T.data(), D.res_T + (size_t)cand * NP, NP * 8, cudaMemcpyDeviceToHost, s->stream), {});
    if (out->coeff)
        TP_CUDA_OK(cudaMemcpyAsync(out->coeff, D.res_coeff + (size_t)cand * 6 * NP * 9, (size_t)6 * NP * 9 * 8,
                                   cudaMemcpyDeviceToHost, s->stream), {});
    std::vector<double> xs(out->x ? D.xs : 0);
    if (out->x) TP_CUDA_OK(cudaMemcpyAsync(xs.data(), D.res_x + (size_t)cand * D.xs, (size_t)D.xs * 8, cudaMemcpyDeviceToHost, s->stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(s->stream), {});
    fill_result(out, 0, st, T.data());
    if (out->T) memcpy(out->T, T.data(), (size_t)NP * 8);
    clear_tail(out, 0, st.N, NP);
    if (out->x) memcpy(out->x, xs.data(), (size_t)st.n * 8);
    return TOPAY_OK;
}

// Developer aid: raw copy of one of the evaluation's intermediate device arrays after topay_solver_eval
// (bit-level A/B runs). which: 0 gnode, 1 gsum, 2 gdC, 3 gdT, 4 tot, 5 Ixy, 6 g. Returns the number of
// doubles written (<= cap) or a negative status.
extern "C" int64_t topay_solver_debug_download(topay_solver* s, int which, double* out, int64_t cap) {
    if (!s || !out) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    const TpSolverDev& D = s->dev;
    const size_t C_ = (size_t)D.n_slots, NP = (size_t)D.max_pieces, K = (size_t)D.K;
    const double* src = nullptr;
    size_t n = 0;
    switch (which) {
        case 0: src = D.gnode; n = C_ * NP * (K + 1) * 2; break;
        case 1: src = D.gsum; n = C_ * NP * 2; break;
        case 2: src = D.gdC; n = C_ * 6 * NP * 9; break;
        case 3: src = D.gdT; n = C_ * NP; break;
        case 4: src = D.tot; n = C_ * NP * 2; break;
        case 5: src = D.Ixy; n = C_ * NP * K * 2; break;
        case 6: src = D.g; n = C_ * (size_t)D.xs; break;
        case 7: src = D.gdC_end; n = C_ * NP * 54; break;
        default: return TOPAY_ERR_INVALID_ARG;
    }
    if ((int64_t)n > cap) n = (size_t)cap;
    TP_CUDA_OK(cudaMemcpy(out, src, n * sizeof(double), cudaMemcpyDeviceToHost), {});
    return (int64_t)n;
}

// Parity hook for the L-BFGS direction update (lbfgs.hpp:657-710). Loads a history into slot 0 and runs ONE launch
// of the L-BFGS kernel in which the line search is accepted, the pair (s, y) = (x - xp, g - gp) enters the ring at
// `end`, and the two-loop recursion over min(bound + 1, m) pairs produces the next direction.
extern "C" int topay_solver_debug_direction(topay_solver* s, int n_vars, int bound, int end, const double* S_rows,
                                            const double* Y_rows, const double* ys, const double* x, const double* xp,
                                            const double* g, const double* gp, double* d_out, int32_t* bound_out,
                                            int32_t* end_out) {
    if (!s || !S_rows || !Y_rows || !ys || !x || !xp || !g || !gp || !d_out) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    const TpSolverDev& D = s->dev;
    const int m = std::min(s->params.opt.s2_lbfgs.mem_size, D.mem);
    if (n_vars < 1 || n_vars > D.xs || bound < 0 || bound > m || end < 0 || end >= m) return TOPAY_ERR_INVALID_ARG;
    TpCandState st;
    memset(&st, 0, sizeof(st));
    st.phase = 2;
    st.N = D.max_pieces;
    st.n = n_vars;
    st.k = bound + 1;
    st.end = end;
    st.bound = bound;
    st.stp = 1.0;
    st.finit = st.fx = 1.0;          // |finit - f| = 0: the reference's early accept (lbfgs.hpp:327-330) ends the search
    st.dgtest = st.dstest = -1.0;
    for (int i = 0; i < TP_LBFGS_MAX_PAST; i++) st.pf[i] = 1e30;   // the past-delta test does not stop the run
    st.rho[0] = st.rho[1] = 1.0;
    cudaStream_t q = s->stream;
    auto up = [&](double* dst, const double* src, size_t rows, size_t row_len) {
        std::vector<double> pad(rows * D.xs, 0.0);
        for (size_t r = 0; r < rows; r++) memcpy(&pad[r * D.xs], src + r * row_len, row_len * sizeof(double));
        return cudaMemcpy(dst, pad.data(), pad.size() * sizeof(double), cudaMemcpyHostToDevice);
    };
    TP_CUDA_OK(up(D.x, x, 1, n_vars), {});
    TP_CUDA_OK(up(D.xp, xp, 1, n_vars), {});
    TP_CUDA_OK(up(D.g, g, 1, n_vars), {});
    TP_CUDA_OK(up(D.gp, gp, 1, n_vars), {});
    TP_CUDA_OK(up(D.lm_s, S_rows, m, n_vars), {});
    TP_CUDA_OK(up(D.lm_y, Y_rows, m, n_vars), {});
    TP_CUDA_OK(cudaMemcpy(D.lm_ys, ys, m * sizeof(double), cudaMemcpyHostToDevice), {});
    const double f = 1.0;
    const int32_t zero = 0, one = 1, queue[3] = {1, 1, 0};
    TP_CUDA_OK(cudaMemcpy(D.f, &f, sizeof(double), cudaMemcpyHostToDevice), {});
    TP_CUDA_OK(cudaMemcpy(D.st, &st, sizeof(st), cudaMemcpyHostToDevice), {});
    TP_CUDA_OK(cudaMemcpy(D.slot_gid, &zero, sizeof(int32_t), cudaMemcpyHostToDevice), {});
    TP_CUDA_OK(cudaMemcpy(D.list + (size_t)TP_TICKS * D.n_slots, &zero, sizeof(int32_t), cudaMemcpyHostToDevice), {});
    TP_CUDA_OK(cudaMemcpy(D.count + TP_TICKS, &one, sizeof(int32_t), cudaMemcpyHostToDevice), {});
    TP_CUDA_OK(cudaMemcpy(D.queue, queue, sizeof(queue), cudaMemcpyHostToDevice), {});
    TpLaunches launches;
    launch_cand(s, s->lane[0], TP_MODE_ADVANCE, TP_TICKS, -1, 1, launches);
    launches.add_to(s->stats);
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    s->n_cand = 0;   // not a solvable upload
    TP_CUDA_OK(cudaMemcpy(d_out, D.d, n_vars * sizeof(double), cudaMemcpyDeviceToHost), {});
    TP_CUDA_OK(cudaMemcpy(&st, D.st, sizeof(st), cudaMemcpyDeviceToHost), {});
    if (st.phase != 2) {
        tp_set_error("debug_direction: the crafted iteration did not reach the two-loop (ys <= cautious bound or "
                     "an ascent direction)");
        return TOPAY_ERR_INVALID_ARG;
    }
    if (bound_out) *bound_out = st.bound;
    if (end_out) *end_out = st.end;
    return TOPAY_OK;
}

// Dev profiling: accumulated clock64() deltas of k_cand's phases for candidate 0 (16 slots).
extern "C" int topay_solver_phase_clocks(topay_solver* s, int enable, long long* out16) {
    if (!s) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    TpSolverDev& D = s->dev;
    drop_graphs(s);   // captured kernel arguments change
    if (enable && !D.prof) {
        TP_CUDA_OK(cudaMalloc(&D.prof, 16 * sizeof(long long)), {});
        cudaMemset(D.prof, 0, 16 * sizeof(long long));
    }
    if (out16 && D.prof) {
        TP_CUDA_OK(cudaMemcpy(out16, D.prof, 16 * sizeof(long long), cudaMemcpyDeviceToHost), {});
        cudaMemset(D.prof, 0, 16 * sizeof(long long));
    }
    if (!enable && D.prof) {
        cudaFree(D.prof);
        D.prof = nullptr;
    }
    return TOPAY_OK;
}

extern "C" int topay_solver_set_timed(topay_solver* s, int timed) {
    if (!s) return TOPAY_ERR_INVALID_ARG;
    s->timed = timed != 0;
    return TOPAY_OK;
}

extern "C" int topay_solver_set_trace(topay_solver* s, int cap) {
    if (!s || cap < 0) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(s->device);
    TpSolverDev& D = s->dev;
    drop_graphs(s);   // captured kernel arguments change
    if (D.trace) {
        cudaFree(D.trace);
        cudaFree(D.trace_len);
        D.trace = nullptr;
        D.trace_len = nullptr;
    }
    D.trace_cap = cap;
    if (cap > 0) {
        TP_CUDA_OK(cudaMalloc(&D.trace, (size_t)D.max_cand * cap * 4 * sizeof(double)), {});
        TP_CUDA_OK(cudaMalloc(&D.trace_len, (size_t)D.max_cand * sizeof(int32_t)), {});
        cudaMemset(D.trace_len, 0, (size_t)D.max_cand * sizeof(int32_t));
    }
    return TOPAY_OK;
}

extern "C" int topay_solver_download_trace(topay_solver* s, int cand, double* out, int cap, int32_t* len) {
    if (!s || !out || !len || cand < 0 || cand >= s->dev.max_cand) return TOPAY_ERR_INVALID_ARG;
    const TpSolverDev& D = s->dev;
    if (!D.trace) return TOPAY_ERR_NOT_READY;
    cudaSetDevice(s->device);
    int32_t n = 0;
    TP_CUDA_OK(cudaMemcpy(&n, D.trace_len + cand, sizeof(int32_t), cudaMemcpyDeviceToHost), {});
    n = std::min(n, cap);
    TP_CUDA_OK(cudaMemcpy(out, D.trace + (size_t)cand * D.trace_cap * 4, (size_t)n * 4 * sizeof(double),
                          cudaMemcpyDeviceToHost), {});
    *len = n;
    return TOPAY_OK;
}

extern "C" int topay_solver_last_stats(topay_solver* s, topay_solver_stats* out) {
    if (!s || !out) return TOPAY_ERR_INVALID_ARG;
    *out = s->stats;
    return TOPAY_OK;
}
