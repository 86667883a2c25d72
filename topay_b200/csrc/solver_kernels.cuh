// sm_100a kernels of the batched NLP solve.
//
// One evaluation of all candidates ("tick") is four launches:
//   k_cand      one warp per candidate: [adjoint of the previous evaluation -> f, g] ->
//               [line search / L-BFGS / ALM state machine -> new x] -> [x -> T, q -> banded
//               LU -> spline coefficients]                       (a2,a3,a4,a5,a11-a15 of SURVEY §8a)
//   k_integrate sub-warp per piece: Simpson interval integrals of (s' cos, s' sin)   (a6/a7 prefix)
//   k_penalty   sub-warp per piece, lane per penalty node: ESDF lookups, FK, all penalties,
//               per-piece reduction of gdC / gdT / cost terms                        (a6,a7,a8,a9,a17,a18)
//   k_chain     sub-warp per piece: suffix sums of the xy adjoints and the contraction with
//               the Simpson-prefix Jacobians                                         (a6 tail, :1812-1822)
// Nothing returns to the host between ticks. Candidates live in working SLOTS; the problems of an upload
// (the STORE, indexed by candidate id `gid`) are handed to slots on the device: the moment a slot's candidate
// reaches a terminal state its results go to the store and the same CTA pops the next waiting candidate
// (continuous batching — the reference's "first success + grace" worker pool of planner.cpp:921-952 turned
// into a device-side queue). Every tick runs over the compacted list of live slots only.
#pragma once
#include <type_traits>
#include <cuda_runtime.h>

#include "hd.cuh"
#include "node.cuh"

#define TP_WARPS_PER_BLOCK 4
#define TP_BAND 14   // band width of a stored LU row: 13 band entries + the reciprocal pivot

enum { TP_MODE_ADJ = 1, TP_MODE_ADVANCE = 2, TP_MODE_GEN = 4 };

// Per-candidate scalar state of the device-side solve (lbfgs.hpp:439-722 locals,
// line_search_lewisoverton locals :288-291, and the ALM loop state of
// moma_traj_opt.cpp:395-460).
struct TpCandState {
    int32_t phase;       // 0 = idle / finished, 1 = stage 1, 2 = stage 2
    int32_t N, n;
    int32_t ls_init;     // the evaluation in flight is the initial one of an lbfgs run
    int32_t k, end, bound, ls_count;
    int32_t brackt, touched;
    int32_t s1_past;
    int32_t alm_round;
    int32_t iters_total, evals_total;
    int32_t last_code, status;
    double stp, mu, nu, finit, dgtest, dstest, fx;
    double pf[TP_LBFGS_MAX_PAST];
    double lambda[2], rho[2];
    double final_xy[2];
    double cost;
};

#define TP_TICKS 16   // ticks per batch (one CUDA graph); the live lists form a ring of TP_TICKS + 1 entries

// All device pointers of a solver; strides are fixed by (max_cand, n_slots, max_pieces, K).
// "[store]" arrays are indexed by candidate id (gid < max_cand), "[slot]" arrays by working slot (< n_slots).
struct TpSolverDev {
    int32_t max_cand, n_slots, max_pieces, K, Kpad, ppw, xs, mem;   // xs = stride of x-like vectors
    int32_t smem_doubles;     // dynamic shared memory of k_cand, in doubles
    int32_t end_tasks;        // 1 when K == Kpad: node j = 2K is handled by separate end-node warps
    // [store] problem data + initial state, written by the upload
    double *head_pva, *tail_pva, *start_xy, *end_xy, *init_inner_xy;
    double *x0;               // [store][xs]
    TpCandState* st0;         // [store]
    // [store] results, written by the CTA that finishes the candidate
    TpCandState* res_st;      // [store]
    double *res_T;            // [store][max_pieces]
    double *res_coeff;        // [store][6*max_pieces][9]   coefficients of the last evaluation (what getTraj() returns)
    double *res_x;            // [store][xs]
    // fields: one per solver (the kernels' grid argument), or — scenario sweeps — one per candidate: grids[field_of[gid]]
    const TpGrid* grids;      // [n_fields] or null
    const int32_t* field_of;  // [store]
    int32_t n_fields;         // 0 / 1: the solver's own field
    int32_t pad_fields_;
    // scheduling
    int32_t *slot_gid;        // [slot] candidate in the slot
    int32_t *list;            // [TP_TICKS + 1][n_slots] live slots before tick t
    int32_t *count;           // [TP_TICKS + 1]
    int32_t *queue;           // [0] next gid to hand out, [1] candidates in the store, [2] finished so far
    TpCandState* st;          // [slot]
    // vectors [slot][xs]
    double *x, *g, *xp, *gp, *d;
    // everything below is [slot]-indexed (the comments say max_cand for the slot count)
    // L-BFGS memory: lm_s, lm_y [max_cand][mem][xs]; lm_ys, lm_alpha [max_cand][mem]
    double *lm_s, *lm_y, *lm_ys, *lm_alpha;
    // spline state
    double *T;        // [max_cand][max_pieces]
    double *coeff;    // [max_cand][6*max_pieces][9]
    double *lu;       // [max_cand][6*max_pieces][TP_BAND]
    // evaluation scratch
    double *Ixy;      // [max_cand][max_pieces][K][2]
    double *tot;      // [max_cand][max_pieces][2]
    double *gnode;    // [max_cand][max_pieces][K+1][2]
    double *gsum;     // [max_cand][max_pieces][2]      sum of gnode over nodes 0..K-1 (+K when in-segment)
    double *gdC;      // [max_cand][6*max_pieces][9]    penalty part
    double *gdC_end;  // [max_cand][max_pieces][54]     end-node part (end_tasks only)
    double *gdT;      // [max_cand][max_pieces]         penalty part
    double *gdT_end;  // [max_cand][max_pieces]
    double *terms;    // [max_cand][max_pieces][TOPAY_NTERMS]
    double *terms_end;// [max_cand][max_pieces][TOPAY_NTERMS]
    // outputs of an evaluation
    double *f;        // [max_cand]
    double *term_out; // [max_cand][TOPAY_NTERMS]
    unsigned long long *node_count; // [0] penalty nodes scheduled for evaluation so far; [1] history rows x n
                                    // walked by the two-loop recursions so far (each row = one s_j and one y_j)
    // optional L-BFGS iterate trace (debug / parity): 4 doubles (f, step, k, ls) per accepted iteration
    double *trace;        // [store][trace_cap][4] or null
    int32_t *trace_len;   // [store]
    int32_t trace_cap;
    long long *prof;      // optional phase clocks of candidate 0 (dev profiling), [16] or null
    // first success + grace (topay_solver_set_plans; in a session stream_set_grace or stream_stop, and then plan_of is
    // row_plan and plan_first is indexed by plan id); plan_of is null when it is off, and then nothing else is read
    const int32_t* plan_of;   // [store] plan of the candidate
    int32_t* plan_first;      // [plan] fewest evaluations of a success of the plan published so far (INT32_MAX: none)
    int32_t* pending;         // [0] count, [1 + i] status-1 candidates waiting for the gate (plan_gate only)
    int32_t grace;            // evaluations a plan's candidates may run past its first success
    int32_t plan_gate;        // a success counts once printConstraintsSituations passed (published by the host's gate)
    // streaming session (topay_solver_stream_begin); qrow is null in batch mode, and then nothing below is read. The
    // queue then holds store rows: pop q hands out row qrow[q % max_cand], and queue[3] counts the entries of done_ring.
    int32_t* qrow;            // [max_cand] ring of queued store rows
    const int32_t* row_plan;  // [store] plan slot of the row's candidate
    const int32_t* plan_size; // [plan slot] candidates of the plan
    int32_t* plan_done;       // [plan slot] candidates of the plan that have finished
    int32_t* done_ring;       // [max_cand] plans whose last candidate finished since the host last read the ring
};

// Session: a candidate of row `gid` has written its results; the last one of its plan puts the plan on the done ring.
// The ring and the results are read between batches, after the kernel has ended.
__device__ __forceinline__ void tp_stream_retire(const TpSolverDev& S, int gid) {
    const int p = S.row_plan[gid];
    if (atomicAdd(S.plan_done + p, 1) == S.plan_size[p] - 1) S.done_ring[atomicAdd(S.queue + 3, 1)] = p;
}

// plan_first[] is lowered by other CTAs and by the host's gate while the solve runs; it only ever decreases, so a value
// read at any moment is an upper bound of the final one and a cancellation made against it stands.
__device__ __forceinline__ int32_t tp_load_relaxed(const int32_t* p) {
    int32_t v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// ------------------------------------------------------------------ warp helpers
__device__ __forceinline__ double tp_shfl_xor(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ double tp_shfl_down(double v, int d, int w) { return __shfl_down_sync(0xffffffffu, v, d, w); }
__device__ __forceinline__ double tp_shfl_up(double v, int d, int w) { return __shfl_up_sync(0xffffffffu, v, d, w); }
__device__ __forceinline__ double tp_shfl(double v, int src, int w) { return __shfl_sync(0xffffffffu, v, src, w); }
// butterfly sum over aligned segments of `w` lanes (w power of two); every lane gets the sum
__device__ __forceinline__ double tp_seg_sum(double v, int w) {
    for (int m = w >> 1; m > 0; m >>= 1) v += tp_shfl_xor(v, m);
    return v;
}
__device__ __forceinline__ double tp_warp_sum(double v) { return tp_seg_sum(v, 32); }
__device__ __forceinline__ double tp_warp_max(double v) {
    for (int m = 16; m > 0; m >>= 1) v = fmax(v, tp_shfl_xor(v, m));
    return v;
}

// Live-list lookup shared by the kernels of a tick: entry `li` of list `tick`.
__device__ __forceinline__ int tp_live_slot(const TpSolverDev& S, int tick, int li) {
    if (li >= S.count[tick]) return -1;
    return S.list[(size_t)tick * S.n_slots + li];
}

// Start of a batch (one CTA): the list the previous batch ended with becomes list 0, the other counters are cleared.
__global__ void k_list_roll(const __grid_constant__ TpSolverDev S) {
    const int n = S.count[TP_TICKS];
    for (int i = threadIdx.x; i < n; i += blockDim.x) S.list[i] = S.list[(size_t)TP_TICKS * S.n_slots + i];
    __syncthreads();
    if (threadIdx.x == 0) {
        S.count[0] = n;
        for (int t = 1; t <= TP_TICKS; t++) S.count[t] = 0;
    }
}

// Hands the first n0 candidates of the store to slots 0..n0-1 and makes them the live list TP_TICKS.
__global__ void k_slot_init(const __grid_constant__ TpSolverDev S, int n0, int n_store) {
    const int slot = blockIdx.x;
    if (slot >= n0) return;
    const TpCandState st = S.st0[slot];
    for (int i = threadIdx.x; i < st.n; i += blockDim.x) S.x[(size_t)slot * S.xs + i] = S.x0[(size_t)slot * S.xs + i];
    if (threadIdx.x == 0) {
        S.st[slot] = st;
        S.slot_gid[slot] = slot;
        S.list[(size_t)TP_TICKS * S.n_slots + slot] = slot;
        if (slot == 0) {
            for (int t = 0; t < TP_TICKS; t++) S.count[t] = 0;
            S.count[TP_TICKS] = n0;
            S.queue[0] = n0;
            S.queue[1] = n_store;
            S.queue[2] = 0;
        }
    }
}

// ------------------------------------------------------------------ k_integrate
// Simpson interval integrals of one piece (moma_traj_opt.cpp:1282-1291, 1731-1732):
//   I[k] = coeff v(2k) + 4 coeff v(2k+1) + coeff v(2k+2),  v = s' (cos yaw, sin yaw)
// and the piece totals (IntegralX.sum(), :1750).
__global__ void __launch_bounds__(TP_WARPS_PER_BLOCK * 32)
k_integrate(const __grid_constant__ TpSolverDev S, int tick) {
    const int cand = tp_live_slot(S, tick, blockIdx.y);   // slot
    if (cand < 0) return;
    const TpCandState& cs = S.st[cand];
    if (cs.phase == 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K = S.K, Kpad = S.Kpad;
    const int seg = lane / Kpad, jn = lane % Kpad;
    const int piece = (blockIdx.x * TP_WARPS_PER_BLOCK + warp) * S.ppw + seg;
    const int N = cs.N;
    extern __shared__ double sm[];
    // per warp: ppw segments x (2K+1) slots x 3 values
    const int L = 2 * K + 1;
    double* base = sm + (size_t)(warp * S.ppw + seg) * 3 * L;
    double *s_ds = base, *s_cy = base + L, *s_sy = base + 2 * L;
    const bool valid = piece < N;
    double T = 1.0;
    const double* c = S.coeff;
    if (valid) {
        T = S.T[(size_t)cand * S.max_pieces + piece];
        c = S.coeff + ((size_t)cand * 6 * S.max_pieces + 6 * piece) * 9;
    }
    const double step = T / K, half_step = step / 2.0, coeff = step / 6.0;
    if (valid) {
        double b0[6], b1[6], b2[6];
        TpSlot sl;
        if (jn < K) {
            for (int r = 0; r < 2; r++) {
                const int j = 2 * jn + r;
                tp_slot(c, j * half_step, sl, b0, b1, b2);
                s_ds[j] = sl.ds;
                s_cy[j] = sl.cy;
                s_sy[j] = sl.sy;
            }
        }
        const int end_lane = K < Kpad ? K : 0;
        if (jn == end_lane) {
            tp_slot(c, (2 * K) * half_step, sl, b0, b1, b2);
            s_ds[2 * K] = sl.ds;
            s_cy[2 * K] = sl.cy;
            s_sy[2 * K] = sl.sy;
        }
    }
    __syncwarp();
    double ix = 0.0, iy = 0.0;
    if (valid && jn < K) {
        const int j = 2 * jn;
        // the reference's accumulation order: even node, midpoint, next even node
        ix = coeff * s_ds[j] * s_cy[j];
        iy = coeff * s_ds[j] * s_sy[j];
        ix += 4 * coeff * s_ds[j + 1] * s_cy[j + 1];
        iy += 4 * coeff * s_ds[j + 1] * s_sy[j + 1];
        ix += coeff * s_ds[j + 2] * s_cy[j + 2];
        iy += coeff * s_ds[j + 2] * s_sy[j + 2];
        double* o = S.Ixy + (((size_t)cand * S.max_pieces + piece) * K + jn) * 2;
        o[0] = ix;
        o[1] = iy;
    }
    const double tx = tp_seg_sum(ix, Kpad), ty = tp_seg_sum(iy, Kpad);
    if (valid && jn == 0) {
        double* o = S.tot + ((size_t)cand * S.max_pieces + piece) * 2;
        o[0] = tx;
        o[1] = ty;
    }
}

// ------------------------------------------------------------------ k_penalty
// Lane = one penalty node (even j). Stage 1: calFirstStagePenalGrad's node body; stage 2:
// calSecondStagePenalGrad's. The piece's 6 x 9 spline coefficients are staged in shared
// memory; the per-thread sphere centres / gradients (dynamically indexed) live in shared
// memory too, everything else in registers.
#define TP_PEN_WARPS 2
#ifndef TP_PEN_MIN_BLOCKS
#define TP_PEN_MIN_BLOCKS 6   // 12 warps per SM = 3 per scheduler: 168 registers; needs <= 37 KB of shared memory per block
#endif

// Sum of 64 values per lane over an aligned segment of KPAD lanes with 64/KPAD results per lane
// ("transpose-reduce": each butterfly step halves the values a lane still carries, so the whole
// reduction costs ~64 shuffles instead of 64 x log2(KPAD)). On return v[i], i < 64/KPAD, holds
// the segment sum of element (64/KPAD) * jn + i.
// The 64 inputs come from a generator with a compile-time index, and the first butterfly step consumes them as
// they are produced: a lane never holds more than 32 partial sums (the 64 products of the penalty kernel used
// to sit in 128 registers on top of the operands they are made from).
template <int KPAD, class Gen>
__device__ __forceinline__ void tp_transpose_reduce64(Gen gen, double* v /*[32]*/, int jn) {
    {
        constexpr int m = KPAD >> 1;
        const bool hi = (jn & m) != 0;
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const double a = gen(i), b = gen(i + 32);
            const double send = hi ? a : b;
            const double keep = hi ? b : a;
            v[i] = keep + tp_shfl_xor(send, m);
        }
    }
    int cnt = 32;
#pragma unroll
    for (int m = KPAD >> 2; m > 0; m >>= 1) {
        const bool hi = (jn & m) != 0;
        const int half = cnt >> 1;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            if (i < half) {
                const double send = hi ? v[i] : v[i + half];
                const double keep = hi ? v[i + half] : v[i];
                v[i] = keep + tp_shfl_xor(send, m);
            }
        }
        cnt = half;
    }
}

// MULTI: every candidate reads the field of its own scenario (S.grids[S.field_of[gid]], staged in shared memory once per
// block) instead of the solver's one field (the constant-bank argument G0).
template <int KPAD, bool MULTI = false>
__global__ void __launch_bounds__(TP_PEN_WARPS * 32, TP_PEN_MIN_BLOCKS)
k_penalty(const __grid_constant__ TpSolverDev S, const __grid_constant__ TpParams P,
          const __grid_constant__ TpGrid G0, int n_groups, int tick) {
    const int cand = tp_live_slot(S, tick, blockIdx.y);   // slot
    if (cand < 0) return;
    const TpCandState& cs = S.st[cand];
    if (cs.phase == 0) return;
    const int gid = S.slot_gid[cand];
    __shared__ TpGrid s_grid;
    if (MULTI) {
        const double* src = reinterpret_cast<const double*>(S.grids + S.field_of[gid]);
        double* dst = reinterpret_cast<double*>(&s_grid);
        for (int i = threadIdx.x; i < (int)(sizeof(TpGrid) / sizeof(double)); i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    const TpGrid& G = MULTI ? s_grid : G0;
    const int STAGE = cs.phase;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K = S.K, N = cs.N;
    constexpr int PPW = 32 / KPAD;
    const int task = blockIdx.x * TP_PEN_WARPS + warp;
    const double* start_xy = S.start_xy + (size_t)gid * 2;
    const double* totc = S.tot + (size_t)cand * S.max_pieces * 2;
    extern __shared__ double sm[];
    // [2 stores][36][block threads] sphere stores, then per-warp coefficient staging
    TpSphereStoreStrided pts{sm + threadIdx.x, TP_PEN_WARPS * 32};
    TpSphereStoreStrided pg{sm + 36 * TP_PEN_WARPS * 32 + threadIdx.x, TP_PEN_WARPS * 32};
    double* s_c = sm + 72 * TP_PEN_WARPS * 32 + warp * (PPW * 54);   // PPW pieces x 54 per warp
    double b0[6], b1[6], b2[6];
    TpNodeOut o;

    // Two kinds of task share ONE inlined copy of the node body (the kernel is instruction-fetch bound when the
    // ~6000-instruction stage-2 body exists twice): piece tasks (a segment of KPAD lanes per piece, lane = node) and,
    // when K == KPAD, end-node tasks (lane = piece, node j = 2K).
    const bool end_task = task >= n_groups;
    // With K < KPAD node 2K lives in the piece's own segment; the spare warp that rounds the grid up to whole
    // blocks must not evaluate it a second time (it would race with the segment's lane on gnode[K] with a
    // differently rounded prefix position).
    if (end_task && !S.end_tasks) return;
    const int seg = lane / KPAD, jn = lane % KPAD;
    const int piece = end_task ? (task - n_groups) * 32 + lane : task * PPW + seg;
    const bool pvalid = piece < N;
    const int n_nodes = S.end_tasks ? K : K + 1;   // nodes handled inside a piece task's segment
    const bool active = pvalid && (end_task || jn < n_nodes);
    const int jnode = end_task ? 2 * K : 2 * jn;
    double T = 1.0;
    const double* c = s_c + seg * 54;
    if (pvalid) {
        T = S.T[(size_t)cand * S.max_pieces + piece];
        const double* cgl = S.coeff + ((size_t)cand * 6 * S.max_pieces + 6 * piece) * 9;
        if (end_task) {
            c = cgl;   // every lane has its own piece: straight from global memory
        } else {
            double* cs_ = s_c + seg * 54;
            for (int e = jn; e < 54; e += KPAD) cs_[e] = cgl[e];
        }
    }
    __syncwarp();
    double xy[2] = {0.0, 0.0};
    if (STAGE == 2) {
        if (end_task) {
            // CurrentXY at the end of the piece: start + all intervals up to and including this piece
            double ax = 0.0, ay = 0.0;
            if (pvalid)
                for (int i = 0; i <= piece; i++) {
                    ax += totc[2 * i];
                    ay += totc[2 * i + 1];
                }
            xy[0] = start_xy[0] + ax;
            xy[1] = start_xy[1] + ay;
        } else {
            // CurrentXY (moma_traj_opt.cpp:1302): start + all earlier intervals
            double px = 0.0, py = 0.0;
            if (pvalid)
                for (int i = jn; i < piece; i += KPAD) {
                    px += totc[2 * i];
                    py += totc[2 * i + 1];
                }
            px = tp_seg_sum(px, KPAD);
            py = tp_seg_sum(py, KPAD);
            // inclusive scan of this piece's intervals; node jn sees intervals 0..jn-1
            double ix = 0.0, iy = 0.0;
            if (pvalid && jn < K) {
                const double* I = S.Ixy + (((size_t)cand * S.max_pieces + piece) * K + jn) * 2;
                ix = I[0];
                iy = I[1];
            }
#pragma unroll
            for (int dlt = 1; dlt < KPAD; dlt <<= 1) {
                const double ux = tp_shfl_up(ix, dlt, KPAD), uy = tp_shfl_up(iy, dlt, KPAD);
                if (jn >= dlt) {
                    ix += ux;
                    iy += uy;
                }
            }
            const double ex = tp_shfl_up(ix, 1, KPAD), ey = tp_shfl_up(iy, 1, KPAD);
            xy[0] = start_xy[0] + px + (jn > 0 ? ex : 0.0);
            xy[1] = start_xy[1] + py + (jn > 0 ? ey : 0.0);
        }
    }
    if (active) {
        if (STAGE == 2)
            tp_node_stage2(P, G, c, T, K, jnode, xy, o, b0, b1, b2, pts, pg);
        else
            tp_node_stage1(P, c, T, K, jnode, o, b0, b1, b2);
    } else {
        tp_node_clear(o);
#pragma unroll
        for (int k = 0; k < 6; k++) b0[k] = b1[k] = b2[k] = 0.0;
    }
    if (end_task) {
        if (!pvalid) return;
        double* gc = S.gdC_end + ((size_t)cand * S.max_pieces + piece) * 54;
#pragma unroll
        for (int k = 0; k < 6; k++)
#pragma unroll
            for (int d = 0; d < 9; d++) gc[k * 9 + d] = b0[k] * o.G0[d] + b1[k] * o.G1[d] + b2[k] * o.G2[d];
        S.gdT_end[(size_t)cand * S.max_pieces + piece] = o.gdT;
        double* tm = S.terms_end + ((size_t)cand * S.max_pieces + piece) * TOPAY_NTERMS;
#pragma unroll
        for (int t = 0; t < TOPAY_NTERMS; t++) tm[t] = o.terms[t];
        double* gn = S.gnode + (((size_t)cand * S.max_pieces + piece) * (K + 1) + K) * 2;
        gn[0] = o.gx;
        gn[1] = o.gy;
        return;
    }
    const size_t prow = (size_t)cand * S.max_pieces + piece;
#ifdef TP_DEBUG_NODE
    // dev: inputs / outputs of node K of every piece into the (otherwise unused when K < Kpad) gdC_end rows
    if (active && STAGE == 2 && !S.end_tasks && jn == K) {
        double* dbg = S.gdC_end + prow * 54;
        double sdf, gs[2];
        tp_field_query2d_flat(G, xy, sdf, gs);
        dbg[0] = xy[0]; dbg[1] = xy[1]; dbg[2] = sdf; dbg[3] = gs[0]; dbg[4] = gs[1];
        dbg[5] = o.gx; dbg[6] = o.gy; dbg[7] = T; dbg[8] = c[0]; dbg[9] = c[53];
        dbg[10] = o.G0[0]; dbg[11] = o.G0[1]; dbg[12] = o.gdT; dbg[13] = o.terms[TOPAY_TERM_CHASSIS_COLLI];
        dbg[14] = o.terms[TOPAY_TERM_MANI_COLLI]; dbg[15] = o.G0[2]; dbg[16] = o.G0[5];
    }
#endif
    // per-node xy adjoint, kept for the suffix sums of k_chain, and its sum over the piece
    if (STAGE == 2) {
        if (active) {
            double* gn = S.gnode + ((prow * (K + 1)) + jn) * 2;
            gn[0] = o.gx;
            gn[1] = o.gy;
        }
        const double sx = tp_seg_sum(o.gx, KPAD), sy = tp_seg_sum(o.gy, KPAD);
        if (pvalid && jn == 0) {
            S.gsum[prow * 2] = sx;
            S.gsum[prow * 2 + 1] = sy;
        }
    }
    // reduction over the piece of gdC (54), gdT (1) and the 9 per-node cost terms
    double v[32];
    auto gen = [&](int e) -> double {
        if (e < 54) {
            const int k = e / 9, d = e % 9;
            return b0[k] * o.G0[d] + b1[k] * o.G1[d] + b2[k] * o.G2[d];
        }
        if (e == 54) return o.gdT;
        return o.terms[TOPAY_TERM_CHASSIS_COLLI + (e - 55)];
    };
    tp_transpose_reduce64<KPAD>(gen, v, jn);
    if (pvalid) {
        constexpr int PER = 64 / KPAD;
#pragma unroll
        for (int i = 0; i < PER; i++) {
            const int idx = PER * jn + i;
            if (idx < 54)
                S.gdC[prow * 54 + idx] = v[i];
            else if (idx == 54)
                S.gdT[prow] = v[i];
            else
                S.terms[prow * TOPAY_NTERMS + TOPAY_TERM_CHASSIS_COLLI + (idx - 55)] = v[i];
        }
        if (jn == 0) {
            double* tm = S.terms + prow * TOPAY_NTERMS;
            tm[TOPAY_TERM_JERK] = 0.0;
            tm[TOPAY_TERM_TIME] = 0.0;
            tm[TOPAY_TERM_MEAN_TIME] = 0.0;
            tm[TOPAY_TERM_ENDP] = 0.0;
        }
    }
}

// ------------------------------------------------------------------ k_chain
// Chain weights of every node slot and their contraction with the prefix Jacobians.
// Stage 2: weight of slot (i, j) = sum of the xy adjoints of all penalty nodes at or after it
// (the reference's `head(i*(2K+1)+j+1) +=`, moma_traj_opt.cpp:1313, 1667) + the ALM term (:1809).
// Stage 1: weight of every slot of piece p = sum over pieces i > p of 2 w (F_{i+1} - target_i)
// (`head(i*(2K+1))`, :1175 — piece i itself excluded, reference quirk 1).
__global__ void __launch_bounds__(TP_WARPS_PER_BLOCK * 32)
k_chain(const __grid_constant__ TpSolverDev S, const __grid_constant__ TpParams P, int tick) {
    const int cand = tp_live_slot(S, tick, blockIdx.y);   // slot
    if (cand < 0) return;
    const TpCandState& cs = S.st[cand];
    if (cs.phase == 0) return;
    const int gid = S.slot_gid[cand];
    const int STAGE = cs.phase;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K = S.K, Kpad = S.Kpad, N = cs.N;
    const int seg = lane / Kpad, jn = lane % Kpad;
    const int piece = (blockIdx.x * TP_WARPS_PER_BLOCK + warp) * S.ppw + seg;
    const bool pvalid = piece < N;
    const size_t prow = (size_t)cand * S.max_pieces + piece;
    const double* totc = S.tot + (size_t)cand * S.max_pieces * 2;
    __shared__ double s_w[TP_WARPS_PER_BLOCK][2 * 64 + 2];   // stage 1: per-piece suffix weights

    double wx = 0.0, wy = 0.0;   // weight common to all slots of this piece
    if (STAGE == 1) {
        // F_{i+1} = F_i + tot_i in piece order (VecTrajFinalXY, :1173), then the suffix sums of
        // 2 w (F_{i+1} - target_i); lane 0 of the warp walks the <= 64 pieces once.
        double* w = s_w[warp];
        for (int i = lane; i < N; i += 32) {
            w[2 * i] = totc[2 * i];
            w[2 * i + 1] = totc[2 * i + 1];
        }
        __syncwarp();
        if (lane == 0) {
            const double wgt = P.opt.s1_path_pos_weight;
            const double* tgt = S.init_inner_xy + (size_t)gid * S.max_pieces * 2;
            double fx = S.start_xy[(size_t)gid * 2], fy = S.start_xy[(size_t)gid * 2 + 1];
            for (int i = 0; i < N; i++) {
                fx += w[2 * i];
                fy += w[2 * i + 1];
                w[2 * i] = wgt * 2.0 * (fx - tgt[2 * i]);
                w[2 * i + 1] = wgt * 2.0 * (fy - tgt[2 * i + 1]);
            }
            double sx = 0.0, sy = 0.0;     // suffix over pieces i > p, accumulated in increasing i
            for (int p = N - 1; p >= 0; p--) {
                const double ax = w[2 * p], ay = w[2 * p + 1];
                w[2 * p] = sx;
                w[2 * p + 1] = sy;
                sx += ax;
                sy += ay;
            }
        }
        __syncwarp();
        if (pvalid) {
            wx = w[2 * piece];
            wy = w[2 * piece + 1];
        }
    } else {
        // trajectory end point -> ALM weight (:1786-1810)
        double tx = 0.0, ty = 0.0;
        for (int i = jn; i < N; i += Kpad) {
            tx += totc[2 * i];
            ty += totc[2 * i + 1];
        }
        tx = tp_seg_sum(tx, Kpad);
        ty = tp_seg_sum(ty, Kpad);
        const double ex = S.start_xy[(size_t)gid * 2] + tx - S.end_xy[(size_t)gid * 2];
        const double ey = S.start_xy[(size_t)gid * 2 + 1] + ty - S.end_xy[(size_t)gid * 2 + 1];
        wx = cs.rho[0] * (ex + cs.lambda[0] / cs.rho[0]);
        wy = cs.rho[1] * (ey + cs.lambda[1] / cs.rho[1]);
        // adjoints of all later pieces
        double lx = 0.0, ly = 0.0;
        if (pvalid)
            for (int i = piece + 1 + jn; i < N; i += Kpad) {
                const size_t r = (size_t)cand * S.max_pieces + i;
                lx += S.gsum[r * 2];
                ly += S.gsum[r * 2 + 1];
                if (S.end_tasks) {
                    lx += S.gnode[(r * (K + 1) + K) * 2];
                    ly += S.gnode[(r * (K + 1) + K) * 2 + 1];
                }
            }
        wx += tp_seg_sum(lx, Kpad);
        wy += tp_seg_sum(ly, Kpad);
    }
    // stage 2: suffix sums of this piece's own node adjoints
    double suf_x = 0.0, suf_y = 0.0;     // sum over nodes jn' >= jn (incl. node K)
    double sufn_x = 0.0, sufn_y = 0.0;   // sum over nodes jn' >  jn
    double end_x = 0.0, end_y = 0.0;     // node K alone
    if (STAGE == 2) {
        double gx = 0.0, gy = 0.0;
        if (pvalid && jn < K) {
            const double* gn = S.gnode + ((prow * (K + 1)) + jn) * 2;
            gx = gn[0];
            gy = gn[1];
        }
        if (pvalid) {
            const double* gn = S.gnode + ((prow * (K + 1)) + K) * 2;
            end_x = gn[0];
            end_y = gn[1];
        }
        double sx = gx, sy = gy;
        for (int dlt = 1; dlt < Kpad; dlt <<= 1) {
            const double ux = tp_shfl_down(sx, dlt, Kpad), uy = tp_shfl_down(sy, dlt, Kpad);
            if (jn + dlt < Kpad) {
                sx += ux;
                sy += uy;
            }
        }
        suf_x = sx + end_x;
        suf_y = sy + end_y;
        const double nx = tp_shfl_down(sx, 1, Kpad), ny = tp_shfl_down(sy, 1, Kpad);
        if (jn + 1 < Kpad) {
            sufn_x = nx + end_x;
            sufn_y = ny + end_y;
        } else {
            sufn_x = end_x;
            sufn_y = end_y;
        }
    }
    double gth[6], gar[6], gdt = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) gth[k] = gar[k] = 0.0;
    if (pvalid) {
        const double T = S.T[prow];
        const double* c = S.coeff + (prow * 6) * 9;
        const double half_step = (T / K) / 2.0;
        double b0[6], b1[6], b2[6];
        TpSlot sl;
        if (jn < K) {
            {   // even slot j = 2 jn: Simpson pattern weight 1 at j = 0, else 2
                const int j = 2 * jn;
                const double icc = j == 0 ? 1.0 : 2.0;
                tp_slot(c, j * half_step, sl, b0, b1, b2);
                tp_chain_slot(sl, b0, b1, T, K, j, (wx + suf_x) * icc, (wy + suf_y) * icc, gth, gar, gdt);
            }
            {   // midpoint j = 2 jn + 1: weight 4
                const int j = 2 * jn + 1;
                tp_slot(c, j * half_step, sl, b0, b1, b2);
                tp_chain_slot(sl, b0, b1, T, K, j, (wx + sufn_x) * 4.0, (wy + sufn_y) * 4.0, gth, gar, gdt);
            }
        }
        const int end_lane = K < Kpad ? K : 0;
        if (jn == end_lane) {   // last slot j = 2K: weight 1, only its own node is at/after it
            tp_slot(c, (2 * K) * half_step, sl, b0, b1, b2);
            tp_chain_slot(sl, b0, b1, T, K, 2 * K, wx + end_x, wy + end_y, gth, gar, gdt);
        }
    }
    // Every lane gets the piece sums (butterfly); the read-modify-writes of the piece's outputs are
    // spread over the lanes so that no lane chains more than two dependent global round trips:
    // element e of the 54-entry gdC block goes to lane e % Kpad, together with the end-node part.
    double ath[6], aar[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        ath[k] = tp_seg_sum(gth[k], Kpad);
        aar[k] = tp_seg_sum(gar[k], Kpad);
    }
    gdt = tp_seg_sum(gdt, Kpad);
    if (pvalid) {
        const double* ge = S.gdC_end + prow * 54;
        for (int e = jn; e < 54; e += Kpad) {
            const int k = e / 9, d = e % 9;
            double add = 0.0;
#pragma unroll
            for (int kk = 0; kk < 6; kk++)
                if (kk == k) add = d == 0 ? ath[kk] : (d == 1 ? aar[kk] : 0.0);
            if (S.end_tasks) add += ge[e];
            if (d < 2 || S.end_tasks) S.gdC[prow * 54 + e] += add;
        }
        const int lt = Kpad > TOPAY_NTERMS ? TOPAY_NTERMS : Kpad - 1;   // the lane that owns gdT
        if (jn == lt) S.gdT[prow] += S.end_tasks ? gdt + S.gdT_end[prow] : gdt;
        if (S.end_tasks)
            for (int t = jn; t < TOPAY_NTERMS; t += Kpad)
                S.terms[prow * TOPAY_NTERMS + t] += S.terms_end[prow * TOPAY_NTERMS + t];
    }
}

// ------------------------------------------------------------------ k_cand
// One CTA of TP_CAND_THREADS threads per candidate. Shared memory: the banded LU
// (6N x TP_BAND), the spline coefficients (6N x 9) and one 6N x 9 work matrix.
//
// Banded storage: row i holds A(i, i-6 .. i+6) at lu[i*TP_BAND + (j - i + 6)]; same
// no-pivot elimination, zero tests and operation order per element as
// BandedSystem::factorizeLU / solve / solveAdj (banded_system.hpp:66-145). The 9
// right-hand-side columns are independent, so the substitutions run on three warps of
// three columns each; the L-BFGS vectors live in registers (thread t owns elements
// t, t+128, ...), only the dot products cross threads.
#define TP_CAND_THREADS 128
#define TP_CAND_WARPS (TP_CAND_THREADS / 32)
#define TP_EPT 5      // vector elements per thread: n <= TP_EPT * TP_CAND_THREADS (N <= 64)
#define LU_AT(i, j) lu[(i) * TP_BAND + ((j) - (i) + 6)]
#define LU_DINV(i) lu[(i) * TP_BAND + 13]   // 1 / U(i,i), kept in the row's padding

// 1/x to within ~1 ulp without the IEEE division sequence: hardware seed + 3 Newton steps.
// The banded solves multiply by the reciprocal pivot where the reference divides
// (banded_system.hpp:75,109,128); the difference is <= 2 ulp per operation, far inside the
// 1e-9 parity tolerance, and takes the divide off the 6N-step critical path.
__device__ __forceinline__ double tp_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;   // seed ~2^-20; three steps leave margin for subnormal-free pivots
}

// ---- TMA bulk copies (cp.async.bulk) of L-BFGS history rows into a shared-memory ring ----
#define TP_RING_MAX 32    // most stages of the two-loop's TMA ring (as many as the row size allows)
__device__ __forceinline__ uint32_t tp_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tp_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tp_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void tp_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tp_smem_u32(bar)), "r"(bytes) : "memory");
}
// The L-BFGS history is a pure stream (665 MB per plan against 126 MB of L2): its lines are marked
// evict-first so that they do not push the small per-candidate state (coefficients, LU, adjoints,
// 150 KB per candidate) and the field out of L2 for the other kernels of the tick.
__device__ __forceinline__ uint64_t tp_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tp_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            tp_smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(tp_smem_u32(bar)), "l"(policy)
        : "memory");
}
// 16-byte asynchronous copies (LDGSTS) for the single-warp two-loop of small problems: a history row of a
// 16-piece candidate is < 1.3 KB, and bulk copies of that size complete one after the other (ncu: ~1300 cycles per
// round of four copies, the warp idle on the mbarrier) — 32 lanes x 16 B in flight per instruction do not.
__device__ __forceinline__ void tp_cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tp_smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void tp_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tp_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
#define TP_SOLO_GROUPS 8     // copy groups (rounds) in flight in the single-warp two-loop: 16 ring stages

__device__ __forceinline__ void tp_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(tp_smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}

// block-wide sums of up to 4 values; every thread gets the results. `red` is a
// [2][4][TP_CAND_WARPS] scratch, `flip` alternates so one barrier per call suffices.
template <int NV>
__device__ __forceinline__ void tp_block_sum(double* v, double* red, int& flip) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* r = red + flip * 4 * TP_CAND_WARPS;
#pragma unroll
    for (int q = 0; q < NV; q++) {
        const double w = tp_warp_sum(v[q]);
        if (lane == 0) r[q * TP_CAND_WARPS + warp] = w;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NV; q++) {
        double a = r[q * TP_CAND_WARPS];
#pragma unroll
        for (int w = 1; w < TP_CAND_WARPS; w++) a += r[q * TP_CAND_WARPS + w];
        v[q] = a;
    }
    flip ^= 1;
}
__device__ __forceinline__ double tp_block_max(double v, double* red, int& flip) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* r = red + flip * 4 * TP_CAND_WARPS;
    const double w = tp_warp_max(v);
    if (lane == 0) r[warp] = w;
    __syncthreads();
    double a = r[0];
#pragma unroll
    for (int q = 1; q < TP_CAND_WARPS; q++) a = fmax(a, r[q]);
    flip ^= 1;
    return a;
}

// MinJerkOpt<9>::generate (minco.hpp:824-906): fill A and the right-hand side.
__device__ __forceinline__ void tp_fill_system(int N, const double* T, const double* head, const double* tail,
                                               const double* xin, const TpParams& P, double* lu, double* cf) {
    const int n = 6 * N;
    const int tid = threadIdx.x;
    for (int e = tid; e < n * TP_BAND; e += TP_CAND_THREADS) lu[e] = 0.0;
    for (int e = tid; e < n * 9; e += TP_CAND_THREADS) cf[e] = 0.0;
    __syncthreads();
    // x layout (moma_traj_opt.cpp:324-344): tau(N) | theta(N-1) | arc(N) | vq(7 x (N-1), column-major)
    const double* Theta = xin + N;
    const double* Arc = Theta + (N - 1);
    const double* Vq = Arc + N;
    for (int r = tid; r < n; r += TP_CAND_THREADS) {
        if (r < 3) {
            LU_AT(r, r) = r == 2 ? 2.0 : 1.0;
            for (int d = 0; d < 9; d++) cf[r * 9 + d] = head[d * 3 + r];
        } else if (r >= n - 3) {
            const int i = N - 1;
            const double t1 = T[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2, t5 = t4 * t1;
            const int q = r - (n - 3);
            const int c0 = 6 * N - 6;
            if (q == 0) {
                LU_AT(r, c0) = 1.0; LU_AT(r, c0 + 1) = t1; LU_AT(r, c0 + 2) = t2;
                LU_AT(r, c0 + 3) = t3; LU_AT(r, c0 + 4) = t4; LU_AT(r, c0 + 5) = t5;
            } else if (q == 1) {
                LU_AT(r, c0 + 1) = 1.0; LU_AT(r, c0 + 2) = 2 * t1; LU_AT(r, c0 + 3) = 3 * t2;
                LU_AT(r, c0 + 4) = 4 * t3; LU_AT(r, c0 + 5) = 5 * t4;
            } else {
                LU_AT(r, c0 + 2) = 2; LU_AT(r, c0 + 3) = 6 * t1; LU_AT(r, c0 + 4) = 12 * t2;
                LU_AT(r, c0 + 5) = 20 * t3;
            }
            for (int d = 0; d < 9; d++) {
                double v = tail[d * 3 + q];
                if (d == 1 && q == 0) v = Arc[N - 1];   // minco_end_state(1,0) = Arc[N-1], :905
                cf[r * 9 + d] = v;
            }
        } else {
            const int i = (r - 3) / 6, q = (r - 3) % 6;   // row 6i+3+q
            const double t1 = T[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2, t5 = t4 * t1;
            const int c0 = 6 * i;
            switch (q) {
                case 0:
                    LU_AT(r, c0 + 3) = 6.0; LU_AT(r, c0 + 4) = 24.0 * t1; LU_AT(r, c0 + 5) = 60.0 * t2;
                    LU_AT(r, c0 + 9) = -6.0;
                    break;
                case 1:
                    LU_AT(r, c0 + 4) = 24.0; LU_AT(r, c0 + 5) = 120.0 * t1; LU_AT(r, c0 + 10) = -24.0;
                    break;
                case 2:
                    LU_AT(r, c0) = 1.0; LU_AT(r, c0 + 1) = t1; LU_AT(r, c0 + 2) = t2; LU_AT(r, c0 + 3) = t3;
                    LU_AT(r, c0 + 4) = t4; LU_AT(r, c0 + 5) = t5;
                    cf[r * 9 + 0] = Theta[i];
                    cf[r * 9 + 1] = Arc[i];
                    for (int j = 0; j < TOPAY_DOF; j++)
                        cf[r * 9 + 2 + j] = tp_sigmoidC2(Vq[(size_t)i * TOPAY_DOF + j], P.robot.joint_pos_limit_max[j]);
                    break;
                case 3:
                    LU_AT(r, c0) = 1.0; LU_AT(r, c0 + 1) = t1; LU_AT(r, c0 + 2) = t2; LU_AT(r, c0 + 3) = t3;
                    LU_AT(r, c0 + 4) = t4; LU_AT(r, c0 + 5) = t5; LU_AT(r, c0 + 6) = -1.0;
                    break;
                case 4:
                    LU_AT(r, c0 + 1) = 1.0; LU_AT(r, c0 + 2) = 2 * t1; LU_AT(r, c0 + 3) = 3 * t2;
                    LU_AT(r, c0 + 4) = 4 * t3; LU_AT(r, c0 + 5) = 5 * t4; LU_AT(r, c0 + 7) = -1.0;
                    break;
                default:
                    LU_AT(r, c0 + 2) = 2.0; LU_AT(r, c0 + 3) = 6 * t1; LU_AT(r, c0 + 4) = 12 * t2;
                    LU_AT(r, c0 + 5) = 20 * t3; LU_AT(r, c0 + 8) = -2.0;
                    break;
            }
        }
    }
    __syncthreads();
}

// factorizeLU (banded_system.hpp:66-91) on one warp. Step k updates the 6 x 6 block below / right of
// the pivot: lane e owns element (k+1 + e/6, k+1 + e%6) (lanes 0..3 also own elements 32..35), loads
// everything it needs before the reciprocal pivot is known, then does one multiply-FMA-store; the
// lanes of column k+1 also store the multipliers. One warp barrier per step. Multiplying by an
// exactly zero factor equals the reference's `!= 0.0` skips.
__device__ __forceinline__ void tp_lu_factor(int n, double* lu, int lane) {
    const int r0 = lane / 6, c0 = lane % 6;            // element 0 of this lane
    const int r1 = (lane + 32) / 6, c1 = (lane + 32) % 6;   // element 1 (lanes 0..3 only)
    for (int k = 0; k <= n - 1; k++) {
        const int iM = min(k + 6, n - 1);
        const double piv = LU_AT(k, k);
        const int i0 = k + 1 + r0, j0 = k + 1 + c0;
        const bool ok0 = lane < 36 && i0 <= iM && j0 <= iM;
        double a0 = 0.0, cv0 = 0.0, v0 = 0.0;
        if (ok0) {
            a0 = LU_AT(i0, k);
            cv0 = LU_AT(k, j0);
            v0 = LU_AT(i0, j0);
        }
        const int i1 = k + 1 + r1, j1 = k + 1 + c1;
        const bool ok1 = lane < 4 && i1 <= iM && j1 <= iM;
        double a1 = 0.0, cv1 = 0.0, v1 = 0.0;
        if (ok1) {
            a1 = LU_AT(i1, k);
            cv1 = LU_AT(k, j1);
            v1 = LU_AT(i1, j1);
        }
        const double rinv = tp_rcp(piv);
        __syncwarp();                                  // every lane has read column k
        if (lane == 31) LU_DINV(k) = rinv;
        if (ok0) {
            const double l = a0 * rinv;
            LU_AT(i0, j0) = v0 - l * cv0;
            if (c0 == 0) LU_AT(i0, k) = l;
        }
        if (ok1) {
            const double l = a1 * rinv;
            LU_AT(i1, j1) = v1 - l * cv1;
            if (c1 == 0) LU_AT(i1, k) = l;
        }
        __syncwarp();
    }
}

// The four triangular sweeps of solve / solveAdj (banded_system.hpp:96-145), row-oriented: one
// lane per right-hand-side column walks the rows with the last six solution entries in registers.
// Each element receives its updates in the reference's order (the column index of the factor
// ascending in the forward sweeps, descending in the backward ones), the update with the
// most recent neighbour comes last, so the dependent chain is one FMA (plus the reciprocal-pivot
// multiply) per row and no lane ever waits for another. Slots of the band outside the matrix
// hold zeros, so no bounds tests are needed; multiplying by an exact zero multiplier equals the
// reference's `!= 0.0` skip.
//   mode 0: L y = b   (unit lower, forward)        mode 1: U x = y   (backward)
//   mode 2: U^T y = b (forward)                    mode 3: L^T x = y (unit, backward)
// The triangular sweeps of solve / solveAdj (banded_system.hpp:96-145), one lane per right-hand-side
// column, in the reference's own loop order: as soon as entry i of the solution is known it is
// subtracted from the six rows it couples to. The six pending rows are six independent
// accumulators in registers, so a row costs six independent FMAs and the dependent chain is one
// FMA (+ the reciprocal-pivot multiply for the factor with the non-unit diagonal). The factor
// entries needed when x_i is known are COLUMN i of the triangular factor, i.e. row i of the
// transposed band:
//   solve():    L y = b (forward)  and U x = y (backward)   want the band of A^T  (GEN transposes it in place)
//   solveAdj(): U^T y = b (forward) and L^T x = y (backward) want the band of A    (as stored)
// `m` is that band: row i holds the entries coupling x_i to rows i+1..i+6 in slots 7..12 and to
// rows i-1..i-6 in slots 5..0; slot 13 is the reciprocal pivot. Slots outside the matrix are zero.
template <bool FWD, bool SCALE>
__device__ __forceinline__ void tp_sweep(int n, const double* __restrict__ m, double* b, int cc) {
    double acc0, acc1, acc2, acc3, acc4, acc5;
    if (FWD) {
        acc0 = b[0 * 9 + cc];
        acc1 = n > 1 ? b[1 * 9 + cc] : 0.0;
        acc2 = n > 2 ? b[2 * 9 + cc] : 0.0;
        acc3 = n > 3 ? b[3 * 9 + cc] : 0.0;
        acc4 = n > 4 ? b[4 * 9 + cc] : 0.0;
        acc5 = n > 5 ? b[5 * 9 + cc] : 0.0;
    } else {
        acc0 = b[(n - 1) * 9 + cc];
        acc1 = n > 1 ? b[(n - 2) * 9 + cc] : 0.0;
        acc2 = n > 2 ? b[(n - 3) * 9 + cc] : 0.0;
        acc3 = n > 3 ? b[(n - 4) * 9 + cc] : 0.0;
        acc4 = n > 4 ? b[(n - 5) * 9 + cc] : 0.0;
        acc5 = n > 5 ? b[(n - 6) * 9 + cc] : 0.0;
    }
#pragma unroll 2
    for (int r = 0; r < n; r++) {
        const int i = FWD ? r : n - 1 - r;
        const double2* row = reinterpret_cast<const double2*>(m + i * TP_BAND);
        double c1, c2, c3, c4, c5, c6, dinv;
        if (FWD) {
            const double2 p3 = row[3], p4 = row[4], p5 = row[5], p6 = row[6];   // slots 6..13
            c1 = p3.y; c2 = p4.x; c3 = p4.y; c4 = p5.x; c5 = p5.y; c6 = p6.x;
            dinv = p6.y;
        } else {
            const double2 p0 = row[0], p1 = row[1], p2 = row[2];                 // slots 0..5
            c6 = p0.x; c5 = p0.y; c4 = p1.x; c3 = p1.y; c2 = p2.x; c1 = p2.y;
            dinv = SCALE ? m[i * TP_BAND + 13] : 1.0;
        }
        const int inew = FWD ? i + 6 : i - 6;        // row entering the window
        const double bnew = (inew >= 0 && inew < n) ? b[inew * 9 + cc] : 0.0;
        const double x = SCALE ? acc0 * dinv : acc0;
        b[i * 9 + cc] = x;
        acc0 = acc1 - c1 * x;
        acc1 = acc2 - c2 * x;
        acc2 = acc3 - c3 * x;
        acc3 = acc4 - c4 * x;
        acc4 = acc5 - c5 * x;
        acc5 = bnew - c6 * x;
    }
}

// In-place transpose of the band (slots 0..12 around the diagonal); slot 13 stays.
__device__ __forceinline__ void tp_band_transpose(int n, double* lu) {
    for (int e = threadIdx.x; e < n * 6; e += TP_CAND_THREADS) {
        const int i = e / 6, k = e % 6 + 1;
        if (i + k < n) {
            double* up = lu + i * TP_BAND + 6 + k;          // A(i, i+k)
            double* lo = lu + (i + k) * TP_BAND + 6 - k;    // A(i+k, i)
            const double t = *up;
            *up = *lo;
            *lo = t;
        }
    }
    __syncthreads();
}

// ---- two-loop recursion of small problems (n <= 160: up to 16 pieces) on ONE warp ----
// lbfgs.hpp:691-710. A history row is < 1.3 KB there, a full history 512 dependent steps: the recursion is a pure
// latency chain, so it runs on a single warp (no block barrier) with NE = ceil(n / 32) elements of the vector per
// lane, and the chain is cut four rows at a time. For rows A, B, C, D of a loop (in processing order), u = the vector
// a row is dotted with (s in loop 1, y in loop 2), v = the vector it adds (y in loop 1, s in loop 2):
//   a = u_A.q, b = u_B.q, c = u_C.q, d = u_D.q   and the six cross products  XY = u_X.v_Y  (Y before X)
//   loop 1:  al_A = rho_A a,  al_B = rho_B (b - al_A BA),  al_C = rho_C (c - al_A CA - al_B CB),
//            al_D = rho_D (d - al_A DA - al_B DB - al_C DC);          q -= al_A v_A + al_B v_B + al_C v_C + al_D v_D
//   loop 2:  k_A = al_A - rho_A a,  k_B = al_B - rho_B (b + k_A BA),  ... ;   q += k_A v_A + k_B v_B + k_C v_C + k_D v_D
// which is the recursion with u_X.(q -/+ ...) expanded, so that ten dot products share ONE reduction: a
// transpose-reduce over the warp (16 exchanges instead of 50) and a broadcast through shared memory. The rows of
// step t sit in stage t mod 16 of a shared-memory ring filled by 16-byte asynchronous copies, one commit group per
// step, so "at most 12 groups pending" is exactly "the four rows of this round have landed". Loop tails of fewer than
// four rows take single-row rounds.
#define TP_SOLO_STAGES 16
template <int NE>
__device__ __forceinline__ void tp_two_loop_solo(double* q, int rowd, int bound, int end, int m,
                                                 const double* __restrict__ lm_s, const double* __restrict__ lm_y, int xs,
                                                 const double* s_rho, double* s_alpha, double* s_red /*[16]*/,
                                                 double* ring, double scale, int lane) {
    const int total = 2 * bound;
    const int chunks = rowd >> 1;     // 16-byte chunks per row
    // row of step t: (end-1-t) mod m in the first loop, (end-bound+u) mod m in the second
    auto row_of = [&](int t) {
        int j = t < bound ? end - 1 - t : end - bound + (t - bound);
        j = j < 0 ? j + m : j;
        j = j < 0 ? j + m : j;
        return j >= m ? j - m : j;
    };
    auto issue = [&](int t) {
        if (t < total) {
            const int j = row_of(t);
            double* dst = ring + (t & (TP_SOLO_STAGES - 1)) * 2 * rowd;
            const double* srs = lm_s + (size_t)j * xs;
            const double* sry = lm_y + (size_t)j * xs;
            for (int c = lane; c < chunks; c += 32) {
                tp_cp_async16(dst + 2 * c, srs + 2 * c);
                tp_cp_async16(dst + rowd + 2 * c, sry + 2 * c);
            }
        }
        tp_cp_async_commit();         // also when the history has run out: one group per step, always
    };
    bool in[NE];
#pragma unroll
    for (int e = 0; e < NE; e++) in[e] = lane + 32 * e < rowd;
    // one row: the plain step of the recursion
    auto round1 = [&](auto first_tag, int t) {
        constexpr bool FIRST = decltype(first_tag)::value;
        tp_cp_async_wait<TP_SOLO_STAGES - 4>();
        __syncwarp();
        const int jA = row_of(t);
        const double* stA = ring + (t & (TP_SOLO_STAGES - 1)) * 2 * rowd;
        const double* uAp = FIRST ? stA : stA + rowd;
        const double* vAp = FIRST ? stA + rowd : stA;
        double vA[NE], d0 = 0.0;
#pragma unroll
        for (int e = 0; e < NE; e++) {
            const double u = in[e] ? uAp[lane + 32 * e] : 0.0;
            vA[e] = in[e] ? vAp[lane + 32 * e] : 0.0;
            d0 += u * q[e];
        }
#pragma unroll
        for (int w = 16; w > 0; w >>= 1) d0 += tp_shfl_xor(d0, w);
        __syncwarp();                 // every lane has read the stage: refill it
        issue(t + TP_SOLO_STAGES);
        double k;
        if (FIRST) {
            k = -(d0 * s_rho[jA]);
            if (lane == 0) s_alpha[jA] = -k;
        } else {
            k = s_alpha[jA] - d0 * s_rho[jA];
        }
#pragma unroll
        for (int e = 0; e < NE; e++) q[e] += k * vA[e];
    };
    // four rows
    auto round4 = [&](auto first_tag, int t) {
        constexpr bool FIRST = decltype(first_tag)::value;
        tp_cp_async_wait<TP_SOLO_STAGES - 4>();
        __syncwarp();                 // every lane's chunks of steps t .. t + 3 are in shared memory
        int j[4];
        double v[4][NE];
        double dots[16];              // a b c d | BA CA CB DA DB DC | padding
#pragma unroll
        for (int i = 0; i < 16; i++) dots[i] = 0.0;
        {
            double u[4][NE];
#pragma unroll
            for (int r = 0; r < 4; r++) {
                j[r] = row_of(t + r);
                const double* stp = ring + ((t + r) & (TP_SOLO_STAGES - 1)) * 2 * rowd;
                const double* up = FIRST ? stp : stp + rowd;
                const double* vp = FIRST ? stp + rowd : stp;
#pragma unroll
                for (int e = 0; e < NE; e++) {
                    u[r][e] = in[e] ? up[lane + 32 * e] : 0.0;
                    v[r][e] = in[e] ? vp[lane + 32 * e] : 0.0;
                }
            }
#pragma unroll
            for (int e = 0; e < NE; e++) {
                dots[0] += u[0][e] * q[e];
                dots[1] += u[1][e] * q[e];
                dots[2] += u[2][e] * q[e];
                dots[3] += u[3][e] * q[e];
                dots[4] += u[1][e] * v[0][e];     // BA
                dots[5] += u[2][e] * v[0][e];     // CA
                dots[6] += u[2][e] * v[1][e];     // CB
                dots[7] += u[3][e] * v[0][e];     // DA
                dots[8] += u[3][e] * v[1][e];     // DB
                dots[9] += u[3][e] * v[2][e];     // DC
            }
        }
        // transpose-reduce of 16 values over 32 lanes: after the steps 16, 8, 4, 2 a lane holds one partial sum, of
        // value index (lane >> 1) & ... ; the last step completes it
        {
#pragma unroll
            for (int i = 0; i < 8; i++) {         // step xor 16: keep values [0,8) in the low half, [8,16) in the high
                const bool hi = (lane & 16) != 0;
                const double send = hi ? dots[i] : dots[i + 8];
                const double keep = hi ? dots[i + 8] : dots[i];
                dots[i] = keep + tp_shfl_xor(send, 16);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const bool hi = (lane & 8) != 0;
                const double send = hi ? dots[i] : dots[i + 4];
                const double keep = hi ? dots[i + 4] : dots[i];
                dots[i] = keep + tp_shfl_xor(send, 8);
            }
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const bool hi = (lane & 4) != 0;
                const double send = hi ? dots[i] : dots[i + 2];
                const double keep = hi ? dots[i + 2] : dots[i];
                dots[i] = keep + tp_shfl_xor(send, 4);
            }
            {
                const bool hi = (lane & 2) != 0;
                const double send = hi ? dots[0] : dots[1];
                const double keep = hi ? dots[1] : dots[0];
                dots[0] = keep + tp_shfl_xor(send, 2);
            }
            dots[0] += tp_shfl_xor(dots[0], 1);
            // lane holds value index  8 [lane & 16] + 4 [lane & 8] + 2 [lane & 4] + [lane & 2]
            if (!(lane & 1)) s_red[((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)] = dots[0];
        }
        __syncwarp();                 // sums visible; every lane has read the four stages: refill them
#pragma unroll
        for (int r = 0; r < 4; r++) issue(t + r + TP_SOLO_STAGES);
        const double a = s_red[0], b = s_red[1], c = s_red[2], d = s_red[3];
        const double BA = s_red[4], CA = s_red[5], CB = s_red[6], DA = s_red[7], DB = s_red[8], DC = s_red[9];
        const double rA = s_rho[j[0]], rB = s_rho[j[1]], rC = s_rho[j[2]], rD = s_rho[j[3]];
        double kA, kB, kC, kD;
        if (FIRST) {
            const double alA = a * rA;
            const double alB = (b - alA * BA) * rB;
            const double alC = (c - alA * CA - alB * CB) * rC;
            const double alD = (d - alA * DA - alB * DB - alC * DC) * rD;
            if (lane == 0) {
                s_alpha[j[0]] = alA;
                s_alpha[j[1]] = alB;
                s_alpha[j[2]] = alC;
                s_alpha[j[3]] = alD;
            }
            kA = -alA; kB = -alB; kC = -alC; kD = -alD;
        } else {
            kA = s_alpha[j[0]] - a * rA;
            kB = s_alpha[j[1]] - (b + kA * BA) * rB;
            kC = s_alpha[j[2]] - (c + kA * CA + kB * CB) * rC;
            kD = s_alpha[j[3]] - (d + kA * DA + kB * DB + kC * DC) * rD;
        }
#pragma unroll
        for (int e = 0; e < NE; e++) {
            q[e] += kA * v[0][e];
            q[e] += kB * v[1][e];
            q[e] += kC * v[2][e];
            q[e] += kD * v[3][e];
        }
        __syncwarp();                 // s_red is free for the next round
    };
    for (int t = 0; t < TP_SOLO_STAGES; t++) issue(t);
    int t = 0;
    while (t + 4 <= bound) {
        round4(std::true_type{}, t);
        t += 4;
    }
    while (t < bound) round1(std::true_type{}, t++);
    __syncwarp();                     // the alpha table is complete
#pragma unroll
    for (int e = 0; e < NE; e++) q[e] *= scale;      // between the loops: d *= ys / yy (lbfgs.hpp:701)
    while (t + 4 <= total) {
        round4(std::false_type{}, t);
        t += 4;
    }
    while (t < total) round1(std::false_type{}, t++);
    tp_cp_async_wait<0>();
}

__device__ __forceinline__ bool tp_ok_code(int r) {
    return r == TOPAY_LBFGS_CONVERGENCE || r == TOPAY_LBFGS_CANCELED || r == TOPAY_LBFGS_STOP ||
           r == TOPAY_LBFGSERR_MAXIMUMITERATION;
}

#define TP_PROF(slot) do { if (S.prof && cand == 0 && tid == 0) S.prof[slot] += clock64() - t_prof; t_prof = clock64(); } while (0)

// The three halves are separate launches with their own footprint — the adjoint and generate halves need the
// whole banded system in shared memory (70 KB at 64 pieces: three CTAs per SM, a 45 / 80 us sequential chain each),
// the L-BFGS half only its TMA ring (50 KB: four CTAs per SM, 128 registers) — so that the long two-loop streams
// at a higher occupancy than the banded solves allow. MODE is a compile-time mask of TP_MODE_*; smem_doubles is
// the launch's dynamic shared memory in doubles.
template <int MODE>
__global__ void __launch_bounds__(TP_CAND_THREADS, (MODE == TP_MODE_ADVANCE) ? 4 : 3)
k_cand(const __grid_constant__ TpSolverDev S, const __grid_constant__ TpParams P, int smem_doubles, int tick_in,
       int tick_out) {
    constexpr int mode = MODE;
    const int cand = tp_live_slot(S, tick_in, blockIdx.x);   // slot: every [slot] array below is indexed by it
    if (cand < 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    TpCandState* gs = S.st + cand;
    if (gs->phase == 0) return;
    TpCandState st = *gs;          // uniform copy per thread
    int gid = S.slot_gid[cand];    // candidate of the store in this slot
    long long t_prof = clock64();
    int N = st.N, n = st.n, n6 = 6 * N;
    const int stage = st.phase;
    extern __shared__ __align__(16) double sm[];
    // Dynamic shared memory (70.7 KB at 64 pieces, three CTAs per SM): the banded LU (6N x TP_BAND) and
    // ONE 6N x 9 right-hand-side matrix — the adjoint half solves A^T on `wk`, the generate half solves A
    // on `cf`, never at the same time; the adjoint half reads the coefficients straight from global
    // memory (element-wise, off the sequential path). The two-loop recursion reuses the whole region as
    // its TMA ring + the alpha / 1/ys tables.
    double* lu = sm;
    double* cf = lu + (size_t)6 * S.max_pieces * TP_BAND;
    double* wk = cf;
    double* s_alpha = sm + smem_doubles - (512 + S.xs);   // tables + scratch at the end of the region
    double* s_ys = s_alpha + 256;
    __shared__ double red[2 * 4 * TP_CAND_WARPS];
    __shared__ double s_small[4 * 64 + 2 * TOPAY_NTERMS];   // T, totals (x,y), scratch
    __shared__ uint64_t s_bar[TP_RING_MAX];
    if (tid == 0) {
#pragma unroll
        for (int q = 0; q < TP_RING_MAX; q++) tp_mbar_init(&s_bar[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
#ifdef TP_DEBUG_ZERO_SMEM
    for (int e = tid; e < smem_doubles; e += TP_CAND_THREADS) sm[e] = TP_DEBUG_ZERO_SMEM;
    __syncthreads();
#endif
    int flip = 0;
    double* x = S.x + (size_t)cand * S.xs;
    double* g = S.g + (size_t)cand * S.xs;
    double* xp = S.xp + (size_t)cand * S.xs;
    double* gp = S.gp + (size_t)cand * S.xs;
    double* dv = S.d + (size_t)cand * S.xs;
    double* Tg = S.T + (size_t)cand * S.max_pieces;
    double* cg = S.coeff + (size_t)cand * 6 * S.max_pieces * 9;
    double* lug = S.lu + (size_t)cand * 6 * S.max_pieces * TP_BAND;
    const topay_lbfgs_params& lp = stage == 1 ? P.opt.s1_lbfgs : P.opt.s2_lbfgs;
    const int past = stage == 1 ? st.s1_past : lp.past;
    double f_eval = 0.0;

    // ================= adjoint half of the evaluation in flight =================
    if constexpr ((mode & TP_MODE_ADJ) != 0) {
        for (int e = tid; e < n6 * TP_BAND; e += TP_CAND_THREADS) lu[e] = lug[e];
        const double* cfr = cg;   // coefficients of this evaluation, written by the previous launch
        const double* gdCp = S.gdC + (size_t)cand * 6 * S.max_pieces * 9;
        const double* gdTp = S.gdT + (size_t)cand * S.max_pieces;
        const double* tmp = S.terms + (size_t)cand * S.max_pieces * TOPAY_NTERMS;
        const double* totc = S.tot + (size_t)cand * S.max_pieces * 2;
        double* sT = s_small;
        double* sTot = s_small + 64;
        double* sTerm = s_small + 192;
        double* sMisc = sTerm + TOPAY_NTERMS;   // fx, fy, cost_path, avg_time, tsum, mt_all
        for (int i = tid; i < N; i += TP_CAND_THREADS) {
            sT[i] = Tg[i];
            sTot[2 * i] = totc[2 * i];
            sTot[2 * i + 1] = totc[2 * i + 1];
        }
        // cost terms: fixed-tree sum over pieces, one warp per term
        for (int t = warp; t < TOPAY_NTERMS; t += TP_CAND_WARPS) {
            double a = 0.0;
            for (int i = lane; i < N; i += 32) a += tmp[i * TOPAY_NTERMS + t];
            a = tp_warp_sum(a);
            if (lane == 0) sTerm[t] = a;
        }
        __syncthreads();
        TP_PROF(0);
        if (tid == 0) {
            // end point, VecTrajFinalXY order (:1750); stage-1 path cost (:1173-1178)
            double fx = S.start_xy[gid * 2], fy = S.start_xy[gid * 2 + 1];
            double cost_path = 0.0, avg = 0.0;
            const double* tgt = S.init_inner_xy + (size_t)gid * S.max_pieces * 2;
            for (int i = 0; i < N; i++) {
                fx += sTot[2 * i];
                fy += sTot[2 * i + 1];
                avg += sT[i];
                if (stage == 1) {
                    const double ex = fx - tgt[2 * i], ey = fy - tgt[2 * i + 1];
                    cost_path += P.opt.s1_path_pos_weight * (ex * ex + ey * ey);
                }
            }
            const double tsum = avg;
            avg /= N;
            // mean-time penalty (:1752-1769, hard-coded 0.5 / 2.0) — stage 2 only
            double mt_all = 0.0, mt_cost = 0.0;
            if (stage == 2) {
                const double w_mt = P.opt.s2_mean_time_weight;
                for (int i = 0; i < N; i++) {
                    const double ti = sT[i];
                    if (ti < avg * 0.5) {
                        mt_cost += w_mt * (ti - avg * 0.5) * (ti - avg * 0.5);
                        mt_all += w_mt * 2.0 * (ti - avg * 0.5) * (-0.5 / N);
                    }
                    if (ti > avg * 2.0) {
                        mt_cost += w_mt * (ti - avg * 2.0) * (ti - avg * 2.0);
                        mt_all += w_mt * 2.0 * (ti - avg * 2.0) * (-2.0 / N);
                    }
                }
            }
            sMisc[0] = fx - S.end_xy[gid * 2];
            sMisc[1] = fy - S.end_xy[gid * 2 + 1];
            sMisc[2] = cost_path;
            sMisc[3] = avg;
            sMisc[4] = tsum;
            sMisc[5] = mt_all;
            sMisc[6] = mt_cost;
        }
        __syncthreads();
        st.final_xy[0] = sMisc[0];
        st.final_xy[1] = sMisc[1];
        const double avg_time = sMisc[3], tsum = sMisc[4], mt_all = sMisc[5];
        double terms[TOPAY_NTERMS];
        for (int t = 0; t < TOPAY_NTERMS; t++) terms[t] = sTerm[t];
        if (stage == 2) {
            terms[TOPAY_TERM_MEAN_TIME] += sMisc[6];
            terms[TOPAY_TERM_ENDP] =
                0.5 * (st.rho[0] * (st.final_xy[0] + st.lambda[0] / st.rho[0]) * (st.final_xy[0] + st.lambda[0] / st.rho[0]) +
                       st.rho[1] * (st.final_xy[1] + st.lambda[1] / st.rho[1]) * (st.final_xy[1] + st.lambda[1] / st.rho[1]));
        } else {
            terms[TOPAY_TERM_ENDP] = sMisc[2];
        }
        double pen = 0.0;
        bool bad = false;
        for (int t = TOPAY_TERM_CHASSIS_COLLI; t < TOPAY_NTERMS; t++) {
            pen += terms[t];
            if (isinf(terms[t]) || isnan(terms[t])) bad = true;
        }
        if (stage == 1) bad = false;          // the guard exists in stage 2 only (:1790-1807)
        if (bad) pen = 1.0e+22;
        // jerk cost (minco.hpp:923-942)
        double js[1] = {0.0};
        for (int i = tid; i < N; i += TP_CAND_THREADS) {
            const double t1 = sT[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2, t5 = t4 * t1;
            const double *c3 = cfr + (6 * i + 3) * 9, *c4 = c3 + 9, *c5 = c4 + 9;
            double d33 = 0, d43 = 0, d44 = 0, d53 = 0, d54 = 0, d55 = 0;
            for (int d = 0; d < 9; d++) {
                const double w = P.opt.energy_weights[d];
                d33 += (c3[d] * w) * c3[d];
                d43 += (c4[d] * w) * c3[d];
                d44 += (c4[d] * w) * c4[d];
                d53 += (c5[d] * w) * c3[d];
                d54 += (c5[d] * w) * c4[d];
                d55 += (c5[d] * w) * c5[d];
            }
            js[0] += 36.0 * d33 * t1 + 144.0 * d43 * t2 + 192.0 * d44 * t3 + 240.0 * d53 * t3 + 720.0 * d54 * t4 +
                     720.0 * d55 * t5;
        }
        tp_block_sum<1>(js, red, flip);
        const double jerk = js[0];
        TP_PROF(1);
        // gdC = jerk part (minco.hpp:951-977) + penalty part -> wk
        for (int e = tid; e < n6 * 9; e += TP_CAND_THREADS) {
            const int r = e / 9, d = e % 9, i = r / 6, q = r % 6;
            const double t1 = sT[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2, t5 = t4 * t1;
            const double w = P.opt.energy_weights[d];
            const double c3 = cfr[(6 * i + 3) * 9 + d], c4 = cfr[(6 * i + 4) * 9 + d], c5 = cfr[(6 * i + 5) * 9 + d];
            double v = 0.0;
            if (q == 5) v = 240.0 * c3 * w * t3 + 720.0 * c4 * w * t4 + 1440.0 * c5 * w * t5;
            else if (q == 4) v = 144.0 * c3 * w * t2 + 384.0 * c4 * w * t3 + 720.0 * c5 * w * t4;
            else if (q == 3) v = 72.0 * c3 * w * t1 + 144.0 * c4 * w * t2 + 240.0 * c5 * w * t3;
            wk[e] = v + (bad ? 0.0 : gdCp[e]);
        }
        __syncthreads();
        TP_PROF(2);
        if (tid < 9) {
            tp_sweep<true, true>(n6, lu, wk, tid);     // U^T y = b  (solveAdj, first loop)
            tp_sweep<false, false>(n6, lu, wk, tid);   // L^T x = y  (second loop)
        }
        __syncthreads();
        TP_PROF(3);
        // gradients w.r.t. the variables (:939-948) with calGradCTtoQT's gdT part (minco.hpp:1016-1067)
        const double tw = stage == 1 ? P.opt.s1_time_weight : P.opt.s2_time_weight;
        const double* Tau = x;
        const double* Vq = x + N + (N - 1) + N;
        double* gTau = g;
        double* gTheta = g + N;
        double* gArc = gTheta + (N - 1);
        double* gVq = gArc + N;
        for (int i = tid; i < N; i += TP_CAND_THREADS) {
            const double t1 = sT[i], t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2;
            const double *c1 = cfr + (6 * i + 1) * 9, *c2 = c1 + 9, *c3 = c2 + 9, *c4 = c3 + 9, *c5 = c4 + 9;
            double d33 = 0, d43 = 0, d44 = 0, d53 = 0, d54 = 0, d55 = 0;
            for (int d = 0; d < 9; d++) {
                const double w = P.opt.energy_weights[d];
                d33 += (c3[d] * w) * c3[d];
                d43 += (c4[d] * w) * c3[d];
                d44 += (c4[d] * w) * c4[d];
                d53 += (c5[d] * w) * c3[d];
                d54 += (c5[d] * w) * c4[d];
                d55 += (c5[d] * w) * c5[d];
            }
            double gt = 36.0 * d33 + 288.0 * d43 * t1 + 576.0 * d44 * t2 + 720.0 * d53 * t2 + 2880.0 * d54 * t3 +
                        3600.0 * d55 * t4;
            if (!bad) gt += gdTp[i] + mt_all;
            if (!bad && stage == 2) {
                const double w_mt = P.opt.s2_mean_time_weight;
                if (t1 < avg_time * 0.5) gt += w_mt * 2.0 * (t1 - avg_time * 0.5);
                if (t1 > avg_time * 2.0) gt += w_mt * 2.0 * (t1 - avg_time * 2.0);
            }
            double s = 0.0;
            if (i < N - 1) {
                for (int d = 0; d < 9; d++) {
                    const double vel = -(c1[d] + 2.0 * t1 * c2[d] + 3.0 * t2 * c3[d] + 4.0 * t3 * c4[d] + 5.0 * t4 * c5[d]);
                    const double acc = -(2.0 * c2[d] + 6.0 * t1 * c3[d] + 12.0 * t2 * c4[d] + 20.0 * t3 * c5[d]);
                    const double jer = -(6.0 * c3[d] + 24.0 * t1 * c4[d] + 60.0 * t2 * c5[d]);
                    const double snp = -(24.0 * c4[d] + 120.0 * t1 * c5[d]);
                    const double crk = -120.0 * c5[d];
                    const double* a = wk + (6 * i + 3) * 9 + d;
                    s += snp * a[0] + crk * a[9] + vel * a[18] + vel * a[27] + acc * a[36] + jer * a[45];
                }
            } else {
                for (int d = 0; d < 9; d++) {
                    const double vel = -(c1[d] + 2.0 * t1 * c2[d] + 3.0 * t2 * c3[d] + 4.0 * t3 * c4[d] + 5.0 * t4 * c5[d]);
                    const double acc = -(2.0 * c2[d] + 6.0 * t1 * c3[d] + 12.0 * t2 * c4[d] + 20.0 * t3 * c5[d]);
                    const double jer = -(6.0 * c3[d] + 24.0 * t1 * c4[d] + 60.0 * t2 * c5[d]);
                    const double* a = wk + (6 * N - 3) * 9 + d;
                    s += vel * a[0] + acc * a[9] + jer * a[18];
                }
            }
            gt += s;
            gTau[i] = (gt + tw) * tp_dT_dtau(Tau[i]);
            if (i < N - 1) {
                const double* a = wk + (6 * i + 5) * 9;
                gTheta[i] = a[0];
                gArc[i] = a[1];
                for (int j = 0; j < TOPAY_DOF; j++)
                    gVq[(size_t)i * TOPAY_DOF + j] =
                        a[2 + j] * tp_dq_dvq(Vq[(size_t)i * TOPAY_DOF + j], P.robot.joint_pos_limit_max[j]);
            } else {
                gArc[N - 1] = wk[(6 * N - 3) * 9 + 1];   // gdP_tail(1, 0)
            }
        }
        __syncthreads();
        terms[TOPAY_TERM_JERK] = jerk;
        terms[TOPAY_TERM_TIME] = tw * tsum;
        f_eval = jerk + pen + tw * tsum;
        if (tid == 0) {
            S.f[cand] = f_eval;
            for (int t = 0; t < TOPAY_NTERMS; t++) S.term_out[(size_t)cand * TOPAY_NTERMS + t] = terms[t];
        }
        st.evals_total++;
        TP_PROF(4);
    }

    // ================= line search / L-BFGS / ALM state machine =================
    bool need_eval = true;
    if constexpr ((mode & TP_MODE_ADVANCE) != 0) {
        const int m = lp.mem_size < S.mem ? lp.mem_size : S.mem;
        double* lm_s = S.lm_s + (size_t)cand * S.mem * S.xs;
        double* lm_y = S.lm_y + (size_t)cand * S.mem * S.xs;
        double* lm_ys = S.lm_ys + (size_t)cand * S.mem;
        // this thread's elements of the five vectors
        double rx[TP_EPT], rg[TP_EPT], rxp[TP_EPT], rgp[TP_EPT], rd[TP_EPT];
#pragma unroll
        for (int e = 0; e < TP_EPT; e++) {
            const int i = tid + e * TP_CAND_THREADS;
            const bool in = i < n;
            rx[e] = in ? x[i] : 0.0;
            rg[e] = in ? g[i] : 0.0;
            rxp[e] = in ? xp[i] : 0.0;
            rgp[e] = in ? gp[i] : 0.0;
            rd[e] = in ? dv[i] : 0.0;
        }
        int ret = 0;
        enum { A_NONE, A_BEGIN_LS, A_LS_DONE, A_FINISH } action = A_NONE;
        const double f = (mode & TP_MODE_ADJ) ? f_eval : S.f[cand];   // a separate adjoint launch left it in S.f
        // first success + grace: past grace evaluations after its plan's earliest success the candidate is cancelled
        // (one thread reads the bound, so that the whole CTA takes the same branch)
        bool cancel = false;
        if (S.plan_of) {
            __shared__ int s_cancel;
            if (tid == 0) s_cancel = st.evals_total - S.grace > tp_load_relaxed(S.plan_first + S.plan_of[gid]);
            __syncthreads();
            cancel = s_cancel != 0;
        }
        if (cancel) {
            ret = TOPAY_LBFGSERR_PLAN_GRACE;
            action = A_FINISH;
        } else if (st.ls_init) {
            // lbfgs.hpp:522-554
            st.ls_init = 0;
            st.fx = f;
            st.pf[0] = f;
            double gm = 0.0, xm = 0.0, dd[1] = {0.0};
#pragma unroll
            for (int e = 0; e < TP_EPT; e++) {
                rd[e] = -rg[e];
                gm = fmax(gm, fabs(rg[e]));
                xm = fmax(xm, fabs(rx[e]));
                dd[0] += rd[e] * rd[e];
            }
            gm = tp_block_max(gm, red, flip);
            xm = tp_block_max(xm, red, flip);
            st.k = 0;
            if (gm / fmax(1.0, xm) < lp.g_epsilon) {
                ret = TOPAY_LBFGS_CONVERGENCE;
                action = A_FINISH;
            } else {
                tp_block_sum<1>(dd, red, flip);
                st.stp = 1.0 / sqrt(dd[0]);
                st.k = 1;
                st.end = 0;
                st.bound = 0;
                action = A_BEGIN_LS;
            }
        } else {
            // one trip of line_search_lewisoverton's loop, lbfgs.hpp:319-387
            st.ls_count++;
            st.fx = f;
            bool done = false, fail = false;
            if (isinf(f) || isnan(f)) {
                ret = TOPAY_LBFGSERR_INVALID_FUNCVAL;
                fail = true;
            } else if (past > 0 && fabs(st.finit - f) / (fabs(st.finit) + 1.0) < lp.delta / past) {
                done = true;   // reference-specific early accept, :327-330
            } else {
                if (f > st.finit + st.stp * st.dgtest) {
                    st.nu = st.stp;
                    st.brackt = 1;
                } else {
                    double gs_[1] = {0.0};
#pragma unroll
                    for (int e = 0; e < TP_EPT; e++) gs_[0] += rg[e] * rd[e];
                    tp_block_sum<1>(gs_, red, flip);
                    if (gs_[0] < st.dstest)
                        st.mu = st.stp;
                    else
                        done = true;
                }
                if (!done) {
                    if (lp.max_linesearch <= st.ls_count) {
                        ret = TOPAY_LBFGSERR_MAXIMUMLINESEARCH;
                        fail = true;
                    } else if (st.brackt && (st.nu - st.mu) < lp.machine_prec * st.nu) {
                        ret = TOPAY_LBFGSERR_WIDTHTOOSMALL;
                        fail = true;
                    } else {
                        if (st.brackt)
                            st.stp = 0.5 * (st.mu + st.nu);
                        else
                            st.stp *= 2.0;
                        if (st.stp < lp.min_step) {
                            ret = TOPAY_LBFGSERR_MINIMUMSTEP;
                            fail = true;
                        } else if (st.stp > lp.max_step) {
                            if (st.touched) {
                                ret = TOPAY_LBFGSERR_MAXIMUMSTEP;
                                fail = true;
                            } else {
                                st.touched = 1;
                                st.stp = lp.max_step;
                            }
                        }
                    }
                }
            }
            if (fail) {
                // lbfgs.hpp:575-582: revert to the previous point
#pragma unroll
                for (int e = 0; e < TP_EPT; e++) {
                    rx[e] = rxp[e];
                    rg[e] = rgp[e];
                }
                action = A_FINISH;
            } else if (done) {
                action = A_LS_DONE;
            } else {
#pragma unroll
                for (int e = 0; e < TP_EPT; e++) rx[e] = rxp[e] + st.stp * rd[e];
            }
        }
        if (action == A_LS_DONE) {
            // lbfgs.hpp:584-715
            const int k = st.k;
            bool fin = false;
            if (S.trace && tid == 0) {   // where the reference calls proc_progress (:585-592)
                const int tl = S.trace_len[gid];
                if (tl < S.trace_cap) {
                    double* tr = S.trace + ((size_t)gid * S.trace_cap + tl) * 4;
                    tr[0] = st.fx;
                    tr[1] = st.stp;
                    tr[2] = (double)k;
                    tr[3] = (double)st.ls_count;
                    S.trace_len[gid] = tl + 1;
                }
            }
            if (stage == 2 && k > lp.max_iterations) {   // progress callback earlyExit, :1873
                ret = TOPAY_LBFGS_CANCELED;
                fin = true;
            }
            if (!fin && lp.g_epsilon > 0.0) {
                double gm = 0.0, xm = 0.0;
#pragma unroll
                for (int e = 0; e < TP_EPT; e++) {
                    gm = fmax(gm, fabs(rg[e]));
                    xm = fmax(xm, fabs(rx[e]));
                }
                gm = tp_block_max(gm, red, flip);
                xm = tp_block_max(xm, red, flip);
                if (gm / fmax(1.0, xm) < lp.g_epsilon) {
                    ret = TOPAY_LBFGS_CONVERGENCE;
                    fin = true;
                }
            }
            if (!fin && 0 < past) {
                if (past <= k) {
                    const double rate = fabs(st.pf[k % past] - st.fx) / fmax(1.0, fabs(st.fx));
                    if (rate < lp.delta) {
                        ret = TOPAY_LBFGS_STOP;
                        fin = true;
                    }
                }
                if (!fin) st.pf[k % past] = st.fx;
            }
            if (!fin && lp.max_iterations != 0 && lp.max_iterations <= k) {
                ret = TOPAY_LBFGSERR_MAXIMUMITERATION;
                fin = true;
            }
            if (fin) {
                action = A_FINISH;
            } else {
                st.k = k + 1;
                double* se = lm_s + (size_t)st.end * S.xs;
                double* ye = lm_y + (size_t)st.end * S.xs;
                double q4[4] = {0.0, 0.0, 0.0, 0.0};   // ys, yy, ss, gg
#pragma unroll
                for (int e = 0; e < TP_EPT; e++) {
                    const int i = tid + e * TP_CAND_THREADS;
                    const double sv = rx[e] - rxp[e], yv = rg[e] - rgp[e];
                    if (i < n) {
                        se[i] = sv;
                        ye[i] = yv;
                    } else if (i == n && (n & 1)) {
                        se[i] = 0.0;      // the pad element of an odd-length row: the copies move rowd = n + 1 doubles
                        ye[i] = 0.0;
                    }
                    q4[0] += yv * sv;
                    q4[1] += yv * yv;
                    q4[2] += sv * sv;
                    q4[3] += rgp[e] * rgp[e];
                    rd[e] = -rg[e];
                }
                for (int j = tid; j < m; j += TP_CAND_THREADS) s_ys[j] = 1.0 / lm_ys[j];   // reciprocals
                tp_block_sum<4>(q4, red, flip);
                const double ys = q4[0], yy = q4[1];
                if (tid == 0) {
                    lm_ys[st.end] = ys;
                    s_ys[st.end] = 1.0 / ys;
                }
                const double cau = q4[2] * sqrt(q4[3]) * lp.cautious_factor;
                TP_PROF(5);
                if (ys > cau) {
                    st.bound = st.bound + 1 < m ? st.bound + 1 : m;
                    st.end = (st.end + 1) % m;
                    // this thread's part of the new history row must be visible to the bulk-copy engine
                    asm volatile("fence.proxy.async;" ::: "memory");
                    __syncthreads();   // s_ys / the new history row are visible
                    // two-loop recursion (lbfgs.hpp:691-710). The 2*bound history rows it walks —
                    // newest to oldest, then oldest to newest — are streamed by TMA bulk copies
                    // into a ring of shared-memory stages (the LU / coefficient region is free
                    // during this phase), `nst` rows of (s_j, y_j) ahead of their use. Only the n live
                    // elements of a row are copied, so small problems get a deep ring (up to 32 rows in
                    // flight) and their short rounds do not wait on the copy latency.
                    const int total = 2 * st.bound;
                    const int rowd = (n + 1) & ~1;                       // 16-byte multiple
                    const uint32_t row_bytes = (uint32_t)(rowd * sizeof(double));
                    const int ring_doubles = smem_doubles - (512 + S.xs);
                    // Small problems (n <= 160, i.e. up to 16 pieces) run the whole recursion on warp 0
                    // with the vector held 5 elements per lane: no block barrier, no shared-memory
                    // partial sums — the 512 rounds of a full history are pure latency at that size.
                    const bool solo = n <= TP_EPT * 32;
                    // even: rounds take two; the single-warp variant keeps exactly 2 * TP_SOLO_GROUPS stages
                    const int nst = solo ? 2 * TP_SOLO_GROUPS : max(2, min(TP_RING_MAX, ring_doubles / (2 * rowd)) & ~1);
                    double* ring = sm;
                    const uint64_t pol = tp_policy_evict_first();
                    // row of step t: (end-1-t) mod m in the first loop, (end-bound+u) mod m in the second;
                    // all operands are within (-2m, 2m), so two conditional wraps replace the modulo
                    auto row_of = [&](int t) {
                        int j = t < st.bound ? st.end - 1 - t : st.end - st.bound + (t - st.bound);
                        j = j < 0 ? j + m : j;
                        j = j < 0 ? j + m : j;
                        return j >= m ? j - m : j;
                    };
                    // Issuing a bulk copy costs the issuing thread a few hundred cycles, so the copies of a
                    // round are spread over the first lane of each warp: part 0 arms the stage's barrier and
                    // fetches s_j, part 1 fetches y_j (the transaction count may complete in any order).
                    auto issue_part = [&](int t, int sg, int part) {
#ifdef TP_DEBUG_NO_TMA
                        return;
#endif
                        const int j = row_of(t);
                        double* dst = ring + (size_t)sg * 2 * rowd;
                        if (part == 0) {
                            tp_mbar_expect_tx(&s_bar[sg], 2 * row_bytes);
                            tp_bulk_g2s(dst, lm_s + (size_t)j * S.xs, row_bytes, &s_bar[sg], pol);
                        } else {
                            tp_bulk_g2s(dst + rowd, lm_y + (size_t)j * S.xs, row_bytes, &s_bar[sg], pol);
                        }
                    };
                    double* scratch = s_ys + 256;     // n doubles, behind the ring and the two tables
                    // Two history rows per reduction round. For rows A (first) and B (second) of a loop
                    //   loop 1:  a = s_A.q, b = s_B.q, c = s_B.y_A;  alpha_A = rho_A a,
                    //            alpha_B = rho_B (b - alpha_A c);    q -= alpha_A y_A + alpha_B y_B
                    //   loop 2:  a = y_A.r, b = y_B.r, c = y_B.s_A;  k_A = alpha_A - rho_A a,
                    //            k_B = alpha_B - rho_B (b + k_A c);  r += k_A s_A + k_B s_B
                    // which is the recursion of lbfgs.hpp:691-710 with s_B.(q - alpha_A y_A) expanded, so
                    // that the three dot products share one reduction (one barrier per two rows).
                    auto two_loop = [&](auto solo_tag, double* q) {
                        constexpr bool SOLO = decltype(solo_tag)::value;
                        constexpr int STRIDE = SOLO ? 32 : TP_CAND_THREADS;
                        const int me = SOLO ? lane : tid;
                        // the four copies of a round (steps t, t + 1; s and y) go to four different threads
                        // step t lives in stage t mod nst, lap parity (t / nst) & 1: tracked incrementally
                        int sg = 0, ph = 0;
                        // refill the stages of steps (t, t + 1) that were just read — stages sg0, sg0 + 1 —
                        // with steps t + nst, t + nst + 1; the four copies go to four different threads
                        auto issue_round = [&](int t, int sg0, int steps) {
                            if (SOLO) {
                                // the whole warp copies the rows of the round, 16 B per lane and instruction; ONE
                                // commit group per round, committed even when the history has run out, so that
                                // "all but the newest TP_SOLO_GROUPS - 1 groups have landed" always covers the
                                // round about to be read
#ifndef TP_DEBUG_NO_TMA
                                const int chunks = rowd >> 1;             // 16-byte chunks per row
                                for (int st_ = 0; st_ < steps; st_++) {
                                    const int tt = t + st_;
                                    if (tt >= total) break;
                                    const int j = row_of(tt);
                                    double* dst = ring + (size_t)(sg0 + st_) * 2 * rowd;
                                    const double* srs = lm_s + (size_t)j * S.xs;
                                    const double* sry = lm_y + (size_t)j * S.xs;
                                    for (int c = lane; c < chunks; c += 32) {
                                        tp_cp_async16(dst + 2 * c, srs + 2 * c);
                                        tp_cp_async16(dst + rowd + 2 * c, sry + 2 * c);
                                    }
                                }
                                tp_cp_async_commit();
#endif
                                return;
                            }
                            const int who = lane == 0 ? warp : -1;
                            if (who >= 0 && who < 2 * steps) {
                                const int tt = t + (who >> 1);
                                if (tt < total) issue_part(tt, sg0 + (who >> 1), who & 1);
                            }
                        };
                        auto load_row = [&](int jrow, double* cs, double* cy) {
#ifdef TP_DEBUG_NO_TMA
                            const double* rs_ = lm_s + (size_t)jrow * S.xs;     // debug: plain loads, no ring
                            const double* ry_ = lm_y + (size_t)jrow * S.xs;
#else
                            if (!SOLO) tp_mbar_wait(&s_bar[sg], (uint32_t)ph);
                            const double* rs_ = ring + (size_t)sg * 2 * rowd;
                            const double* ry_ = rs_ + rowd;
#endif
#pragma unroll
                            for (int e = 0; e < TP_EPT; e++) {
                                const int i = me + e * STRIDE;
                                cs[e] = i < n ? rs_[i] : 0.0;
                                cy[e] = i < n ? ry_[i] : 0.0;
                            }
                            if (++sg == nst) {
                                sg = 0;
                                ph ^= 1;
                            }
                        };
                        auto reduce3 = [&](double* d3) {
                            if (SOLO) {
#pragma unroll
                                for (int k = 0; k < 3; k++) d3[k] = tp_warp_sum(d3[k]);
                                __syncwarp();             // every lane has read both stages
                            } else {
                                tp_block_sum<3>(d3, red, flip);   // one barrier: every thread has read both stages
                            }
                        };
                        if (SOLO) {
                            for (int t = 0; t < nst; t += 2) issue_round(t, t, 2);      // exactly TP_SOLO_GROUPS groups
                        } else {
                            for (int t = 0; t < min(total, nst); t += 2) issue_round(t, t, 2);
                        }
                        for (int t = 0; t < total;) {
                            if (SOLO) {
#ifndef TP_DEBUG_NO_TMA
                                tp_cp_async_wait<TP_SOLO_GROUPS - 1>();
                                __syncwarp();             // every lane's chunks of the round are in shared memory
#endif
                            }
                            if (t == st.bound) {
                                // between the loops: d *= ys / yy (lbfgs.hpp:701)
                                const double sc = ys / yy;
#pragma unroll
                                for (int e = 0; e < TP_EPT; e++) q[e] *= sc;
                            }
                            const bool first = t < st.bound;
                            const bool pair = t + 1 < (first ? st.bound : total);
                            const int jA = row_of(t);
                            const int jB = pair ? row_of(t + 1) : jA;
                            double sA[TP_EPT], yA[TP_EPT], sB[TP_EPT], yB[TP_EPT];
                            const int sg0 = sg;            // nst is even and pairs start on even steps of a loop;
                            load_row(jA, sA, yA);          // a stage pair never straddles the ring's end unless
                            if (pair) {                    // a loop has odd length, which the refill handles per step
                                load_row(jB, sB, yB);
                            } else {
#pragma unroll
                                for (int e = 0; e < TP_EPT; e++) sB[e] = yB[e] = 0.0;
                            }
                            double d3[3] = {0.0, 0.0, 0.0};
#pragma unroll
                            for (int e = 0; e < TP_EPT; e++) {
                                const double uA = first ? sA[e] : yA[e], uB = first ? sB[e] : yB[e];
                                const double vA = first ? yA[e] : sA[e];
                                d3[0] += uA * q[e];
                                d3[1] += uB * q[e];
                                d3[2] += uB * vA;
                            }
                            reduce3(d3);
                            // refill exactly the stages just read (the second one may have wrapped to stage 0)
                            if (pair && sg0 + 1 == nst) {
                                issue_round(t + nst, sg0, 1);
                                issue_round(t + nst + 1, 0, 1);
                            } else {
                                issue_round(t + nst, sg0, pair ? 2 : 1);
                            }
                            if (first) {
                                const double alA = d3[0] * s_ys[jA];
                                const double alB = pair ? (d3[1] - alA * d3[2]) * s_ys[jB] : 0.0;
                                if (me == 0) {
                                    s_alpha[jA] = alA;
                                    if (pair) s_alpha[jB] = alB;
                                }
#pragma unroll
                                for (int e = 0; e < TP_EPT; e++) {
                                    q[e] += (-alA) * yA[e];
                                    if (pair) q[e] += (-alB) * yB[e];
                                }
                            } else {
                                const double kA = s_alpha[jA] - d3[0] * s_ys[jA];
                                const double kB = pair ? s_alpha[jB] - (d3[1] + kA * d3[2]) * s_ys[jB] : 0.0;
#pragma unroll
                                for (int e = 0; e < TP_EPT; e++) {
                                    q[e] += kA * sA[e];
                                    if (pair) q[e] += kB * sB[e];
                                }
                            }
                            if (SOLO) __syncwarp();       // alpha table writes visible to the warp
                            t += pair ? 2 : 1;
                        }
                        if (SOLO) {
#ifndef TP_DEBUG_NO_TMA
                            tp_cp_async_wait<0>();
#endif
                        }
                    };
                    if (tid == 0) atomicAdd(S.node_count + 1, (unsigned long long)total * (unsigned long long)n);
                    // the ring region was last written through the generic proxy and the block's new
                    // history row has to be visible to the bulk-copy engine
                    asm volatile("fence.proxy.async;" ::: "memory");
                    if (solo) {
#pragma unroll
                        for (int e = 0; e < TP_EPT; e++) {
                            const int i = tid + e * TP_CAND_THREADS;
                            if (i < n) scratch[i] = rd[e];
                        }
                        __syncthreads();
                        if (warp == 0) {
                            double q[TP_EPT];
#pragma unroll
                            for (int e = 0; e < TP_EPT; e++) q[e] = lane + 32 * e < n ? scratch[lane + 32 * e] : 0.0;
                            const double sc = ys / yy;
                            switch ((rowd + 31) >> 5) {
                                case 1: tp_two_loop_solo<1>(q, rowd, st.bound, st.end, m, lm_s, lm_y, S.xs, s_ys, s_alpha, red, ring, sc, lane); break;
                                case 2: tp_two_loop_solo<2>(q, rowd, st.bound, st.end, m, lm_s, lm_y, S.xs, s_ys, s_alpha, red, ring, sc, lane); break;
                                case 3: tp_two_loop_solo<3>(q, rowd, st.bound, st.end, m, lm_s, lm_y, S.xs, s_ys, s_alpha, red, ring, sc, lane); break;
                                case 4: tp_two_loop_solo<4>(q, rowd, st.bound, st.end, m, lm_s, lm_y, S.xs, s_ys, s_alpha, red, ring, sc, lane); break;
                                default: tp_two_loop_solo<5>(q, rowd, st.bound, st.end, m, lm_s, lm_y, S.xs, s_ys, s_alpha, red, ring, sc, lane); break;
                            }
#pragma unroll
                            for (int e = 0; e < TP_EPT; e++)
                                if (lane + 32 * e < n) scratch[lane + 32 * e] = q[e];
                        }
                        __syncthreads();
#pragma unroll
                        for (int e = 0; e < TP_EPT; e++) {
                            const int i = tid + e * TP_CAND_THREADS;
                            if (i < n) rd[e] = scratch[i];
                        }
                    } else {
                        two_loop(std::false_type{}, rd);
                    }
                    if (total == 0) {
                        const double sc = ys / yy;
#pragma unroll
                        for (int e = 0; e < TP_EPT; e++) rd[e] *= sc;
                    }
                    __syncthreads();
                }
                TP_PROF(7);
                st.stp = 1.0;
                action = A_BEGIN_LS;
            }
        }
        if (action == A_BEGIN_LS) {
            // lbfgs.hpp:558-573 and line search prologue :288-311
#pragma unroll
            for (int e = 0; e < TP_EPT; e++) {
                rxp[e] = rx[e];
                rgp[e] = rg[e];
            }
            st.ls_count = 0;
            st.brackt = 0;
            st.touched = 0;
            st.mu = 0.0;
            st.nu = lp.max_step;
            if (!(st.stp > 0.0)) {
                ret = TOPAY_LBFGSERR_INVALIDPARAMETERS;
                action = A_FINISH;
            } else {
                double dg[1] = {0.0};
#pragma unroll
                for (int e = 0; e < TP_EPT; e++) dg[0] += rgp[e] * rd[e];
                tp_block_sum<1>(dg, red, flip);
                const double dginit = dg[0];
                if (0.0 < dginit) {
                    ret = TOPAY_LBFGSERR_INCREASEGRADIENT;
                    action = A_FINISH;
                } else {
                    st.finit = st.fx;
                    st.dgtest = lp.f_dec_coeff * dginit;
                    st.dstest = lp.s_curv_coeff * dginit;
#pragma unroll
                    for (int e = 0; e < TP_EPT; e++) rx[e] = rxp[e] + st.stp * rd[e];
                }
            }
        }
        if (action == A_FINISH) {
            // end of one lbfgs_optimize call; the outer logic of optimizeTraj (:362-460)
            st.iters_total += st.k;
            st.last_code = ret;
            st.cost = st.fx;
            bool next_round = false;
            if (cancel) {
                st.status = 0;
                st.phase = 0;
            } else if (st.phase == 1) {
                if (tp_ok_code(ret)) {
                    st.phase = 2;
                    st.lambda[0] = P.opt.alm_init_lambda[0];
                    st.lambda[1] = P.opt.alm_init_lambda[1];
                    st.rho[0] = P.opt.alm_init_rho[0];
                    st.rho[1] = P.opt.alm_init_rho[1];
                    st.alm_round = 0;
                    next_round = true;
                } else {
                    st.status = 0;
                    st.phase = 0;
                }
            } else {
                if (tp_ok_code(ret) || ret == TOPAY_LBFGSERR_MAXIMUMLINESEARCH) {
                    const double en = sqrt(st.final_xy[0] * st.final_xy[0] + st.final_xy[1] * st.final_xy[1]);
                    if (en < P.opt.alm_tolerance) {
                        st.status = 1;
                        st.phase = 0;
                    } else {
                        st.lambda[0] += st.rho[0] * st.final_xy[0];
                        st.lambda[1] += st.rho[1] * st.final_xy[1];
                        st.rho[0] = fmin((1 + P.opt.alm_gamma[0]) * st.rho[0], P.opt.alm_rho_max[0]);
                        st.rho[1] = fmin((1 + P.opt.alm_gamma[1]) * st.rho[1], P.opt.alm_rho_max[1]);
                        next_round = true;
                    }
                } else {
                    st.status = 0;
                    st.phase = 0;
                }
            }
            if (next_round) {
                if (st.alm_round >= P.opt.alm_max_rounds) {
                    st.status = 0;
                    st.phase = 0;
                } else {
                    st.alm_round++;
                    st.ls_init = 1;
                }
            }
            need_eval = st.phase != 0;
        }
        if (action == A_FINISH && st.phase == 0) {
            // ---- the candidate is done: results to the store, then the slot takes the next waiting candidate
#pragma unroll
            for (int e = 0; e < TP_EPT; e++) {
                const int i = tid + e * TP_CAND_THREADS;
                if (i < n) S.res_x[(size_t)gid * S.xs + i] = rx[e];
            }
            for (int i = tid; i < N; i += TP_CAND_THREADS) S.res_T[(size_t)gid * S.max_pieces + i] = Tg[i];
            {
                double* rc = S.res_coeff + (size_t)gid * 6 * S.max_pieces * 9;
                for (int e = tid; e < n6 * 9; e += TP_CAND_THREADS) rc[e] = cg[e];
            }
            __shared__ int s_next;
            if (tid == 0) {
                S.res_st[gid] = st;
                if (S.plan_of && st.status == 1) {   // publish the success (through the host's gate with plan_gate)
                    if (S.plan_gate) S.pending[1 + atomicAdd(S.pending, 1)] = gid;
                    else atomicMin(S.plan_first + S.plan_of[gid], st.evals_total);
                }
                atomicAdd(S.queue + 2, 1);
                if (S.qrow) tp_stream_retire(S, gid);
                const int q = atomicAdd(S.queue, 1);
                s_next = q < S.queue[1] ? (S.qrow ? S.qrow[q % S.max_cand] : q) : -1;
            }
            __syncthreads();
            const int nxt = s_next;
            if (nxt >= 0) {
                gid = nxt;
                st = S.st0[gid];
                N = st.N;
                n = st.n;
                n6 = 6 * N;
                const double* xn = S.x0 + (size_t)gid * S.xs;
                for (int i = tid; i < n; i += TP_CAND_THREADS) x[i] = xn[i];
                if (tid == 0) S.slot_gid[cand] = gid;
                need_eval = true;
            }
            __syncthreads();
        } else {
            // write this thread's elements back
#pragma unroll
            for (int e = 0; e < TP_EPT; e++) {
                const int i = tid + e * TP_CAND_THREADS;
                if (i < n) {
                    x[i] = rx[e];
                    g[i] = rg[e];
                    xp[i] = rxp[e];
                    gp[i] = rgp[e];
                    dv[i] = rd[e];
                }
            }
            __syncthreads();
        }
        TP_PROF(8);
    }

    // ================= generate half of the next evaluation =================
    if ((mode & TP_MODE_GEN) && need_eval) {
        if (!(mode & TP_MODE_ADVANCE)) gid = S.slot_gid[cand];
        double* sT = s_small;
        for (int i = tid; i < N; i += TP_CAND_THREADS) {
            const double t = tp_expC2(x[i]);
            sT[i] = t;
            Tg[i] = t;
        }
        __syncthreads();
        tp_fill_system(N, sT, S.head_pva + (size_t)gid * 27, S.tail_pva + (size_t)gid * 27, x, P, lu, cf);
        TP_PROF(9);
        if (warp == 0) tp_lu_factor(n6, lu, lane);
        __syncthreads();
        TP_PROF(10);
        tp_band_transpose(n6, lu);
        if (tid < 9) {
            tp_sweep<true, false>(n6, lu, cf, tid);    // L y = b   (solve, first loop)
            tp_sweep<false, true>(n6, lu, cf, tid);    // U x = y   (second loop)
        }
        __syncthreads();
        tp_band_transpose(n6, lu);
        TP_PROF(11);
        for (int e = tid; e < n6 * TP_BAND; e += TP_CAND_THREADS) lug[e] = lu[e];
        for (int e = tid; e < n6 * 9; e += TP_CAND_THREADS) cg[e] = cf[e];
        TP_PROF(12);
    }
    if (tid == 0) {
        *gs = st;
        if (st.phase != 0 && (mode & TP_MODE_GEN)) {
            if (tick_out >= 0) {
                const int q = atomicAdd(S.count + tick_out, 1);
                S.list[(size_t)tick_out * S.n_slots + q] = cand;
            }
            atomicAdd(S.node_count, (unsigned long long)(N * (S.K + 1)));
        }
    }
}
#undef LU_AT
#undef LU_DINV
