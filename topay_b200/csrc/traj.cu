// Result post-processing and the worker's success gate on the device (SURVEY.md §8 row a16 and
// "next" row N1):
//
//   car_seq     MomaTraj constructor          src/planner/include/planner/moma_traj_opt.h:38-68
//   sample      MomaTraj::getState/getDState  moma_traj_opt.h:121-160
//   feasible    MomaTrajOpt::checkFeasible / printConstraintsSituations   moma_traj_opt.h:948-1210
//   select      shortest successful duration  src/planner/src/planner.cpp:999-1010
//
// One thread block per trajectory. The pose table is a running sum in the reference, so its
// increments are evaluated in parallel and added by one thread in the reference's order; the
// feasibility scan visits the reference's own sample clock (t += 0.01 accumulated in fp64, a
// table shared by all trajectories), keeps "the first sample with the largest magnitude" per
// quantity through an (|v|, index) reduction, and reads the field through the same lookups as
// the solver (field_query.cuh) and the same forward kinematics (robot.cuh).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "common_host.h"
#include "rog_query.cuh"
#include "robot.cuh"
#include "traj.cuh"
#include "traj_host.h"

#define TP_TRAJ_THREADS 128

namespace {

__device__ __forceinline__ int traj_of(const TpTrajView& V, int i) { return V.idx ? V.idx[i] : i; }

__device__ __forceinline__ TpPoly poly_of(const TpTrajView& V, int i) {
    i = traj_of(V, i);
    TpPoly p;
    p.N = V.piece_num[i];
    p.T = V.T + (size_t)i * V.max_pieces;
    p.c = V.coeff + (size_t)i * 6 * V.max_pieces * 9;
    return p;
}

// the solver keeps piece counts inside its per-candidate state and the start pose split over two arrays
__global__ void k_traj_meta(TpTrajView V, const double* __restrict__ ttab, int ttab_len, TpTrajMeta* meta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V.n) return;
    const TpPoly p = poly_of(V, i);
    const double total = tp_poly_total(p);
    // samples: t_k < total on the accumulated clock
    int lo = 0, hi = ttab_len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ttab[mid] < total) lo = mid + 1;
        else hi = mid;
    }
    const double r = TP_SEQ_RES / TP_APPROX_RES;
    TpTrajMeta m;
    m.total = total;
    m.n_samples = lo < ttab_len ? lo : -1;   // -1: longer than the clock table
    m.seq_num = (int)floor(total / r);
    m.n_seq = 1 + m.seq_num / TP_APPROX_RES;
    m.seq_off = 0;
    meta[i] = m;
}

// moma_traj_opt.h:38-68
__global__ void __launch_bounds__(TP_TRAJ_THREADS)
k_car_seq(TpTrajView V, const TpTrajMeta* __restrict__ meta, double* __restrict__ car_seq) {
    __shared__ double s_dx[TP_TRAJ_THREADS], s_dy[TP_TRAJ_THREADS], s_th[TP_TRAJ_THREADS];
    const int i = blockIdx.x;
    const TpPoly p = poly_of(V, i);
    const TpTrajMeta m = meta[i];
    double* out = car_seq + (size_t)m.seq_off * 4;
    const double r = TP_SEQ_RES / TP_APPROX_RES, half = r / 2.0, r16 = r / 6.0;
    const double* start = V.start + 3 * traj_of(V, i);
    double cx = start[0], cy = start[1];
    if (threadIdx.x == 0) {
        out[0] = cx;
        out[1] = cy;
        out[2] = start[2];
        out[3] = 0.0;
    }
    for (int base = 0; base < m.seq_num; base += TP_TRAJ_THREADS) {
        const int k = base + threadIdx.x;
        if (k < m.seq_num) {
            double a[2], b[2], c[2];
            // p1/v1 are the previous step's p3/v3, i.e. evaluated at (k-1)*r + r, not at k*r
            tp_theta_speed(p, k == 0 ? 0.0 : (k - 1) * r + r, a);
            tp_theta_speed(p, k * r + half, b);
            tp_theta_speed(p, k * r + r, c);
            tp_simpson_xy(r16, a, b, c, s_dx[threadIdx.x], s_dy[threadIdx.x]);
            s_th[threadIdx.x] = c[0];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int cnt = min(TP_TRAJ_THREADS, m.seq_num - base);
            for (int j = 0; j < cnt; j++) {
                const int k2 = base + j;
                cx += s_dx[j];
                cy += s_dy[j];
                if (k2 % TP_APPROX_RES == TP_APPROX_RES - 1) {
                    double* e = out + (size_t)(k2 / TP_APPROX_RES + 1) * 4;
                    e[0] = cx;
                    e[1] = cy;
                    e[2] = s_th[j];
                    e[3] = (k2 + 1) * r;
                }
            }
        }
        __syncthreads();
    }
}

__global__ void k_traj_sample(TpTrajView V, const TpTrajMeta* __restrict__ meta, const double* __restrict__ car_seq,
                              const double* __restrict__ t, int m, double* state, double* dstate) {
    const int i = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const TpPoly p = poly_of(V, i);
    const TpTrajMeta mt = meta[i];
    const double tt = t[(size_t)i * m + j];
    if (state) {
        double s[10];
        tp_traj_state(p, car_seq + (size_t)mt.seq_off * 4, mt.n_seq, mt.total, tt, s);
        for (int k = 0; k < 10; k++) state[((size_t)i * m + j) * 10 + k] = s[k];
    }
    if (dstate) {
        double s[10];
        tp_traj_dstate(p, mt.total, tt, s);
        for (int k = 0; k < 10; k++) dstate[((size_t)i * m + j) * 10 + k] = s[k];
    }
}

struct MaxAbs {
    double a, v;
    int idx;
};
__device__ __forceinline__ void maxabs_take(MaxAbs& m, double v, int idx) {
    if (fabs(v) > m.a) {   // == fabs(v) > fabs(max): strictly greater, so the first such sample stays
        m.a = fabs(v);
        m.v = v;
        m.idx = idx;
    }
}
__device__ __forceinline__ void maxabs_merge(MaxAbs& m, double oa, double ov, int oi) {
    if (oa > m.a || (oa == m.a && oi < m.idx)) {
        m.a = oa;
        m.v = ov;
        m.idx = oi;
    }
}

// moma_traj_opt.h:948-1045 / :1047-1210
__global__ void __launch_bounds__(TP_TRAJ_THREADS)
k_feasible(TpTrajView V, const __grid_constant__ TpParams P, const __grid_constant__ TpGrid g0,
           const TpGrid* __restrict__ grids, const int32_t* __restrict__ field_of, const TpTrajMeta* __restrict__ meta,
           const double* __restrict__ car_seq, const double* __restrict__ ttab, TpFeasOut* out) {
    // scenario sweeps: trajectory i is checked against the field of its own scenario, grids[field_of[i]]
    __shared__ TpGrid s_grid;
    if (grids) {
        const double* src = reinterpret_cast<const double*>(grids + field_of[traj_of(V, blockIdx.x)]);
        double* dst = reinterpret_cast<double*>(&s_grid);
        for (int w = threadIdx.x; w < (int)(sizeof(TpGrid) / sizeof(double)); w += TP_TRAJ_THREADS) dst[w] = src[w];
        __syncthreads();
    }
    const TpGrid& g = grids ? s_grid : g0;
    __shared__ double s_a[TP_TRAJ_THREADS / 32][TP_NMAXABS], s_v[TP_TRAJ_THREADS / 32][TP_NMAXABS];
    __shared__ int s_i[TP_TRAJ_THREADS / 32][TP_NMAXABS];
    __shared__ double s_m[TP_TRAJ_THREADS / 32][TP_NMIN];
    const int i = blockIdx.x;
    const TpPoly p = poly_of(V, i);
    const TpTrajMeta mt = meta[i];
    const double* seq = car_seq + (size_t)mt.seq_off * 4;
    MaxAbs mx[TP_NMAXABS];
    double mn[TP_NMIN];
#pragma unroll
    for (int q = 0; q < TP_NMAXABS; q++) mx[q] = MaxAbs{0.0, 0.0, INT_MAX};
#pragma unroll
    for (int q = 0; q < TP_NMIN; q++) mn[q] = 1.0e+10;
    for (int k = threadIdx.x; k < mt.n_samples; k += TP_TRAJ_THREADS) {
        const double t = ttab[k];
        double state[10], vel[9], acc[9];
        tp_traj_state(p, seq, mt.n_seq, mt.total, t, state);
        tp_poly_vel(p, t, 0, 9, vel);
        tp_poly_acc(p, t, 0, 9, acc);
        maxabs_take(mx[0], vel[1], k);
        maxabs_take(mx[1], acc[1], k);
        maxabs_take(mx[2], vel[0], k);
        maxabs_take(mx[3], acc[0], k);
#pragma unroll
        for (int q = 0; q < TOPAY_DOF; q++) {
            maxabs_take(mx[4 + q], state[3 + q], k);
            maxabs_take(mx[11 + q], vel[2 + q], k);
            maxabs_take(mx[18 + q], acc[2 + q], k);
        }
        const double d2 = tp_field_distance2d(g, state);
        if (d2 < mn[0]) mn[0] = d2;
        TpFK fk;
        TpSphereStoreLocal pts;
        tp_fk(P, state, fk, pts);
#pragma unroll
        for (int a = 0; a < TOPAY_NSPHERE; a++) {
            if (a < P.n_sphere) {
                const double pa[3] = {pts.at(a, 0), pts.at(a, 1), pts.at(a, 2)};
                const double d3 = tp_field_distance3d(g, pa);
                if (d3 < mn[1 + a]) mn[1 + a] = d3;
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < TP_NMAXABS; q++) {
        MaxAbs m = mx[q];
        for (int off = 16; off > 0; off >>= 1) {
            const double oa = __shfl_xor_sync(0xffffffffu, m.a, off);
            const double ov = __shfl_xor_sync(0xffffffffu, m.v, off);
            const int oi = __shfl_xor_sync(0xffffffffu, m.idx, off);
            maxabs_merge(m, oa, ov, oi);
        }
        if (lane == 0) {
            s_a[warp][q] = m.a;
            s_v[warp][q] = m.v;
            s_i[warp][q] = m.idx;
        }
    }
#pragma unroll
    for (int q = 0; q < TP_NMIN; q++) {
        double m = mn[q];
        for (int off = 16; off > 0; off >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, off));
        if (lane == 0) s_m[warp][q] = m;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    TpFeasOut F;
    for (int q = 0; q < TP_NMAXABS; q++) {
        MaxAbs m{s_a[0][q], s_v[0][q], s_i[0][q]};
        for (int w = 1; w < TP_TRAJ_THREADS / 32; w++) maxabs_merge(m, s_a[w][q], s_v[w][q], s_i[w][q]);
        F.maxabs[q] = m.v;
    }
    for (int q = 0; q < TP_NMIN; q++) {
        double m = s_m[0][q];
        for (int w = 1; w < TP_TRAJ_THREADS / 32; w++) m = fmin(m, s_m[w][q]);
        F.mins[q] = m;
    }
    const topay_robot_params& rp = P.robot;
    bool ok = true;
    if (fabs(F.maxabs[0]) > 1.01 * rp.max_v) ok = false;
    if (fabs(F.maxabs[1]) > 1.01 * rp.max_a) ok = false;
    if (fabs(F.maxabs[2]) > 1.01 * rp.max_w) ok = false;
    if (fabs(F.maxabs[3]) > 1.01 * rp.max_dw) ok = false;
    for (int q = 0; q < TOPAY_DOF; q++) {
        if (fabs(F.maxabs[4 + q]) > 1.01 * rp.joint_pos_limit_max[q]) ok = false;
        if (fabs(F.maxabs[11 + q]) > 1.01 * rp.joint_vel_limit[q]) ok = false;
        if (fabs(F.maxabs[18 + q]) > 1.01 * rp.joint_acc_limit[q]) ok = false;
    }
    if (F.mins[0] < 0.99 * rp.chassis_colli_radius) ok = false;
    F.feasible_print = ok ? 1 : 0;
    for (int a = 0; a < P.n_sphere; a++)
        if (F.mins[1 + a] < 0.99 * P.sphere_r[a]) ok = false;
    F.feasible = ok ? 1 : 0;
    F.n_samples = mt.n_samples;
    F.pad = 0;
    out[i] = F;
}

// The reference's sample clock: t = 0; t += 0.01 (moma_traj_opt.h:972). One table for every trajectory.
const std::vector<double>& clock_table() {
    static std::vector<double> tab;
    static std::once_flag once;
    std::call_once(once, [] {
        tab.resize(1 << 17);   // 1310 s
        double t = 0.0;
        for (size_t k = 0; k < tab.size(); k++) {
            tab[k] = t;
            t += 0.01;
        }
    });
    return tab;
}

}  // namespace

// ------------------------------------------------------------------ TpTrajChecker

TpTrajChecker::~TpTrajChecker() {
    cudaSetDevice(device);
    for (void* p : {(void*)ttab, (void*)meta, (void*)car_seq, (void*)feas})
        if (p) cudaFree(p);
}

int TpTrajChecker::init(int dev, cudaStream_t q) {
    device = dev;
    stream = q;
    const std::vector<double>& tab = clock_table();
    ttab_len = (int)tab.size();
    TP_CUDA_OK(cudaMalloc(&ttab, tab.size() * 8), {});
    TP_CUDA_OK(cudaMemcpyAsync(ttab, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, q), {});
    return TOPAY_OK;
}

int TpTrajChecker::prepare(const TpTrajView& V) {
    if (V.n > cap_n) {
        if (meta) cudaFree(meta);
        if (feas) cudaFree(feas);
        meta = nullptr;
        feas = nullptr;
        TP_CUDA_OK(cudaMalloc(&meta, (size_t)V.n * sizeof(TpTrajMeta)), {});
        TP_CUDA_OK(cudaMalloc(&feas, (size_t)V.n * sizeof(TpFeasOut)), {});
        cap_n = V.n;
    }
    k_traj_meta<<<(V.n + 63) / 64, 64, 0, stream>>>(V, ttab, ttab_len, meta);
    h_meta.resize(V.n);
    TP_CUDA_OK(cudaMemcpyAsync(h_meta.data(), meta, (size_t)V.n * sizeof(TpTrajMeta), cudaMemcpyDeviceToHost, stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(stream), {});
    size_t off = 0;
    for (int i = 0; i < V.n; i++) {
        if (h_meta[i].n_samples < 0 || !(h_meta[i].total >= 0.0)) {
            tp_set_error("trajectory duration outside the supported range (0 .. 1310 s)");
            return TOPAY_ERR_TOO_LARGE;
        }
        h_meta[i].seq_off = (int32_t)off;
        off += (size_t)h_meta[i].n_seq;
    }
    if (off > cap_seq) {
        if (car_seq) cudaFree(car_seq);
        car_seq = nullptr;
        TP_CUDA_OK(cudaMalloc(&car_seq, off * 4 * 8), {});
        cap_seq = off;
    }
    TP_CUDA_OK(cudaMemcpyAsync(meta, h_meta.data(), (size_t)V.n * sizeof(TpTrajMeta), cudaMemcpyHostToDevice, stream), {});
    k_car_seq<<<V.n, TP_TRAJ_THREADS, 0, stream>>>(V, meta, car_seq);
    return TOPAY_OK;
}

int TpTrajChecker::check(const TpTrajView& V, const TpParams& P, const TpGrid& g, topay_feasibility* out,
                         const TpGrid* grids, const int32_t* field_of) {
    const int rc = run(V, P, g, grids, field_of);
    return rc != TOPAY_OK ? rc : fetch(V.n, out);
}

int TpTrajChecker::run(const TpTrajView& V, const TpParams& P, const TpGrid& g, const TpGrid* grids,
                       const int32_t* field_of) {
    int rc = prepare(V);
    if (rc != TOPAY_OK) return rc;
    k_feasible<<<V.n, TP_TRAJ_THREADS, 0, stream>>>(V, P, g, grids, field_of, meta, car_seq, ttab, feas);
    return TOPAY_OK;
}

int TpTrajChecker::fetch(int n, topay_feasibility* out) {
    std::vector<TpFeasOut> h(n);
    TP_CUDA_OK(cudaMemcpyAsync(h.data(), feas, (size_t)n * sizeof(TpFeasOut), cudaMemcpyDeviceToHost, stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(stream), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    for (int i = 0; i < n; i++) {
        const TpFeasOut& F = h[i];
        out->feasible[i] = F.feasible;
        if (out->feasible_print) out->feasible_print[i] = F.feasible_print;
        if (out->n_samples) out->n_samples[i] = F.n_samples;
        if (out->max_vel) out->max_vel[i] = F.maxabs[0];
        if (out->max_acc) out->max_acc[i] = F.maxabs[1];
        if (out->max_domega) out->max_domega[i] = F.maxabs[2];
        if (out->max_d2omega) out->max_d2omega[i] = F.maxabs[3];
        for (int q = 0; q < TOPAY_DOF; q++) {
            if (out->max_q) out->max_q[i * TOPAY_DOF + q] = F.maxabs[4 + q];
            if (out->max_dq) out->max_dq[i * TOPAY_DOF + q] = F.maxabs[11 + q];
            if (out->max_d2q) out->max_d2q[i * TOPAY_DOF + q] = F.maxabs[18 + q];
        }
        if (out->min_dist) out->min_dist[i] = F.mins[0];
        if (out->min_dist_mani)
            for (int a = 0; a < TOPAY_NSPHERE; a++) out->min_dist_mani[i * TOPAY_NSPHERE + a] = F.mins[1 + a];
    }
    return TOPAY_OK;
}

namespace {

// Checks a host batch and stages it through `io`; *V views the device copy.
int stage_batch(const topay_traj_batch* b, TpStaging& io, TpTrajView* V) {
    if (!b || b->n_traj < 1 || b->max_pieces < 1 || !b->piece_num || !b->T || !b->coeff || !b->start_se2) {
        tp_set_error("trajectory batch: null pointer or empty batch");
        return TOPAY_ERR_INVALID_ARG;
    }
    const size_t n = b->n_traj, NP = b->max_pieces;
    for (size_t i = 0; i < n; i++)
        if (b->piece_num[i] < 1 || b->piece_num[i] > (int)NP) {
            tp_set_error("trajectory batch: piece_num outside 1..max_pieces");
            return TOPAY_ERR_INVALID_ARG;
        }
    V->n = (int)n;
    V->max_pieces = (int)NP;
    V->T = io.in(b->T, n * NP);
    V->coeff = io.in(b->coeff, n * 6 * NP * 9);
    V->start = io.in(b->start_se2, n * 3);
    V->piece_num = io.in(b->piece_num, n);
    return io.ok() ? TOPAY_OK : io.finish();
}

// The checker of both entry points on stream q, against grid g (a dense field or the ROG ring).
int check_feasible_on(int dev, cudaStream_t q, const TpGrid& g, const topay_robot_params* robot,
                      const topay_traj_batch* trajs, topay_feasibility* out) {
    int rc;
    {
        TpStaging io(q);
        TpTrajView V{};
        TpTrajChecker ck;
        TpParams P;
        memset(&P, 0, sizeof(P));
        P.robot = *robot;
        topay_opt_params_default(&P.opt);
        tp_derive_params(P);
        rc = stage_batch(trajs, io, &V);
        if (rc == TOPAY_OK) rc = ck.init(dev, q);
        if (rc == TOPAY_OK) rc = ck.check(V, P, g, out);
        cudaStreamSynchronize(q);
    }
    return rc;
}

}  // namespace

extern "C" int topay_traj_check_feasible(topay_field* f, const topay_robot_params* robot, const topay_traj_batch* trajs,
                                         topay_feasibility* out) {
    if (!f || !robot || !out || !out->feasible) return TOPAY_ERR_INVALID_ARG;
    int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    const int dev = tp_field_device(f);
    cudaSetDevice(dev);
    cudaStream_t q;
    TP_CUDA_OK(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking), {});
    TpGrid g;
    tp_field_grid(f, &g);
    rc = check_feasible_on(dev, q, g, robot, trajs, out);
    cudaStreamDestroy(q);
    return rc;
}

// On the ring's stream, so that the check reads the ring after every update queued on it.
extern "C" int topay_traj_check_feasible_rog(topay_rogfield* f, const topay_robot_params* robot,
                                             const topay_traj_batch* trajs, topay_feasibility* out) {
    if (!f || !robot || !out || !out->feasible) return TOPAY_ERR_INVALID_ARG;
    if (!tp_rogfield_ready(f)) {
        tp_set_error("ring not built: call topay_rogfield_update_esdf first");
        return TOPAY_ERR_NOT_READY;
    }
    const int dev = tp_rogfield_device(f);
    cudaSetDevice(dev);
    TpGrid g;
    tp_rogfield_grid(f, &g);
    return check_feasible_on(dev, tp_rogfield_stream(f), g, robot, trajs, out);
}

extern "C" int topay_traj_car_seq(int device, const topay_traj_batch* trajs, int cap, double* car_seq, int32_t* len) {
    if (!car_seq || !len || cap < 1) return TOPAY_ERR_INVALID_ARG;
    int rc = tp_require_device(device);
    if (rc != TOPAY_OK) return rc;
    cudaSetDevice(device);
    cudaStream_t q;
    TP_CUDA_OK(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking), {});
    {
        TpStaging io(q);
        TpTrajView V{};
        TpTrajChecker ck;
        rc = stage_batch(trajs, io, &V);
        if (rc == TOPAY_OK) rc = ck.init(device, q);
        if (rc == TOPAY_OK) rc = ck.prepare(V);
        if (rc == TOPAY_OK) {
            for (int i = 0; i < V.n && rc == TOPAY_OK; i++) {
                len[i] = ck.h_meta[i].n_seq;
                if (len[i] > cap) {
                    tp_set_error("car_seq longer than cap");
                    rc = TOPAY_ERR_TOO_LARGE;
                    break;
                }
                cudaMemcpyAsync(car_seq + (size_t)i * cap * 4, ck.car_seq + (size_t)ck.h_meta[i].seq_off * 4,
                                (size_t)len[i] * 32, cudaMemcpyDeviceToHost, q);
            }
        }
        cudaError_t e = cudaStreamSynchronize(q);
        if (rc == TOPAY_OK && e != cudaSuccess) {
            tp_set_error(std::string("car_seq: ") + cudaGetErrorString(e));
            rc = TOPAY_ERR_CUDA;
        }
    }
    cudaStreamDestroy(q);
    return rc;
}

extern "C" int topay_traj_sample(int device, const topay_traj_batch* trajs, const double* t, int m, double* state,
                                 double* dstate) {
    if (!t || m < 1 || (!state && !dstate)) return TOPAY_ERR_INVALID_ARG;
    int rc = tp_require_device(device);
    if (rc != TOPAY_OK) return rc;
    cudaSetDevice(device);
    cudaStream_t q;
    TP_CUDA_OK(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking), {});
    {
        TpStaging io(q);
        TpTrajView V{};
        TpTrajChecker ck;
        rc = stage_batch(trajs, io, &V);
        if (rc == TOPAY_OK) rc = ck.init(device, q);
        if (rc == TOPAY_OK) rc = ck.prepare(V);
        if (rc == TOPAY_OK) {
            const size_t nm = (size_t)V.n * m;
            const double* dt = io.in(t, nm);
            double* ds = io.out(state, nm * 10);
            double* dd = io.out(dstate, nm * 10);
            if (io.ok())
                k_traj_sample<<<dim3((m + 127) / 128, V.n), 128, 0, q>>>(V, ck.meta, ck.car_seq, dt, m, ds, dd);
            rc = io.finish();
        }
    }
    cudaStreamDestroy(q);
    return rc;
}

// planner.cpp:999-1010
extern "C" int topay_select_shortest(const int32_t* success, const double* duration, int n) {
    int best = -1;
    if (!success || !duration) return -1;
    for (int i = 0; i < n; i++) {
        if (!success[i]) continue;
        if (best == -1) best = i;
        if (duration[i] < duration[best]) best = i;
    }
    return best;
}
