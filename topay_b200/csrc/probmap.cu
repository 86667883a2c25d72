// topay_probmap: rog_map::ProbMap on the device — the probabilistic occupancy layer that turns point clouds into
// the UNKNOWN / OCCUPIED / KNOWN_FREE transitions the ESDF counter map consumes (SURVEY §8 row N3).
//
//   initProbMap               src/rog_map/src/rog_map/prob_map.cpp:25-88   (+ InfMap's ceil / ground adjustment,
//                                                                            inf_map.cpp:81-89)
//   updateProbMap             prob_map.cpp:302-373      host control flow below, kernels for the per-point work
//   raycastProcess            prob_map.cpp:666-778      k_prob_points (filters on the host, clipping per point) +
//                                                       k_prob_rays (one thread per ray, RayCaster::step's walk)
//   insertUpdateCandidate     prob_map.cpp:780-789      one atomicAdd on a packed (hit << 16 | operations) word;
//                                                       the thread that takes a cell from 0 appends it to the cache
//   probabilisticMapFromCache prob_map.cpp:543-569      k_prob_apply: hit / miss log-odds update in float,
//   hitPointUpdate / miss     prob_map.cpp:571-664      type transition -> 16-bit CAS on the ESDF counters
//   mapSliding + resetCell    sliding_map.cpp:113-166, prob_map.cpp:512-541   k_prob_clear
//
// Every per-cell operation of the reference commutes (counts, one log-odds update per cell and batch, +-1 on the
// counters), so the parallel order is immaterial and the buffers are bit-identical to the reference's. All
// floating-point chains that feed a floor() or a comparison use round-to-nearest intrinsics: the reference is built
// without FMA contraction. The inflation map and the frontier counters get the same notifications in the reference;
// they do not feed the ESDF and are not built.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common_host.h"
#include "rog_query.cuh"

#define PM(a, b) __dmul_rn((a), (b))
#define PA(a, b) __dadd_rn((a), (b))
#define PS(a, b) __dadd_rn((a), -(b))
#define PD(a, b) __ddiv_rn((a), (b))
#define PQ(a) __dsqrt_rn(a)

struct TpProbView {
    TpRog g;                 // res, res_inv, half, size of the probability ring (pointers unused)
    int origin_i[3];
    float* occ;              // occupancy_buffer_
    unsigned int* cnt;       // hit_cnt << 16 | operation_cnt
    int32_t* cache;          // update_cache_id_g as ring hashes
    int32_t* cache_n;
    float l_hit, l_miss, l_min, l_max, l_occ, l_free;
};

struct TpProbRay {
    double odom[3], box_min[3], box_max[3];
    double ceil_h, ground_h, range_min, range_max, sqr_range_max;
    int raycasting_en;
};

namespace {

__host__ __device__ __forceinline__ bool pm_inside(const TpProbView& v, int gx, int gy, int gz) {
    const int g[3] = {gx, gy, gz};
    for (int i = 0; i < 3; i++) {
        const int d = g[i] - v.origin_i[i];
        if ((d < 0 ? -d : d) - v.g.half[i] > 0) return false;
    }
    return true;
}
// hashIdToPos (sliding_map.cpp:234-268) under the view's origin
__host__ __device__ __forceinline__ void pm_hash_to_pos(const TpProbView& v, size_t h, double p[3]) {
    int l[3];
    l[0] = (int)(h / ((size_t)v.g.size[1] * v.g.size[2]));
    l[1] = (int)((h - (size_t)l[0] * v.g.size[1] * v.g.size[2]) / v.g.size[2]);
    l[2] = (int)(h - (size_t)l[0] * v.g.size[1] * v.g.size[2] - (size_t)l[1] * v.g.size[2]);
    for (int i = 0; i < 3; i++) {
        l[i] -= v.g.half[i];
        const int min_g = -v.g.half[i] + v.origin_i[i];
        int min_l = min_g % v.g.size[i];
        min_l -= min_l > v.g.half[i] ? v.g.size[i] : 0;
        min_l += min_l < -v.g.half[i] ? v.g.size[i] : 0;
        int d = l[i] - min_l;
        d = d < 0 ? v.g.size[i] + d : d;
        p[i] = ((double)(d + min_g) + 0.5) * v.g.res;      // exact: integer + 0.5, one multiply
    }
}
__device__ __forceinline__ int pm_type(const TpProbView& v, float x) {
    return (double)x >= (double)v.l_occ ? TOPAY_ROG_OCCUPIED : ((double)x < (double)v.l_free ? TOPAY_ROG_KNOWN_FREE : TOPAY_ROG_UNKNOWN);
}
// CounterMap::updateGridCounter (counter_map.cpp:94-151) on the ESDF ring
__device__ __forceinline__ void pm_notify(const TpRog& e, int16_t* occ_cnt, int16_t* unk_cnt, const double pos[3], int from,
                                          int to) {
    const size_t m = tp_rog_hash3(e, tp_rog_cell(e, pos[0]), tp_rog_cell(e, pos[1]), tp_rog_cell(e, pos[2]));
    const int d_occ = (to == TOPAY_ROG_OCCUPIED) - (from == TOPAY_ROG_OCCUPIED);
    const int d_unk = (to == TOPAY_ROG_UNKNOWN) - (from == TOPAY_ROG_UNKNOWN);
    if (d_occ) tp_atomic_add16(occ_cnt, m, d_occ);
    if (d_unk) tp_atomic_add16(unk_cnt, m, d_unk);
}
// insertUpdateCandidate (prob_map.cpp:780-789)
__device__ __forceinline__ void pm_insert(const TpProbView& v, int gx, int gy, int gz, bool hit) {
    const size_t h = tp_rog_hash3(v.g, gx, gy, gz);
    const unsigned int old = atomicAdd(v.cnt + h, hit ? 0x10001u : 1u);
    if ((old & 0xffffu) == 0u) v.cache[atomicAdd(v.cache_n, 1)] = (int32_t)h;
}

// prob_map.cpp:688-757: one kept point -> the end of its ray (+ its hit)
__global__ void k_prob_points(TpProbView v, TpProbRay r, const float4* __restrict__ pts, int64_t n, double* __restrict__ rays) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 c = pts[i];
    double p[3] = {(double)c.x, (double)c.y, (double)c.z};
    if (!r.raycasting_en) {
        const int g[3] = {tp_rog_cell(v.g, p[0]), tp_rog_cell(v.g, p[1]), tp_rog_cell(v.g, p[2])};
        if (pm_inside(v, g[0], g[1], g[2])) pm_insert(v, g[0], g[1], g[2], true);
        return;
    }
    bool update_hit = true;
    const double* o = r.odom;
    if (p[2] > r.ceil_h || p[2] < r.ground_h) {
        // the intersection with the virtual ceiling / ground (:711-723)
        update_hit = false;
        const double lim = p[2] > r.ceil_h ? r.ceil_h : r.ground_h;
        const double dz = PS(p[2], o[2]), pc = PS(lim, o[2]);
        const double d[3] = {PS(p[0], o[0]), PS(p[1], o[1]), PS(p[2], o[2])};
        const double nn = PQ(PA(PA(PM(d[0], d[0]), PM(d[1], d[1])), PM(d[2], d[2])));
        for (int k = 0; k < 3; k++) p[k] = PA(o[k], PD(PM(PD(d[k], nn), pc), dz));
    }
    {
        const double d[3] = {PS(p[0], o[0]), PS(p[1], o[1]), PS(p[2], o[2])};
        const double sqr = PA(PA(PM(d[0], d[0]), PM(d[1], d[1])), PM(d[2], d[2]));
        if (sqr > r.sqr_range_max) {
            const double k = PD(r.range_max, PQ(sqr));
            for (int a = 0; a < 3; a++) p[a] = PA(PM(k, d[a]), o[a]);
            update_hit = false;
        }
    }
    {
        double lo = PS(p[0], r.box_min[0]), hi = PS(p[0], r.box_max[0]);
        for (int a = 1; a < 3; a++) {
            lo = fmin(lo, PS(p[a], r.box_min[a]));
            hi = fmax(hi, PS(p[a], r.box_max[a]));
        }
        if (lo < 0 || hi > 0) {
            // lineBoxIntersectPoint (common_lib.hpp:148-170)
            double diff[3], min_t = 1000000;
            for (int a = 0; a < 3; a++) diff[a] = PS(p[a], o[a]);
            for (int a = 0; a < 3; a++)
                if (fabs(diff[a]) > 0) {
                    const double t1 = PD(PS(r.box_max[a], o[a]), diff[a]);
                    if (t1 > 0 && t1 < min_t) min_t = t1;
                    const double t2 = PD(PS(r.box_min[a], o[a]), diff[a]);
                    if (t2 > 0 && t2 < min_t) min_t = t2;
                }
            for (int a = 0; a < 3; a++) p[a] = PA(o[a], PM(PS(min_t, 1e-3), diff[a]));
            update_hit = false;
        }
    }
    rays[3 * i] = p[0];
    rays[3 * i + 1] = p[1];
    rays[3 * i + 2] = p[2];
    if (update_hit) pm_insert(v, tp_rog_cell(v.g, p[0]), tp_rog_cell(v.g, p[1]), tp_rog_cell(v.g, p[2]), true);
}

// prob_map.cpp:762-776 with RayCaster::setInput / step (raycaster.cpp:66-192): one thread walks one ray from
// range_min along it to its end cell (exclusive) or to the edge of the local map
__global__ void k_prob_rays(TpProbView v, TpProbRay r, const double* __restrict__ rays, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {rays[3 * i], rays[3 * i + 1], rays[3 * i + 2]};
    const double res = v.g.res;
    const double DMAX = 1.7976931348623157e308;
    double s[3];
    {
        const double d[3] = {PS(p[0], r.odom[0]), PS(p[1], r.odom[1]), PS(p[2], r.odom[2])};
        const double nn = PQ(PA(PA(PM(d[0], d[0]), PM(d[1], d[1])), PM(d[2], d[2])));
        for (int a = 0; a < 3; a++) s[a] = PA(PM(PD(d[a], nn), r.range_min), r.odom[a]);
    }
    int ei[3], cur[3], dir[3];
    double t_step[3], t_bound[3], dd[3];
    for (int a = 0; a < 3; a++) {
        const int si = (int)floor(PD(s[a], res));
        ei[a] = (int)floor(PD(p[a], res));
        cur[a] = si;
        const int dlt = ei[a] - si;
        dir[a] = (0 < dlt) - (dlt < 0);
        dd[a] = fabs(PS(p[a], s[a]));
    }
    if (dir[0] == 0 && dir[1] == 0 && dir[2] == 0) return;
    const double tmax = PQ(PA(PA(PM(dd[0], dd[0]), PM(dd[1], dd[1])), PM(dd[2], dd[2])));
    for (int a = 0; a < 3; a++) dd[a] = PD(dd[a], tmax);
    for (int a = 0; a < 3; a++) {
        t_step[a] = dir[a] == 0 ? DMAX : fabs(PD(res, dd[a]));
        const double centre = PM(PA((double)cur[a], 0.5), res);
        const double nb = PA(centre, PM(PM((double)dir[a], res), 0.5));
        t_bound[a] = dir[a] == 0 ? DMAX : PD(fabs(PS(nb, s[a])), dd[a]);
    }
    while (true) {
        double pt[3];
        for (int a = 0; a < 3; a++) pt[a] = PM(PA((double)cur[a], 0.5), res);
        if (cur[0] == ei[0] && cur[1] == ei[1] && cur[2] == ei[2]) break;
        if (t_bound[0] < t_bound[1]) {
            if (t_bound[0] < t_bound[2]) { cur[0] += dir[0]; t_bound[0] = PA(t_bound[0], t_step[0]); }
            else { cur[2] += dir[2]; t_bound[2] = PA(t_bound[2], t_step[2]); }
        } else {
            if (t_bound[1] < t_bound[2]) { cur[1] += dir[1]; t_bound[1] = PA(t_bound[1], t_step[1]); }
            else { cur[2] += dir[2]; t_bound[2] = PA(t_bound[2], t_step[2]); }
        }
        const int g[3] = {tp_rog_cell(v.g, pt[0]), tp_rog_cell(v.g, pt[1]), tp_rog_cell(v.g, pt[2])};
        if (!pm_inside(v, g[0], g[1], g[2])) break;
        pm_insert(v, g[0], g[1], g[2], false);
    }
}

// probabilisticMapFromCache (prob_map.cpp:543-569). first_frame: every cached cell takes `operations` misses of
// weight 999 one after the other (the sphere clearing of :357-372 visits a cell once per sample that falls in it).
__global__ void k_prob_apply(TpProbView v, TpRog e, int16_t* occ_cnt, int16_t* unk_cnt, int first_frame) {
    const int n = *v.cache_n;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const size_t h = (size_t)v.cache[k];
        const unsigned int c = v.cnt[h];
        const int hits = (int)(c >> 16), ops = (int)(c & 0xffffu);
        v.cnt[h] = 0u;
        float ret = v.occ[h];
        double pos[3];
        pm_hash_to_pos(v, h, pos);
        const int reps = first_frame ? ops : 1;
        for (int rep = 0; rep < reps; rep++) {
            const int from = pm_type(v, ret);
            if (!first_frame && hits > 0) {
                ret = __fadd_rn(ret, __fmul_rn(v.l_hit, (float)hits));
                if (ret > v.l_max) ret = v.l_max;
            } else {
                ret = __fadd_rn(ret, __fmul_rn(v.l_miss, (float)(first_frame ? 999 : ops - hits)));
                if (ret < v.l_min) ret = v.l_min;
            }
            const int to = pm_type(v, ret);
            if (from != to) pm_notify(e, occ_cnt, unk_cnt, pos, from, to);
        }
        v.occ[h] = ret;
    }
}

// SlidingMap::clearMemoryOutOfMap with ProbMap::resetCell (sliding_map.cpp:99-111, prob_map.cpp:512-541): the
// `count` planes that leave the ring along `axis`; v carries the OLD origin (hashIdToPos runs before it moves)
__global__ void k_prob_clear(TpProbView v, TpRog e, int16_t* occ_cnt, int16_t* unk_cnt, int axis, int min_l, int count,
                             int step) {
    const int a1 = (axis + 1) % 3, a2 = (axis + 2) % 3;
    const size_t plane = (size_t)v.g.size[a1] * v.g.size[a2];
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= plane * count) return;
    const int k = (int)(idx / plane);
    const size_t rr = idx % plane;
    const int kk = step > 0 ? k : -1 - k;
    const int range = v.g.size[axis];
    int yv = (min_l + kk + v.g.half[axis]) % range;
    if (yv < 0) yv += range;
    int l[3];
    l[axis] = yv;
    l[a1] = (int)(rr / v.g.size[a2]);
    l[a2] = (int)(rr % v.g.size[a2]);
    const size_t h = ((size_t)l[0] * v.g.size[1] + l[1]) * v.g.size[2] + l[2];
    const float ret = v.occ[h];
    const int from = pm_type(v, ret);
    if (from != TOPAY_ROG_UNKNOWN) {
        double pos[3];
        pm_hash_to_pos(v, h, pos);
        pm_notify(e, occ_cnt, unk_cnt, pos, from, TOPAY_ROG_UNKNOWN);
    }
    v.occ[h] = 0.f;
}

// the first-frame sphere (prob_map.cpp:357-372): every cell of the list takes `count` misses of weight 999 one after
// the other, straight on the log-odds (the hit / operation caches may hold a pending batch and are not touched)
__global__ void k_prob_first(TpProbView v, TpRog e, int16_t* occ_cnt, int16_t* unk_cnt, const int32_t* __restrict__ cells,
                             const int32_t* __restrict__ counts, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const size_t h = (size_t)cells[k];
    float ret = v.occ[h];
    double pos[3];
    pm_hash_to_pos(v, h, pos);
    for (int rep = 0; rep < counts[k]; rep++) {
        const int from = pm_type(v, ret);
        ret = __fadd_rn(ret, __fmul_rn(v.l_miss, 999.f));
        if (ret < v.l_min) ret = v.l_min;
        const int to = pm_type(v, ret);
        if (from != to) pm_notify(e, occ_cnt, unk_cnt, pos, from, to);
    }
    v.occ[h] = ret;
}

}  // namespace

struct topay_probmap {
    topay_rogfield* esdf;
    TpRogCounters E;
    topay_prob_desc desc;
    TpProbView V;            // device pointers + geometry; origin_i kept current
    size_t vox;
    double origin_d[3], bound_min_d[3], bound_max_d[3];
    double sliding_thresh;
    bool sliding_en;
    double ceil_h, ground_h;
    int half_update_box_i[3];
    int point_filt_num, batch_update_size, intensity_thresh;
    bool raycasting_en;
    int batch_counter;
    bool inited, map_empty, first_frame;
    double box_min[3], box_max[3];
    float4* d_pts;
    double* d_rays;
    size_t cap_pts;
    TpDevBuffers bufs;       // the ring's buffers; d_pts / d_rays grow with the largest cloud and are freed apart
};

namespace {

int pfloor(double v) { return (int)std::floor(v); }

void pm_set_origin(topay_probmap* m, const double od[3], const int oi[3]) {   // sliding_map.cpp:85-97
    for (int i = 0; i < 3; i++) {
        m->V.origin_i[i] = oi[i];
        m->origin_d[i] = od[i];
        m->bound_max_d[i] = ((double)(oi[i] + m->V.g.half[i]) + 0.5) * m->V.g.res;
        m->bound_min_d[i] = ((double)(oi[i] - m->V.g.half[i]) + 0.5) * m->V.g.res;
    }
}

void pm_reset_local_map(topay_probmap* m) {   // prob_map.cpp:822-833
    cudaStream_t q = m->E.stream;
    cudaMemsetAsync(m->V.occ, 0, m->vox * sizeof(float), q);
    cudaMemsetAsync(m->V.cnt, 0, m->vox * sizeof(unsigned int), q);
    cudaMemsetAsync(m->V.cache_n, 0, sizeof(int32_t), q);
    m->batch_counter = 0;
}

// SlidingMap::mapSliding (sliding_map.cpp:113-166) of the probability ring
void pm_map_sliding(topay_probmap* m, const double odom[3]) {
    const TpRog& g = m->V.g;
    int no[3], shift[3];
    double nd[3];
    for (int i = 0; i < 3; i++) {
        no[i] = pfloor(odom[i] * g.res_inv);
        nd[i] = (double)no[i] * g.res;
        shift[i] = no[i] - m->V.origin_i[i];
    }
    for (int i = 0; i < 3; i++)
        if (std::fabs((double)shift[i]) > g.size[i]) {
            pm_reset_local_map(m);
            pm_set_origin(m, nd, no);
            return;
        }
    for (int i = 0; i < 3; i++) {
        if (shift[i] == 0) continue;
        const int min_g = -g.half[i] + m->V.origin_i[i];
        const int min_l = min_g % g.size[i];
        const int count = std::abs(shift[i]);
        const size_t n = (size_t)g.size[(i + 1) % 3] * g.size[(i + 2) % 3] * count;
        k_prob_clear<<<(unsigned)((n + 255) / 256), 256, 0, m->E.stream>>>(m->V, m->E.view, m->E.occ_cnt, m->E.unk_cnt, i,
                                                                          min_l, count, shift[i] > 0 ? 1 : -1);
    }
    pm_set_origin(m, nd, no);
}

int pm_slide_all(topay_probmap* m, const double pos[3]) {   // prob_map.cpp:291-300
    pm_map_sliding(m, pos);
    TP_CUDA_OK(cudaStreamSynchronize(m->E.stream), {});
    return topay_rogfield_slide(m->esdf, pos);
}

void pm_apply(topay_probmap* m, int first_frame) {
    k_prob_apply<<<148 * 4, 256, 0, m->E.stream>>>(m->V, m->E.view, m->E.occ_cnt, m->E.unk_cnt, first_frame);
    cudaMemsetAsync(m->V.cache_n, 0, sizeof(int32_t), m->E.stream);
}

}  // namespace

extern "C" int topay_probmap_create(topay_rogfield* esdf, const topay_prob_desc* p, topay_probmap** out) {
    if (!esdf || !p || !out) return TOPAY_ERR_INVALID_ARG;
    topay_probmap* m = new topay_probmap();
    m->esdf = esdf;
    tp_rogfield_counters(esdf, &m->E);
    m->desc = *p;
    cudaSetDevice(m->E.device);
    const topay_rog_desc& d = m->E.desc;
    TpRog& g = m->V.g;
    memset(&g, 0, sizeof(g));
    g.res = d.prob_resolution;
    g.res_inv = 1.0 / d.prob_resolution;
    for (int i = 0; i < 3; i++) {
        g.half[i] = d.half_prob_map_size_i[i];
        g.size[i] = 2 * g.half[i] + 1;
    }
    m->vox = (size_t)g.size[0] * g.size[1] * g.size[2];
    if (m->vox >= ((size_t)1 << 31)) {
        delete m;
        tp_set_error("probability map too large for 32-bit cell hashes");
        return TOPAY_ERR_TOO_LARGE;
    }
    m->sliding_en = d.map_sliding_en != 0;
    m->sliding_thresh = p->map_sliding_thresh;
    auto logit = [](float x) -> float { return std::log(x / (1 - x)); };   // config.hpp:229-235, in float
    m->V.l_hit = logit(p->p_hit); m->V.l_miss = logit(p->p_miss); m->V.l_min = logit(p->p_min);
    m->V.l_max = logit(p->p_max); m->V.l_occ = logit(p->p_occ); m->V.l_free = logit(p->p_free);
    m->point_filt_num = p->point_filt_num <= 0 ? 1 : p->point_filt_num;
    m->batch_update_size = p->batch_update_size <= 0 ? 1 : p->batch_update_size;
    m->intensity_thresh = p->intensity_thresh;
    m->raycasting_en = p->raycasting_en != 0;
    for (int i = 0; i < 3; i++) m->half_update_box_i[i] = (int)((p->local_update_box[i] / 2) / d.prob_resolution);   // config.hpp:377-379
    {
        // InfMap's constructor pulls ceil / ground in by inflation_step cells of the inflation grid (inf_map.cpp:81-89;
        // config.hpp:338-349 rounds that grid up to a multiple of the resolution), initProbMap then snaps them
        // (prob_map.cpp:66-71)
        const double inf_req = p->inflation_resolution > 0 ? p->inflation_resolution : d.prob_resolution;
        const int inf_ratio = (int)std::ceil(inf_req / d.prob_resolution);
        const double inf_res = d.prob_resolution * inf_ratio;
        const int ceil_id = (int)(p->virtual_ceil_height / inf_res + 0.5) - p->inflation_step;
        const int ground_id = (int)(p->virtual_ground_height / inf_res + 0.5) + p->inflation_step;
        m->ceil_h = (double)pfloor((ceil_id * inf_res) * g.res_inv) * d.prob_resolution;
        m->ground_h = (double)pfloor((ground_id * inf_res) * g.res_inv) * d.prob_resolution;
    }
    m->map_empty = true;
    m->first_frame = true;
    TpDevBuffers& b = m->bufs;
    b.stream = m->E.stream;
    b.alloc(&m->V.occ, m->vox);
    b.alloc(&m->V.cnt, m->vox);
    b.alloc(&m->V.cache, m->vox);
    b.alloc(&m->V.cache_n, 1);
    if (b.status != TOPAY_OK) {
        const int rc = b.status;
        topay_probmap_destroy(m);
        return rc;
    }
    pm_reset_local_map(m);
    if (!m->sliding_en) {
        // sliding_map.cpp:58-61 + prob_map.cpp:73-77
        int oi[3];
        for (int i = 0; i < 3; i++) oi[i] = pfloor(d.fix_map_origin[i] * g.res_inv);
        for (int i = 0; i < 3; i++) {
            m->V.origin_i[i] = oi[i];
            m->origin_d[i] = d.fix_map_origin[i];
        }
        int rc = pm_slide_all(m, d.fix_map_origin);
        if (rc != TOPAY_OK) {
            topay_probmap_destroy(m);
            return rc;
        }
    }
    TP_CUDA_OK(cudaStreamSynchronize(m->E.stream), { topay_probmap_destroy(m); });
    *out = m;
    return TOPAY_OK;
}

extern "C" void topay_probmap_destroy(topay_probmap* m) {
    if (!m) return;
    cudaSetDevice(m->E.device);
    cudaStreamSynchronize(m->E.stream);
    for (void* p : {(void*)m->d_pts, (void*)m->d_rays})
        if (p) cudaFree(p);
    delete m;
}

extern "C" int topay_probmap_set_first_frame(topay_probmap* m, int armed) {
    if (!m) return TOPAY_ERR_INVALID_ARG;
    m->first_frame = armed != 0;
    return TOPAY_OK;
}

extern "C" int topay_probmap_download(topay_probmap* m, float* occupancy, int32_t origin_i[3]) {
    if (!m) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(m->E.device);
    if (occupancy) {
        TP_CUDA_OK(cudaMemcpyAsync(occupancy, m->V.occ, m->vox * sizeof(float), cudaMemcpyDeviceToHost, m->E.stream), {});
        TP_CUDA_OK(cudaStreamSynchronize(m->E.stream), {});
    }
    if (origin_i)
        for (int i = 0; i < 3; i++) origin_i[i] = m->V.origin_i[i];
    return TOPAY_OK;
}

extern "C" int topay_probmap_update(topay_probmap* m, const float* cloud, int64_t n, const double pos[3]) {
    if (!m || !pos || n < 0 || (n > 0 && !cloud)) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(m->E.device);
    cudaStream_t q = m->E.stream;
    const TpRog& g = m->V.g;
    int rc;
    auto inside = [&](const double p[3]) {
        return pm_inside(m->V, pfloor(p[0] * g.res_inv), pfloor(p[1] * g.res_inv), pfloor(p[2] * g.res_inv));
    };
    // prob_map.cpp:302-340
    if (m->sliding_en && !inside(pos) && m->batch_counter == 0) return pm_slide_all(m, pos);
    if (pos[2] > m->ceil_h) return TOPAY_OK;
    else if (pos[2] < m->ground_h) return TOPAY_OK;
    {
        const double d[3] = {pos[0] - m->origin_d[0], pos[1] - m->origin_d[1], pos[2] - m->origin_d[2]};
        const double nrm = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        if (m->batch_counter == 0 && (m->map_empty || (m->sliding_en && nrm > m->sliding_thresh)))
            if ((rc = pm_slide_all(m, pos)) != TOPAY_OK) return rc;
    }
    if (!m->inited) {
        m->inited = true;
        if ((rc = pm_slide_all(m, pos)) != TOPAY_OK) return rc;
    }
    // updateLocalBox (prob_map.cpp:791-820)
    for (int i = 0; i < 3; i++) {
        const int oi = pfloor(pos[i] * g.res_inv);
        const int hi = m->raycasting_en ? oi + m->half_update_box_i[i] : 0, lo = m->raycasting_en ? oi - m->half_update_box_i[i] : 0;
        m->box_max[i] = std::min(((double)hi + 0.5) * g.res, m->bound_max_d[i]);
        m->box_min[i] = std::max(((double)lo + 0.5) * g.res, m->bound_min_d[i]);
    }
    // raycastProcess: the two order-dependent filters (intensity, every point_filt_num-th of what is left,
    // prob_map.cpp:689-699) run on the host while the cloud is staged; everything per point is on the device
    std::vector<float> kept;
    kept.reserve((size_t)n * 4);
    int temporal = 0;
    for (int64_t i = 0; i < n; i++) {
        const float* c = cloud + 4 * i;
        if (m->intensity_thresh > 0 && c[3] < m->intensity_thresh) continue;
        if (temporal++ % m->point_filt_num) continue;
        kept.insert(kept.end(), c, c + 4);
    }
    const int64_t nk = (int64_t)kept.size() / 4;
    if (nk > 0) {
        if ((size_t)nk > m->cap_pts) {
            if (m->d_pts) cudaFree(m->d_pts);
            if (m->d_rays) cudaFree(m->d_rays);
            m->cap_pts = (size_t)nk * 2;
            TP_CUDA_OK(cudaMalloc(&m->d_pts, m->cap_pts * sizeof(float4)), {});
            TP_CUDA_OK(cudaMalloc(&m->d_rays, m->cap_pts * 3 * sizeof(double)), {});
        }
        TP_CUDA_OK(cudaMemcpyAsync(m->d_pts, kept.data(), (size_t)nk * sizeof(float4), cudaMemcpyHostToDevice, q), {});
        TpProbRay r;
        for (int i = 0; i < 3; i++) {
            r.odom[i] = pos[i];
            r.box_min[i] = m->box_min[i];
            r.box_max[i] = m->box_max[i];
        }
        r.ceil_h = m->ceil_h;
        r.ground_h = m->ground_h;
        r.range_min = m->desc.raycast_range_min;
        r.range_max = m->desc.raycast_range_max;
        r.sqr_range_max = m->desc.raycast_range_max * m->desc.raycast_range_max;
        r.raycasting_en = m->raycasting_en ? 1 : 0;
        const unsigned blocks = (unsigned)((nk + 127) / 128);
        k_prob_points<<<blocks, 128, 0, q>>>(m->V, r, m->d_pts, nk, m->d_rays);
        if (m->raycasting_en) k_prob_rays<<<blocks, 128, 0, q>>>(m->V, r, m->d_rays, nk);
        TP_CUDA_OK(cudaStreamSynchronize(q), {});     // `kept` is pageable host memory
    }
    m->batch_counter++;
    if (m->batch_counter >= m->batch_update_size) {
        m->batch_counter = 0;
        pm_apply(m, 0);
        m->map_empty = false;
    }
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    if ((rc = topay_rogfield_update_esdf(m->esdf, pos)) != TOPAY_OK) return rc;
    if (m->first_frame) {
        // prob_map.cpp:357-372: the samples of the triple loop (offsets accumulated exactly as `dx += resolution`
        // does), grouped per cell on the host — a few thousand samples, once in the life of the map
        m->first_frame = false;
        std::vector<double> off;
        const double rmin = m->desc.raycast_range_min;
        for (double dx = -rmin; dx <= rmin; dx += g.res) off.push_back(dx);
        std::vector<int32_t> cells, counts;
        for (double dx : off)
            for (double dy : off)
                for (double dz : off) {
                    if (!(std::sqrt(dx * dx + dy * dy + dz * dz) <= rmin)) continue;
                    const int32_t h = (int32_t)tp_rog_hash3(g, tp_rog_cell(g, pos[0] + dx), tp_rog_cell(g, pos[1] + dy),
                                                            tp_rog_cell(g, pos[2] + dz));
                    size_t k = 0;
                    while (k < cells.size() && cells[k] != h) k++;
                    if (k == cells.size()) {
                        cells.push_back(h);
                        counts.push_back(0);
                    }
                    counts[k]++;
                }
        if (!cells.empty()) {
            const size_t nc = cells.size();
            TpStaging io(q);
            const int32_t* d_cells = io.in(cells.data(), nc);
            const int32_t* d_counts = io.in(counts.data(), nc);
            if (io.ok())
                k_prob_first<<<(unsigned)((nc + 127) / 128), 128, 0, q>>>(m->V, m->E.view, m->E.occ_cnt, m->E.unk_cnt,
                                                                         d_cells, d_counts, (int)nc);
            return io.finish();
        }
    }
    return TOPAY_OK;
}
