// topay_rogfield: the sliding ring-buffer distance field of the reference's ROG-Map in HBM —
// rog_map::ESDFMap over CounterMap / SlidingMap (src/rog_map/src/rog_map/{esdf_map,counter_map,
// sliding_map}.cpp, ORIGIN_AT_CORNER).
//
//   slide            SlidingMap::mapSliding               sliding_map.cpp:113-166
//   update_counters  CounterMap::updateGridCounter        counter_map.cpp:94-151
//   update_esdf      ESDFMap::updateESDF3D + fillESDF     esdf_map.cpp:154-500, 842-900
//   query / line     evaluateEDT ... isLineFree2d         esdf_map.cpp:78-152, 903-1097
//
// The local update box is gathered out of the ring into a dense [bx][by][bz] occupancy array
// (one coalesced pass), transformed by the same exact integer EDT kernels as the dense field
// (edt.cu: z, y, x, both signs), and scattered back through the per-axis wrap rule. What the
// reference leaves behind in its persistent buffers is reproduced cell for cell, including the
// cells its combine step reads without the wrap (box coordinates used as memory coordinates,
// esdf_map.cpp:305-315, 391-398), which is why the negative distances live in their own ring
// buffer (tmp_buffer1_) here too.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common_host.h"
#include "rog_query.cuh"

struct topay_rogfield {
    topay_rog_desc desc;
    int device;
    cudaStream_t stream;
    double res, res_inv;
    int half[3], size[3];
    int origin_i[3], bmin_i[3], bmax_i[3], half_box_i[3];
    int sub_grid_num, unk_thresh;
    size_t n2, n3;
    int16_t *occ_cnt, *unk_cnt;
    double *dist3, *neg3, *crit, *flat, *neg2;
    int8_t *box_occ, *col_occ;          // dense box occupancy; [2][bx*by] column occupancy (critical, flat)
    int16_t* packed16;
    int32_t* packed32;
    cudaEvent_t ev0, ev1, ev2;
    float ms_total, ms_3d;
    bool updated;               // updateESDF3D ran at least once
    uint64_t generation;        // bumped by every update_esdf, the only writer of dist3 / crit / flat; read by a solver's
                                // submit, which the caller serialises with updates (one host thread at a time)
    TpDevBuffers bufs;
};

namespace {

struct RogBox {
    int lo[3], hi[3], idl[3], mem_end[3], size[3];
    int b[3];            // hi - lo + 1
};
__host__ __device__ __forceinline__ int rog_wrap(const RogBox& B, int q, int a) {
    return q > B.mem_end[a] ? q + B.idl[a] - B.size[a] : q + B.idl[a];
}

// ring -> dense box occupancy (z fastest on both sides)
__global__ void k_rog_gather(const int16_t* __restrict__ cnt, RogBox B, int8_t* __restrict__ out) {
    const size_t n = (size_t)B.b[0] * B.b[1] * B.b[2];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int z = (int)(i % B.b[2]);
        const size_t t = i / B.b[2];
        const int y = (int)(t % B.b[1]), x = (int)(t / B.b[1]);
        const size_t m = ((size_t)rog_wrap(B, x + B.lo[0], 0) * B.size[1] + rog_wrap(B, y + B.lo[1], 1)) * B.size[2] +
                         rog_wrap(B, z + B.lo[2], 2);
        out[i] = cnt[m] > 0 ? 1 : 0;
    }
}

// column occupancy of the box: any occupied cell over the whole z range (critical map,
// esdf_map.cpp:331-343) and over box z <= z_flat (flat map, :413-434)
__global__ void k_rog_columns(const int8_t* __restrict__ box, RogBox B, int nz_flat, int8_t* __restrict__ crit,
                              int8_t* __restrict__ flat) {
    const size_t n = (size_t)B.b[0] * B.b[1];
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int8_t* c = box + i * B.b[2];
    int any_c = 0, any_f = 0;
    for (int z = 0; z < B.b[2]; z++) {
        const int o = c[z];
        any_c |= o;
        if (z < nz_flat) any_f |= o;
    }
    crit[i] = (int8_t)any_c;
    flat[i] = (int8_t)any_f;
}

// esdf_map.cpp:305-315 over the un-wrapped box
__global__ void k_rog_combine3(RogBox B, double res, double* __restrict__ dist3, const double* __restrict__ neg3) {
    const size_t n = (size_t)B.b[0] * B.b[1] * B.b[2];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int z = (int)(i % B.b[2]);
        const size_t t = i / B.b[2];
        const int y = (int)(t % B.b[1]), x = (int)(t / B.b[1]);
        const size_t m = ((size_t)(x + B.lo[0]) * B.size[1] + (y + B.lo[1])) * B.size[2] + (z + B.lo[2]);
        const double dn = neg3[m];
        if (dn > 0.0) dist3[m] = __dadd_rn(dist3[m], __dadd_rn(-dn, res));
    }
}

// esdf_map.cpp:391-398 / :491-498: x and y both walk [lo_x, hi_x], un-wrapped; y clipped to the row
__global__ void k_rog_combine2(RogBox B, double res, double* __restrict__ out, const double* __restrict__ neg) {
    const int w = B.b[0];
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)w * w) return;
    const int x = (int)(i / w) + B.lo[0], y = (int)(i % w) + B.lo[0];
    if (y >= B.size[1]) return;
    const size_t m = (size_t)x * B.size[1] + y;
    const double dn = neg[m];
    if (dn > 0.0) out[m] = __dadd_rn(__dsub_rn(out[m], dn), res);
}

// clearMemoryOutOfMap (sliding_map.cpp:99-111): `count` planes of axis `axis`, local ids
// normalize(min_l + k*step), both counters reset (counter_map.h:127-131)
__global__ void k_rog_clear(int16_t* occ, int16_t* unk, int axis, int min_l, int count, int step, int h0, int h1,
                            int h2, int16_t sub_grid_num) {
    const int half[3] = {h0, h1, h2};
    const int size[3] = {2 * h0 + 1, 2 * h1 + 1, 2 * h2 + 1};
    const int a1 = (axis + 1) % 3, a2 = (axis + 2) % 3;
    const size_t plane = (size_t)size[a1] * size[a2];
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= plane * count) return;
    const int k = (int)(i / plane);
    const size_t r = i % plane;
    const int kk = step > 0 ? k : -1 - k;
    const int range = size[axis];
    int yv = (min_l + kk + half[axis]) % range;
    if (yv < 0) yv += range;
    int l[3];
    l[axis] = yv - half[axis];
    l[a1] = (int)(r / size[a2]) - half[a1];
    l[a2] = (int)(r % size[a2]) - half[a2];
    const size_t m = ((size_t)(l[0] + h0) * size[1] + (l[1] + h1)) * size[2] + (l[2] + h2);
    occ[m] = 0;
    unk[m] = sub_grid_num;
}

__global__ void k_fill16(int16_t* p, int16_t v, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// updateGridCounter (counter_map.cpp:94-151); additions commute, so the batch order is immaterial
__global__ void k_rog_counters(TpRog r, const double* __restrict__ pos, const uint8_t* __restrict__ from,
                               const uint8_t* __restrict__ to, int64_t n, int16_t* occ, int16_t* unk) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t m = tp_rog_hash3(r, tp_rog_cell(r, pos[3 * i]), tp_rog_cell(r, pos[3 * i + 1]),
                                  tp_rog_cell(r, pos[3 * i + 2]));
    const int d_occ = (to[i] == TOPAY_ROG_OCCUPIED) - (from[i] == TOPAY_ROG_OCCUPIED);
    const int d_unk = (to[i] == TOPAY_ROG_UNKNOWN) - (from[i] == TOPAY_ROG_UNKNOWN);
    if (d_occ) tp_atomic_add16(occ, m, d_occ);
    if (d_unk) tp_atomic_add16(unk, m, d_unk);
}

__global__ void k_rog_query(TpRog r, int kind, const double* __restrict__ pos, int64_t n, double* dist, double* grad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
    double d, g[3];
    bool has_grad = true;
    switch (kind) {
        case TOPAY_ROG_Q_EDT: tp_rog_value_grad(r, p, d, g); break;
        case TOPAY_ROG_Q_FLAT: tp_rog_value_grad2d(r, r.flat, p, d, g); break;
        case TOPAY_ROG_Q_CRITICAL: tp_rog_value_grad2d(r, r.crit, p, d, g); break;
        case TOPAY_ROG_Q_CELL: d = tp_rog_cell3(r, p); has_grad = false; break;
        case TOPAY_ROG_Q_CELL_FLAT: d = tp_rog_cell2(r, r.flat, p); has_grad = false; break;
        default: d = tp_rog_cell2(r, r.crit, p); has_grad = false; break;
    }
    dist[i] = d;
    if (grad && has_grad) {
        grad[3 * i] = g[0];
        grad[3 * i + 1] = g[1];
        grad[3 * i + 2] = g[2];
    }
}

__global__ void k_rog_line(TpRog r, const double* __restrict__ s, const double* __restrict__ e, int64_t n,
                           double threshold, int8_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a[2] = {s[2 * i], s[2 * i + 1]}, b[2] = {e[2 * i], e[2 * i + 1]};
    const long cap = labs((long)floor(b[0] / r.res) - (long)floor(a[0] / r.res)) +
                     labs((long)floor(b[1] / r.res) - (long)floor(a[1] / r.res)) + 1;
    out[i] = tp_rog_line_free2d(r, a, b, threshold, cap > (1L << 30) ? (1 << 30) : (int)cap) ? 1 : 0;
}

int ifloor(double v) { return (int)std::floor(v); }

// globalIndexToLocalIndex (sliding_map.cpp:205-218)
int to_local(const topay_rogfield* f, int g, int a) {
    int v = g % f->size[a];
    if (v > f->half[a]) v -= f->size[a];
    else if (v < -f->half[a]) v += f->size[a];
    return v;
}

void set_origin(topay_rogfield* f, const int o[3]) {   // sliding_map.cpp:85-97
    for (int i = 0; i < 3; i++) {
        f->origin_i[i] = o[i];
        f->bmax_i[i] = o[i] + f->half[i];
        f->bmin_i[i] = o[i] - f->half[i];
    }
}

TpRog rog_view(const topay_rogfield* f) {
    TpRog r;
    r.res = f->res;
    r.res_inv = f->res_inv;
    for (int i = 0; i < 3; i++) {
        r.half[i] = f->half[i];
        r.size[i] = f->size[i];
    }
    r.dist3 = f->dist3;
    r.crit = f->crit;
    r.flat = f->flat;
    return r;
}

int reset_counters(topay_rogfield* f) {   // esdf_map.cpp:72-76
    TP_CUDA_OK(cudaMemsetAsync(f->occ_cnt, 0, (f->n3 + 1) * sizeof(int16_t), f->stream), {});
    k_fill16<<<1024, 256, 0, f->stream>>>(f->unk_cnt, (int16_t)f->sub_grid_num, f->n3);
    return TOPAY_OK;
}

}  // namespace

int tp_rogfield_device(const topay_rogfield* f) { return f->device; }
void tp_rogfield_counters(topay_rogfield* f, TpRogCounters* out) {
    out->view = rog_view(f);
    out->occ_cnt = f->occ_cnt;
    out->unk_cnt = f->unk_cnt;
    out->stream = f->stream;
    out->device = f->device;
    out->desc = f->desc;
}
bool tp_rogfield_ready(const topay_rogfield* f) { return f->updated; }
void tp_rogfield_grid(const topay_rogfield* f, TpGrid* out) {
    memset(out, 0, sizeof(*out));
    out->kind = 1;
    out->rog = rog_view(f);
    out->resolution = f->res;
    out->resolution_inv = f->res_inv;
    out->ready = f->updated ? 1 : 0;
}
cudaStream_t tp_rogfield_stream(const topay_rogfield* f) { return f->stream; }
uint64_t tp_rogfield_generation(const topay_rogfield* f) { return f->generation; }
int tp_rogfield_snapshot(topay_rogfield* f, double* dist3, double* crit, double* flat, cudaEvent_t done) {
    cudaSetDevice(f->device);
    TP_CUDA_OK(cudaMemcpyAsync(dist3, f->dist3, f->n3 * 8, cudaMemcpyDeviceToDevice, f->stream), {});
    TP_CUDA_OK(cudaMemcpyAsync(crit, f->crit, f->n2 * 8, cudaMemcpyDeviceToDevice, f->stream), {});
    TP_CUDA_OK(cudaMemcpyAsync(flat, f->flat, f->n2 * 8, cudaMemcpyDeviceToDevice, f->stream), {});
    TP_CUDA_OK(cudaEventRecord(done, f->stream), {});
    return TOPAY_OK;
}

extern "C" int topay_rogfield_create(const topay_rog_desc* d, int device, topay_rogfield** out) {
    if (!d || !out || d->prob_resolution <= 0.0 || d->esdf_resolution < d->prob_resolution || d->unk_thresh < 0.0 ||
        d->unk_thresh > 1.0) {
        tp_set_error("rogfield: bad descriptor (counter_map.cpp:48-56 rejects these too)");
        return TOPAY_ERR_INVALID_ARG;
    }
    int rc = tp_require_device(device);
    if (rc != TOPAY_OK) return rc;
    topay_rogfield* f = new topay_rogfield();
    f->desc = *d;
    f->device = device;
    cudaSetDevice(device);
    tp_pool_keep(device);
    // counter_map.cpp:58-86 with inflation_step = 0 (esdf_map.cpp:37-44)
    const int ratio = (int)std::round(d->esdf_resolution / d->prob_resolution);
    const double cres = d->prob_resolution * ratio;
    for (int i = 0; i < 3; i++) {
        const double half_d = (double)d->half_prob_map_size_i[i] * d->prob_resolution;
        f->half[i] = (int)(half_d / cres) + 1;
        f->size[i] = 2 * f->half[i] + 1;
    }
    f->res = cres;
    f->res_inv = 1.0 / cres;
    if (f->size[0] >= 16383 || f->size[1] >= 16383 || f->size[2] >= 16383) {
        delete f;
        tp_set_error("rogfield: map dimensions out of range");
        return TOPAY_ERR_INVALID_ARG;
    }
    int o[3] = {0, 0, 0};
    if (!d->map_sliding_en)
        for (int i = 0; i < 3; i++) o[i] = ifloor(d->fix_map_origin[i] * f->res_inv);
    set_origin(f, o);
    f->sub_grid_num = (int)std::pow(std::round(cres / d->prob_resolution), 3);
    f->unk_thresh = (int)std::ceil(d->unk_thresh * f->sub_grid_num);
    f->unk_thresh = std::min(std::max(1, f->unk_thresh), f->sub_grid_num);
    for (int i = 0; i < 3; i++) f->half_box_i[i] = ifloor(d->local_update_box[i] * f->res_inv) / 2;   // esdf_map.cpp:51-52
    f->n2 = (size_t)f->size[0] * f->size[1];
    f->n3 = f->n2 * f->size[2];
    TP_CUDA_OK(cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking), { delete f; });
    TpDevBuffers& b = f->bufs;
    b.stream = f->stream;
    b.alloc(&f->occ_cnt, f->n3 + 1);   // +1: the 16-bit atomics work on aligned 32-bit words
    b.alloc(&f->unk_cnt, f->n3 + 1);
    b.alloc(&f->dist3, f->n3);
    b.alloc(&f->neg3, f->n3);
    b.alloc(&f->crit, f->n2);
    b.alloc(&f->flat, f->n2);
    b.alloc(&f->neg2, f->n2);
    b.alloc(&f->box_occ, f->n3);
    b.alloc(&f->col_occ, 2 * f->n2);
    b.alloc(&f->packed16, f->n3);
    b.alloc(&f->packed32, f->n3);
    if ((rc = b.status) != TOPAY_OK || (rc = reset_counters(f)) != TOPAY_OK) {
        topay_rogfield_destroy(f);
        return rc;
    }
    cudaEventCreate(&f->ev0);
    cudaEventCreate(&f->ev1);
    cudaEventCreate(&f->ev2);
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), { topay_rogfield_destroy(f); });
    *out = f;
    return TOPAY_OK;
}

extern "C" void topay_rogfield_destroy(topay_rogfield* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    if (f->stream) cudaStreamSynchronize(f->stream);
    if (f->ev0) cudaEventDestroy(f->ev0);
    if (f->ev1) cudaEventDestroy(f->ev1);
    if (f->ev2) cudaEventDestroy(f->ev2);
    if (f->stream) cudaStreamDestroy(f->stream);
    delete f;
}

extern "C" int topay_rogfield_geometry(const topay_rogfield* f, int32_t half[3], int32_t size[3], double* resolution,
                                       int32_t origin_i[3], int32_t half_box_i[3]) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    for (int i = 0; i < 3; i++) {
        if (half) half[i] = f->half[i];
        if (size) size[i] = f->size[i];
        if (origin_i) origin_i[i] = f->origin_i[i];
        if (half_box_i) half_box_i[i] = f->half_box_i[i];
    }
    if (resolution) *resolution = f->res;
    return TOPAY_OK;
}

extern "C" int topay_rogfield_slide(topay_rogfield* f, const double odom[3]) {
    if (!f || !odom) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    int no[3], shift[3];
    for (int i = 0; i < 3; i++) {
        no[i] = ifloor(odom[i] * f->res_inv);
        shift[i] = no[i] - f->origin_i[i];
    }
    for (int i = 0; i < 3; i++)
        if (std::fabs((double)shift[i]) > f->size[i]) {   // sliding_map.cpp:121-128
            int rc = reset_counters(f);
            if (rc != TOPAY_OK) return rc;
            set_origin(f, no);
            TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
            return TOPAY_OK;
        }
    for (int i = 0; i < 3; i++) {
        if (shift[i] == 0) continue;
        const int min_g = -f->half[i] + f->origin_i[i];
        const int min_l = min_g % f->size[i];
        const int count = std::abs(shift[i]);
        const size_t plane = (size_t)f->size[(i + 1) % 3] * f->size[(i + 2) % 3];
        const size_t n = plane * count;
        k_rog_clear<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(f->occ_cnt, f->unk_cnt, i, min_l, count,
                                                                       shift[i] > 0 ? 1 : -1, f->half[0], f->half[1],
                                                                       f->half[2], (int16_t)f->sub_grid_num);
    }
    set_origin(f, no);
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    return TOPAY_OK;
}

extern "C" int topay_rogfield_update_counters(topay_rogfield* f, const double* pos, const uint8_t* from_type,
                                              const uint8_t* to_type, int64_t n) {
    if (!f || n < 0 || (n > 0 && (!pos || !from_type || !to_type))) return TOPAY_ERR_INVALID_ARG;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* dp = io.in(pos, (size_t)n * 3);
    const uint8_t* dfrom = io.in(from_type, (size_t)n);
    const uint8_t* dto = io.in(to_type, (size_t)n);
    if (io.ok())
        k_rog_counters<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(rog_view(f), dp, dfrom, dto, n, f->occ_cnt,
                                                                          f->unk_cnt);
    return io.finish();
}

extern "C" int topay_rogfield_set_occupied_cnt(topay_rogfield* f, const int16_t* cnt) {
    if (!f || !cnt) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    TP_CUDA_OK(cudaMemcpyAsync(f->occ_cnt, cnt, f->n3 * 2, cudaMemcpyHostToDevice, f->stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
    return TOPAY_OK;
}

extern "C" int topay_rogfield_download_counters(topay_rogfield* f, int16_t* occupied_cnt, int16_t* unknown_cnt) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    if (occupied_cnt)
        TP_CUDA_OK(cudaMemcpyAsync(occupied_cnt, f->occ_cnt, f->n3 * 2, cudaMemcpyDeviceToHost, f->stream), {});
    if (unknown_cnt)
        TP_CUDA_OK(cudaMemcpyAsync(unknown_cnt, f->unk_cnt, f->n3 * 2, cudaMemcpyDeviceToHost, f->stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
    return TOPAY_OK;
}

extern "C" int topay_rogfield_update_esdf(topay_rogfield* f, const double cur_odom[3]) {
    if (!f || !cur_odom) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    cudaStream_t q = f->stream;
    RogBox B;
    bool wrapped = false;
    for (int i = 0; i < 3; i++) {
        const int cur = ifloor(cur_odom[i] * f->res_inv);
        B.size[i] = f->size[i];
        B.idl[i] = to_local(f, f->bmin_i[i], i) + f->half[i];
        B.mem_end[i] = f->size[i] - 1 - B.idl[i];
        const int umin = std::max(cur - f->half_box_i[i], f->bmin_i[i]);
        const int umax = std::min(cur + f->half_box_i[i], f->bmax_i[i]) - 1;
        B.lo[i] = umin - f->bmin_i[i];
        B.hi[i] = umax - f->bmin_i[i];
        B.b[i] = B.hi[i] - B.lo[i] + 1;
        if (B.idl[i] != 0) wrapped = true;
    }
    f->ms_total = f->ms_3d = 0.f;
    f->generation++;            // what a solver's snapshot copied before this call may no longer be the ring
    if (B.b[0] <= 0 || B.b[1] <= 0 || B.b[2] <= 0) {
        f->updated = true;
        return TOPAY_OK;
    }
    // the ring counts as built only once this update has completed: a failed update leaves it not ready
    f->updated = false;
    const size_t nb3 = (size_t)B.b[0] * B.b[1] * B.b[2], nb2 = (size_t)B.b[0] * B.b[1];
    const unsigned g3 = (unsigned)std::min<size_t>((nb3 + 255) / 256, 148 * 32);
    // the EDT's last pass writes res*sqrt of both transforms straight into the ring (TpRogSink)
    TpEdtScratch sc{q, f->packed16, f->packed32, false, f->res, TpRogSink{}};
    TpRogSink& sk = sc.sink;
    sk.enabled = 1;
    for (int i = 0; i < 3; i++) {
        sk.lo[i] = B.lo[i];
        sk.idl[i] = B.idl[i];
        sk.mem_end[i] = B.mem_end[i];
        sk.size[i] = B.size[i];
    }
    int rc;
    cudaEventRecord(f->ev0, q);
    k_rog_gather<<<g3, 256, 0, q>>>(f->occ_cnt, B, f->box_occ);
    sk.dims3 = 1;
    sk.B = B.b[1];
    sk.C = B.b[2];
    sk.fuse = wrapped ? 0 : 1;     // no wrap: the image is the memory box, combine on the spot
    sk.dist = f->dist3;
    sk.neg = f->neg3;
    if ((rc = tp_signed_edt(sc, f->box_occ, B.b[0], B.b[1], B.b[2], nullptr, nullptr, nullptr)) != TOPAY_OK) {
        cudaStreamSynchronize(q);
        return rc;
    }
    if (wrapped) k_rog_combine3<<<g3, 256, 0, q>>>(B, f->res, f->dist3, f->neg3);
    cudaEventRecord(f->ev1, q);
    // 2-D maps: flat covers box z up to the ring coordinate of z = 0.155 m (esdf_map.cpp:413-421)
    const int lz = to_local(f, ifloor(0.155 * f->res_inv), 2) + f->half[2];
    const int z_hi = lz < B.hi[2] ? lz : B.hi[2];
    const int nz_flat = std::max(0, z_hi - B.lo[2] + 1);
    const unsigned g2 = (unsigned)((nb2 + 255) / 256);
    k_rog_columns<<<g2, 256, 0, q>>>(f->box_occ, B, nz_flat, f->col_occ, f->col_occ + nb2);
    sk.dims3 = 0;
    sk.B = B.b[0];
    sk.C = B.b[1];
    sk.fuse = 0;                   // the 2-D combine walks its own (quirky) index range
    sk.neg = f->neg2;
    for (int which = 0; which < 2; which++) {
        sk.dist = which == 0 ? f->crit : f->flat;
        cudaMemsetAsync(f->neg2, 0, f->n2 * 8, q);
        if ((rc = tp_signed_edt(sc, f->col_occ + which * nb2, 1, B.b[0], B.b[1], nullptr, nullptr, nullptr)) != TOPAY_OK) {
            cudaStreamSynchronize(q);
            return rc;
        }
        const size_t nc = (size_t)B.b[0] * B.b[0];
        k_rog_combine2<<<(unsigned)((nc + 255) / 256), 256, 0, q>>>(B, f->res, sk.dist, f->neg2);
    }
    cudaEventRecord(f->ev2, q);
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, f->ev0, f->ev1);
    cudaEventElapsedTime(&b, f->ev1, f->ev2);
    f->ms_total = a + b;
    f->ms_3d = a;
    f->updated = true;
    return TOPAY_OK;
}

extern "C" int topay_rogfield_last_update_ms(topay_rogfield* f, float* ms_total, float* ms_3d) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    if (ms_total) *ms_total = f->ms_total;
    if (ms_3d) *ms_3d = f->ms_3d;
    return TOPAY_OK;
}

extern "C" int topay_rogfield_query(topay_rogfield* f, int kind, const double* pos, int64_t n, double* dist,
                                    double* grad) {
    if (!f || n < 0 || kind < 0 || kind > TOPAY_ROG_Q_CELL_CRITICAL || (n > 0 && (!pos || !dist)))
        return TOPAY_ERR_INVALID_ARG;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* dpos = io.in(pos, (size_t)n * 3);
    double* ddist = io.out(dist, (size_t)n);
    double* dgrad = io.inout(grad, (size_t)n * 3);   // the cell kinds leave it as passed in
    if (io.ok())
        k_rog_query<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(rog_view(f), kind, dpos, n, ddist, dgrad);
    return io.finish();
}

extern "C" int topay_rogfield_is_line_free2d(topay_rogfield* f, const double* start, const double* end, int64_t n,
                                             double threshold, int8_t* out) {
    if (!f || n < 0 || (n > 0 && (!start || !end || !out))) return TOPAY_ERR_INVALID_ARG;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* ds = io.in(start, (size_t)n * 2);
    const double* de = io.in(end, (size_t)n * 2);
    int8_t* dout = io.out(out, (size_t)n);
    if (io.ok())
        k_rog_line<<<(unsigned)((n + 127) / 128), 128, 0, f->stream>>>(rog_view(f), ds, de, n, threshold, dout);
    return io.finish();
}

extern "C" int topay_rogfield_download(topay_rogfield* f, int which, double* out) {
    if (!f || !out || which < 0 || which > TOPAY_ROG_BUF_FLAT) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    const double* src = which == TOPAY_ROG_BUF_DIST3 ? f->dist3
                        : which == TOPAY_ROG_BUF_NEG3 ? f->neg3
                        : which == TOPAY_ROG_BUF_CRITICAL ? f->crit : f->flat;
    const size_t n = which <= TOPAY_ROG_BUF_NEG3 ? f->n3 : f->n2;
    return tp_download(f->stream, out, src, n * 8);
}
