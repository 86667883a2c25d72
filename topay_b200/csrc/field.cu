// topay_field: the dense occupancy / ESDF grid of the reference's GridMap in HBM.
//
//   rasterise   GridMap::regenerateMap ingest         src/map/src/grid_map.cpp:733-747
//   rebuild     GridMap::updateESDF + fillESDF        src/map/src/grid_map.cpp:89-123, 125-521
//   queries     getDisWithGradI2d/3d, getDistance2d/3d, isWholeBodyCollision
//                                                      src/map/include/map/grid_map.h:256-509, 613-650
//
// The distance transform itself is the exact integer EDT of edt.cu; this file holds the field's buffers and runs
// its five transforms in the reference's order.
//
// Layout (as the reference): 3-D x*Ny*Nz + y*Nz + z, 2-D x*Ny + y.
#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common_host.h"
#include "edt_line.cuh"
#include "field_query.cuh"
#include "robot.cuh"

static thread_local std::string g_last_error;
void tp_set_error(const std::string& msg) { g_last_error = msg; }
extern "C" const char* topay_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* topay_version(void) { return "topay_b200 0.1 (sm_100a)"; }
extern "C" const char* topay_strerror(int code) {
    switch (code) {
        case TOPAY_OK: return "ok";
        case TOPAY_ERR_INVALID_ARG: return "invalid argument";
        case TOPAY_ERR_NO_DEVICE: return "no usable CUDA device (the B200 path has no CPU fallback)";
        case TOPAY_ERR_CUDA: return "CUDA runtime error";
        case TOPAY_ERR_ALLOC: return "device allocation failed";
        case TOPAY_ERR_TOO_LARGE: return "problem larger than the configured capacity";
        case TOPAY_ERR_NOT_READY: return "field not built";
        default: return "unknown error";
    }
}

int tp_require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        tp_set_error("no usable CUDA device: libtopay_b200 runs on the GPU only");
        return TOPAY_ERR_NO_DEVICE;
    }
    return TOPAY_OK;
}

struct topay_field {
    topay_grid_desc desc;
    int device;
    cudaStream_t stream;
    TpGrid grid;            // device pointers + geometry
    int nx, ny, nz;
    size_t n2, n3;
    int8_t *occ3d, *occ2d, *occ2d_crit, *src2d;
    double *esdf3d, *esdf2d, *esdf2d_inflate, *esdf2d_crit;
    int16_t* packed16;      // pass-1 output, sign-packed 1-D distances (3-D sized)
    int32_t* packed32;      // pass-2 output, sign-packed squared distances (3-D sized)
    int32_t *sq_pos[4], *sq_neg[4];
    bool keep_sq;
    bool ready;
    cudaEvent_t ev0, ev1, ev2;
    float ms_total, ms_3d;
    TpDevBuffers bufs;
};

int tp_field_device(const topay_field* f) { return f->device; }
bool tp_field_ready(const topay_field* f) { return f->ready; }
int tp_field_require_ready(const topay_field* f) {
    if (f->ready) return TOPAY_OK;
    tp_set_error("field not built: call topay_field_rebuild first");
    return TOPAY_ERR_NOT_READY;
}
void tp_field_grid(const topay_field* f, TpGrid* out) { *out = f->grid; }

// ------------------------------------------------------------------ kernels

// grid_map.cpp:733-747: one thread per float32 point.
__global__ void k_rasterize(const float* __restrict__ xyz, int64_t n, TpGrid g, double chassis_height,
                            int8_t* occ3d, int8_t* occ2d, int8_t* occ2d_crit) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float px = xyz[3 * i], py = xyz[3 * i + 1], pz = xyz[3 * i + 2];
    const int nx = g.dims[0], ny = g.dims[1], nz = g.dims[2];
    const int ix = (int)floor(((double)px - g.origin[0]) * g.resolution_inv);
    const int iy = (int)floor(((double)py - g.origin[1]) * g.resolution_inv);
    const int iz = (int)floor(((double)pz - g.origin[2]) * g.resolution_inv);
    if (ix >= 0 && iy >= 0 && ix <= nx - 1 && iy <= ny - 1) {
        occ2d_crit[(size_t)ix * ny + iy] = 1;
        if ((double)pz < chassis_height) occ2d[(size_t)ix * ny + iy] = 1;
        if (iz >= 0 && iz <= nz - 1) occ3d[((size_t)ix * ny + iy) * nz + iz] = 1;
    }
}

// inflated maps: source = previous ESDF below the chassis radius (grid_map.cpp:288, 360)
__global__ void k_threshold(const double* __restrict__ esdf, double thr, int8_t* out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = esdf[i] < thr ? 1 : 0;
}

__global__ void k_query3d(TpGrid g, const double* __restrict__ pos, int64_t n, double* dist, double* grad,
                          int value_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
    if (value_only) {
        dist[i] = tp_distance3d(g, p);
        return;
    }
    double d, gr[3];
    tp_query3d(g, p, d, gr);
    dist[i] = d;
    if (grad) {
        grad[3 * i] = gr[0];
        grad[3 * i + 1] = gr[1];
        grad[3 * i + 2] = gr[2];
    }
}

__global__ void k_query2d(TpGrid g, const double* __restrict__ buf, const double* __restrict__ pos, int64_t n,
                          double* dist, double* grad, int value_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double p[2] = {pos[2 * i], pos[2 * i + 1]};
    if (value_only) {
        dist[i] = tp_distance2d(g, p);
        return;
    }
    double d, gr[2];
    tp_query2d(g, buf, p, d, gr);
    dist[i] = d;
    if (grad) {
        grad[2 * i] = gr[0];
        grad[2 * i + 1] = gr[1];
    }
}

// Batched predicates and nearest-cell lookups the front-end and the feasibility check use
// (grid_map.h:511-611, 695-724, 887-940). kind: 0 isCollision2d, 1 isCollision3d,
// 2 isLineCollisionGrid2d (a = p1, b = p2), 3 getDistCoarse2d, 4 getDistCoarse2i (ia = indices).
__global__ void k_field_misc(TpGrid g, int kind, const double* __restrict__ a, const double* __restrict__ b,
                             const int32_t* __restrict__ ia, int64_t n, double threshold, int critical, int8_t* flag,
                             double* val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    switch (kind) {
        case 0: {
            const double p[2] = {a[2 * i], a[2 * i + 1]};
            flag[i] = tp_is_collision2d(g, p, threshold) ? 1 : 0;
            break;
        }
        case 1: {
            const double p[3] = {a[3 * i], a[3 * i + 1], a[3 * i + 2]};
            flag[i] = tp_is_collision3d(g, p, threshold) ? 1 : 0;
            break;
        }
        case 2: {
            const double p[2] = {a[2 * i], a[2 * i + 1]}, q[2] = {b[2 * i], b[2 * i + 1]};
            flag[i] = tp_line_collision_grid2d(g, p, q, threshold) ? 1 : 0;
            break;
        }
        case 3: {
            const double p[2] = {a[2 * i], a[2 * i + 1]};
            int id[2];
            tp_pos_to_index2(g, p, id);
            val[i] = tp_dist_coarse2i(g, id[0], id[1], critical != 0);
            break;
        }
        default: val[i] = tp_dist_coarse2i(g, ia[2 * i], ia[2 * i + 1], critical != 0); break;
    }
}

// TopologyPRM::lineVisib (topo_prm.cpp:278-315), one thread per segment.
__global__ void k_line_visib(TpGrid g, const double* __restrict__ p1, const double* __restrict__ p2, int64_t n,
                             double thresh, int critical, int8_t* visible, double* pc) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a[3] = {p1[3 * i], p1[3 * i + 1], p1[3 * i + 2]}, b[3] = {p2[3 * i], p2[3 * i + 1], p2[3 * i + 2]};
    double c[3] = {pc[3 * i], pc[3 * i + 1], pc[3 * i + 2]};
    visible[i] = tp_line_visib(g, a, b, thresh, critical != 0, c) ? 1 : 0;
    pc[3 * i] = c[0];
    pc[3 * i + 1] = c[1];
    pc[3 * i + 2] = c[2];
}

// GridMap::isWholeBodyCollision (grid_map.h:613-650), one thread per 10-D state.
__global__ void k_whole_body(TpGrid g, TpParams P, const double* __restrict__ states, int64_t n, int8_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* s = states + 10 * i;
    const topay_robot_params& rp = P.robot;
    bool hit = false;
    for (int q = 0; q < TOPAY_DOF; q++)
        if (s[3 + q] > rp.joint_pos_limit_max[q] || s[3 + q] < -rp.joint_pos_limit_max[q]) hit = true;
    if (!hit) {
        const double p2[2] = {s[0], s[1]};
        if (!tp_in_map2(g, p2) || tp_distance2d(g, p2) < rp.chassis_colli_radius) hit = true;
    }
    if (!hit) {
        double pos[10];
        for (int k = 0; k < 10; k++) pos[k] = s[k];
        TpFK fk;
        TpSphereStoreLocal pts;
        tp_fk(P, pos, fk, pts);
        for (int a = 0; a < P.n_sphere && !hit; a++) {
            const double r = P.sphere_r[a];
            const double pa[3] = {pts.at(a, 0), pts.at(a, 1), pts.at(a, 2)};
            if (!tp_in_map3(g, pa) || tp_distance3d(g, pa) < r) hit = true;
            if (a > 2 && pa[2] < rp.chassis_height + r) {
                const double dx = pa[0] - s[0], dy = pa[1] - s[1];
                if (sqrt(dx * dx + dy * dy) < rp.chassis_colli_radius + r) hit = true;
            }
            for (int b = a + 1; b < P.n_sphere; b++) {
                const double dx = pa[0] - pts.at(b, 0), dy = pa[1] - pts.at(b, 1), dz = pa[2] - pts.at(b, 2);
                if (sqrt(dx * dx + dy * dy + dz * dz) < r + P.sphere_r[b] && ((P.pair_mask[a] >> b) & 1u)) hit = true;
            }
        }
    }
    out[i] = hit ? 1 : 0;
}

// ------------------------------------------------------------------ host

namespace {

// One signed transform over a [A][B][C] array through the field's scratch (edt.cu).
int signed_edt(topay_field* f, const int8_t* src, int A, int B, int C, double* esdf, int32_t* sqp, int32_t* sqn) {
    TpEdtScratch sc{f->stream, f->packed16, f->packed32, f->keep_sq, f->desc.resolution, TpRogSink{}};
    return tp_signed_edt(sc, src, A, B, C, esdf, sqp, sqn);
}

}  // namespace

extern "C" int topay_field_create(const topay_grid_desc* desc, int device, topay_field** out) {
    if (!desc || !out || desc->resolution <= 0.0) return TOPAY_ERR_INVALID_ARG;
    int rc = tp_require_device(device);
    if (rc != TOPAY_OK) return rc;
    topay_field* f = new topay_field();
    f->desc = *desc;
    f->device = device;
    f->keep_sq = true;
    cudaSetDevice(device);
    tp_pool_keep(device);
    // grid_map.cpp:33-54
    TpGrid& g = f->grid;
    g.resolution = desc->resolution;
    g.resolution_inv = 1.0 / desc->resolution;
    for (int i = 0; i < 3; i++) {
        g.min_boundary[i] = -desc->map_size[i] / 2.0;
        g.max_boundary[i] = desc->map_size[i] / 2.0;
    }
    g.min_boundary[2] = 0.0;
    g.max_boundary[2] = desc->map_size[2];
    for (int i = 0; i < 3; i++) {
        g.origin[i] = g.min_boundary[i];
        g.dims[i] = (int)ceil(desc->map_size[i] / desc->resolution);
    }
    f->nx = g.dims[0];
    f->ny = g.dims[1];
    f->nz = g.dims[2];
    if (f->nx < 1 || f->ny < 1 || f->nz < 1 || f->nx >= TP_INF16 || f->ny >= TP_INF16 || f->nz >= TP_INF16) {
        delete f;
        tp_set_error("grid dimensions out of range");
        return TOPAY_ERR_INVALID_ARG;
    }
    f->n2 = (size_t)f->nx * f->ny;
    f->n3 = f->n2 * f->nz;
    TP_CUDA_OK(cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking), { delete f; });
    TpDevBuffers& b = f->bufs;
    b.stream = f->stream;
    b.alloc(&f->occ3d, f->n3);
    b.alloc(&f->occ2d, f->n2);
    b.alloc(&f->occ2d_crit, f->n2);
    b.alloc(&f->src2d, f->n2);
    b.alloc(&f->esdf3d, f->n3);
    b.alloc(&f->esdf2d, f->n2);
    b.alloc(&f->esdf2d_inflate, f->n2);
    b.alloc(&f->esdf2d_crit, f->n2);
    b.alloc(&f->packed16, f->n3);
    b.alloc(&f->packed32, f->n3);
    for (int w = 0; w < 4; w++) {
        b.alloc(&f->sq_pos[w], w < 3 ? f->n2 : f->n3);
        b.alloc(&f->sq_neg[w], w < 3 ? f->n2 : f->n3);
    }
    if (b.status != TOPAY_OK) {
        rc = b.status;
        topay_field_destroy(f);
        return rc;
    }
    g.esdf3d = f->esdf3d;
    g.esdf2d = f->esdf2d;
    g.esdf2d_inflate = f->esdf2d_inflate;
    g.esdf2d_critical = f->esdf2d_crit;
    g.ready = 0;
    cudaEventCreate(&f->ev0);
    cudaEventCreate(&f->ev1);
    cudaEventCreate(&f->ev2);
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), { topay_field_destroy(f); });
    *out = f;
    return TOPAY_OK;
}

extern "C" void topay_field_destroy(topay_field* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    if (f->stream) cudaStreamSynchronize(f->stream);
    if (f->ev0) cudaEventDestroy(f->ev0);
    if (f->ev1) cudaEventDestroy(f->ev1);
    if (f->ev2) cudaEventDestroy(f->ev2);
    if (f->stream) cudaStreamDestroy(f->stream);
    delete f;
}

extern "C" int topay_field_dims(const topay_field* f, int32_t dims[3]) {
    if (!f || !dims) return TOPAY_ERR_INVALID_ARG;
    dims[0] = f->nx;
    dims[1] = f->ny;
    dims[2] = f->nz;
    return TOPAY_OK;
}

extern "C" int topay_field_set_keep_sqdist(topay_field* f, int keep) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    f->keep_sq = keep != 0;
    return TOPAY_OK;
}

extern "C" int topay_field_set_occupancy(topay_field* f, const int8_t* occ3d, const int8_t* occ2d,
                                         const int8_t* occ2d_critical) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    if (occ3d) TP_CUDA_OK(cudaMemcpyAsync(f->occ3d, occ3d, f->n3, cudaMemcpyHostToDevice, f->stream), {});
    if (occ2d) TP_CUDA_OK(cudaMemcpyAsync(f->occ2d, occ2d, f->n2, cudaMemcpyHostToDevice, f->stream), {});
    if (occ2d_critical)
        TP_CUDA_OK(cudaMemcpyAsync(f->occ2d_crit, occ2d_critical, f->n2, cudaMemcpyHostToDevice, f->stream), {});
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
    f->ready = false;
    f->grid.ready = 0;
    return TOPAY_OK;
}

extern "C" int topay_field_clear(topay_field* f, int clear_critical) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    cudaMemsetAsync(f->occ3d, 0, f->n3, f->stream);
    cudaMemsetAsync(f->occ2d, 0, f->n2, f->stream);
    if (clear_critical) cudaMemsetAsync(f->occ2d_crit, 0, f->n2, f->stream);
    f->ready = false;
    f->grid.ready = 0;
    return TOPAY_OK;
}

extern "C" int topay_field_rasterize_points(topay_field* f, const float* xyz, int64_t n) {
    if (!f || (!xyz && n > 0) || n < 0) return TOPAY_ERR_INVALID_ARG;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const float* d = io.in(xyz, (size_t)n * 3);
    if (io.ok())
        k_rasterize<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(d, n, f->grid, f->desc.chassis_height, f->occ3d,
                                                                      f->occ2d, f->occ2d_crit);
    const int rc = io.finish();
    if (rc != TOPAY_OK) return rc;
    f->ready = false;
    f->grid.ready = 0;
    return TOPAY_OK;
}

extern "C" int topay_field_rebuild(topay_field* f) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    cudaStream_t q = f->stream;
    const unsigned tb = (unsigned)((f->n2 + 255) / 256);
    int rc;
    cudaEventRecord(f->ev0, q);
    // the four 2-D maps, in the reference's order (grid_map.cpp:138-423)
    if ((rc = signed_edt(f, f->occ2d, 1, f->nx, f->ny, f->esdf2d, f->sq_pos[0], f->sq_neg[0])) != TOPAY_OK) return rc;
    if ((rc = signed_edt(f, f->occ2d_crit, 1, f->nx, f->ny, f->esdf2d_crit, f->sq_pos[2], f->sq_neg[2])) != TOPAY_OK)
        return rc;
    k_threshold<<<tb, 256, 0, q>>>(f->esdf2d_crit, f->desc.chassis_colli_radius, f->src2d, f->n2);
    if ((rc = signed_edt(f, f->src2d, 1, f->nx, f->ny, f->esdf2d_crit, f->sq_pos[2], f->sq_neg[2])) != TOPAY_OK)
        return rc;
    k_threshold<<<tb, 256, 0, q>>>(f->esdf2d, f->desc.chassis_colli_radius, f->src2d, f->n2);
    if ((rc = signed_edt(f, f->src2d, 1, f->nx, f->ny, f->esdf2d_inflate, f->sq_pos[1], f->sq_neg[1])) != TOPAY_OK)
        return rc;
    cudaEventRecord(f->ev1, q);
    // the 3-D map (grid_map.cpp:425-518): z, y, x
    if ((rc = signed_edt(f, f->occ3d, f->nx, f->ny, f->nz, f->esdf3d, f->sq_pos[3], f->sq_neg[3])) != TOPAY_OK)
        return rc;
    cudaEventRecord(f->ev2, q);
    TP_CUDA_OK(cudaStreamSynchronize(q), {});
    TP_CUDA_OK(cudaGetLastError(), {});
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, f->ev0, f->ev1);
    cudaEventElapsedTime(&b, f->ev1, f->ev2);
    f->ms_total = a + b;
    f->ms_3d = b;
    f->ready = true;
    f->grid.ready = 1;
    return TOPAY_OK;
}

extern "C" int topay_field_last_rebuild_ms(topay_field* f, float* ms_total, float* ms_3d) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    if (ms_total) *ms_total = f->ms_total;
    if (ms_3d) *ms_3d = f->ms_3d;
    return TOPAY_OK;
}

static int query_common(topay_field* f, const double* pos, int64_t n, int dim, int which, double* dist,
                        double* grad, int value_only) {
    if (!f || (!pos && n > 0) || !dist || n < 0) return TOPAY_ERR_INVALID_ARG;
    const int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* dpos = io.in(pos, (size_t)n * dim);
    double* dd = io.out(dist, (size_t)n);
    double* dg = io.out(grad, (size_t)n * dim);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const double* buf = which == TOPAY_MAP2D_CRITICAL ? f->esdf2d_crit
                        : which == TOPAY_MAP2D_INFLATE ? f->esdf2d_inflate : f->esdf2d;
    if (io.ok() && dim == 3) k_query3d<<<blocks, 256, 0, f->stream>>>(f->grid, dpos, n, dd, dg, value_only);
    if (io.ok() && dim == 2) k_query2d<<<blocks, 256, 0, f->stream>>>(f->grid, buf, dpos, n, dd, dg, value_only);
    return io.finish();
}

extern "C" int topay_field_query3d(topay_field* f, const double* pos, int64_t n, double* dist, double* grad) {
    return query_common(f, pos, n, 3, TOPAY_MAP3D, dist, grad, 0);
}
extern "C" int topay_field_query2d(topay_field* f, const double* pos, int64_t n, int which, double* dist,
                                   double* grad) {
    if (which < 0 || which > 2) return TOPAY_ERR_INVALID_ARG;
    return query_common(f, pos, n, 2, which, dist, grad, 0);
}
extern "C" int topay_field_distance3d(topay_field* f, const double* pos, int64_t n, double* dist) {
    return query_common(f, pos, n, 3, TOPAY_MAP3D, dist, nullptr, 1);
}
extern "C" int topay_field_distance2d(topay_field* f, const double* pos, int64_t n, double* dist) {
    return query_common(f, pos, n, 2, TOPAY_MAP2D_FLAT, dist, nullptr, 1);
}

extern "C" int topay_field_query3d_dev(topay_field* f, const double* pos_dev, int64_t n, double* dist_dev,
                                       double* grad_dev) {
    if (!f || !pos_dev || !dist_dev || n < 0) return TOPAY_ERR_INVALID_ARG;
    const int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    k_query3d<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(f->grid, pos_dev, n, dist_dev, grad_dev, 0);
    TP_CUDA_OK(cudaGetLastError(), {});
    return TOPAY_OK;
}
extern "C" int topay_field_sync(topay_field* f) {
    if (!f) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    TP_CUDA_OK(cudaStreamSynchronize(f->stream), {});
    return TOPAY_OK;
}

extern "C" int topay_field_whole_body_collision(topay_field* f, const topay_robot_params* robot,
                                                const double* states, int64_t n, int8_t* out) {
    if (!f || !robot || (!states && n > 0) || !out || n < 0) return TOPAY_ERR_INVALID_ARG;
    const int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpParams P;
    memset(&P, 0, sizeof(P));
    P.robot = *robot;
    topay_opt_params_default(&P.opt);
    tp_derive_params(P);
    TpStaging io(f->stream);
    const double* ds = io.in(states, (size_t)n * 10);
    int8_t* dout = io.out(out, (size_t)n);
    if (io.ok()) k_whole_body<<<(unsigned)((n + 127) / 128), 128, 0, f->stream>>>(f->grid, P, ds, n, dout);
    return io.finish();
}

// kind as k_field_misc; in_a / in_b: n x wa doubles (host), in_i: n x 2 int32 (host)
static int field_misc(topay_field* f, int kind, const double* in_a, int wa, const double* in_b, const int32_t* in_i,
                      int64_t n, double threshold, int critical, int8_t* flag, double* val) {
    if (!f || n < 0 || (n > 0 && ((kind <= 3 && !in_a) || (kind == 2 && !in_b) || (kind == 4 && !in_i) ||
                                  (kind <= 2 && !flag) || (kind >= 3 && !val))))
        return TOPAY_ERR_INVALID_ARG;
    const int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* da = io.in(in_a, (size_t)n * wa);
    const double* db = io.in(in_b, (size_t)n * wa);
    const int32_t* di = io.in(in_i, (size_t)n * 2);
    int8_t* df = io.out(kind <= 2 ? flag : nullptr, (size_t)n);
    double* dv = io.out(kind <= 2 ? nullptr : val, (size_t)n);
    if (io.ok())
        k_field_misc<<<(unsigned)((n + 255) / 256), 256, 0, f->stream>>>(f->grid, kind, da, db, di, n, threshold,
                                                                        critical, df, dv);
    return io.finish();
}

extern "C" int topay_field_is_collision2d(topay_field* f, const double* pos, int64_t n, double threshold, int8_t* out) {
    return field_misc(f, 0, pos, 2, nullptr, nullptr, n, threshold, 0, out, nullptr);
}
extern "C" int topay_field_is_collision3d(topay_field* f, const double* pos, int64_t n, double threshold, int8_t* out) {
    return field_misc(f, 1, pos, 3, nullptr, nullptr, n, threshold, 0, out, nullptr);
}
extern "C" int topay_field_is_line_collision_grid2d(topay_field* f, const double* p1, const double* p2, int64_t n,
                                                    double threshold, int8_t* out) {
    return field_misc(f, 2, p1, 2, p2, nullptr, n, threshold, 0, out, nullptr);
}
extern "C" int topay_field_dist_coarse2d(topay_field* f, const double* pos, int64_t n, int critical, double* out) {
    return field_misc(f, 3, pos, 2, nullptr, nullptr, n, 0.0, critical, nullptr, out);
}
extern "C" int topay_field_dist_coarse2i(topay_field* f, const int32_t* idx, int64_t n, int critical, double* out) {
    return field_misc(f, 4, nullptr, 2, nullptr, idx, n, 0.0, critical, nullptr, out);
}

extern "C" int topay_field_line_visible(topay_field* f, const double* p1, const double* p2, int64_t n, double thresh,
                                        int use_critical, int8_t* visible, double* pc) {
    if (!f || n < 0 || (n > 0 && (!p1 || !p2 || !visible || !pc))) return TOPAY_ERR_INVALID_ARG;
    const int rc = tp_field_require_ready(f);
    if (rc != TOPAY_OK) return rc;
    if (n == 0) return TOPAY_OK;
    cudaSetDevice(f->device);
    TpStaging io(f->stream);
    const double* d1 = io.in(p1, (size_t)n * 3);
    const double* d2 = io.in(p2, (size_t)n * 3);
    double* dc = io.inout(pc, (size_t)n * 3);      // pc of a visible segment stays as passed in
    int8_t* dv = io.out(visible, (size_t)n);
    if (io.ok())
        k_line_visib<<<(unsigned)((n + 127) / 128), 128, 0, f->stream>>>(f->grid, d1, d2, n, thresh, use_critical, dv,
                                                                        dc);
    return io.finish();
}

extern "C" int topay_discretize_path(const double* path, int n, int pt_num, double* out);
extern "C" double topay_path_length(const double* path, int n);

// TopologyPRM::sameTopoPath (topo_prm.cpp:424-448) for many pairs of paths at once: the equally spaced points of
// both paths of every pair (host arithmetic) become one batch of visibility rays (one launch), a pair is the same
// class when all of its rays are free.
extern "C" int topay_field_same_topo_paths(topay_field* f, const double* pts, const int32_t* offsets, int n_paths,
                                           const int32_t* pairs, int n_pairs, double thresh, int use_critical,
                                           int8_t* same) {
    if (!f || !pts || !offsets || !pairs || !same || n_paths < 1 || n_pairs < 0) return TOPAY_ERR_INVALID_ARG;
    std::vector<double> p1, p2;
    std::vector<int64_t> first(n_pairs + 1, 0);
    std::vector<double> a, b;
    for (int k = 0; k < n_pairs; k++) {
        const int i = pairs[2 * k], j = pairs[2 * k + 1];
        if (i < 0 || j < 0 || i >= n_paths || j >= n_paths) return TOPAY_ERR_INVALID_ARG;
        const double *pa = pts + 3 * (size_t)offsets[i], *pb = pts + 3 * (size_t)offsets[j];
        const int na = offsets[i + 1] - offsets[i], nb = offsets[j + 1] - offsets[j];
        if (na < 2 || nb < 2) return TOPAY_ERR_INVALID_ARG;
        const double max_len = std::max(topay_path_length(pa, na), topay_path_length(pb, nb));
        const int pt_num = (int)ceil(max_len / f->desc.resolution);
        if (pt_num < 2) {       // both paths inside one cell: the reference divides by pt_num - 1 = 0 here
            tp_set_error("same_topo_paths: paths shorter than one cell");
            return TOPAY_ERR_INVALID_ARG;
        }
        a.resize((size_t)pt_num * 3);
        b.resize((size_t)pt_num * 3);
        topay_discretize_path(pa, na, pt_num, a.data());
        topay_discretize_path(pb, nb, pt_num, b.data());
        p1.insert(p1.end(), a.begin(), a.end());
        p2.insert(p2.end(), b.begin(), b.end());
        first[k + 1] = first[k] + pt_num;
    }
    const int64_t n = first[n_pairs];
    std::vector<int8_t> vis((size_t)std::max<int64_t>(n, 1));
    std::vector<double> pc((size_t)std::max<int64_t>(n, 1) * 3, 0.0);
    const int rc = topay_field_line_visible(f, p1.data(), p2.data(), n, thresh, use_critical, vis.data(), pc.data());
    if (rc != TOPAY_OK) return rc;
    for (int k = 0; k < n_pairs; k++) {
        int8_t all = 1;
        for (int64_t r = first[k]; r < first[k + 1]; r++) all &= vis[r];
        same[k] = all;
    }
    return TOPAY_OK;
}

extern "C" int topay_field_download(topay_field* f, int which, double* esdf_out) {
    if (!f || !esdf_out || which < 0 || which > 3) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    const double* src = which == TOPAY_MAP3D ? f->esdf3d
                        : which == TOPAY_MAP2D_CRITICAL ? f->esdf2d_crit
                        : which == TOPAY_MAP2D_INFLATE ? f->esdf2d_inflate : f->esdf2d;
    const size_t n = which == TOPAY_MAP3D ? f->n3 : f->n2;
    return tp_download(f->stream, esdf_out, src, n * 8);
}

extern "C" int topay_field_download_sqdist(topay_field* f, int which, int32_t* pos_sq, int32_t* neg_sq) {
    if (!f || which < 0 || which > 3) return TOPAY_ERR_INVALID_ARG;
    if (!f->keep_sq) {
        tp_set_error("integer grids were not kept (topay_field_set_keep_sqdist(f, 0))");
        return TOPAY_ERR_NOT_READY;
    }
    cudaSetDevice(f->device);
    const size_t n = which == TOPAY_MAP3D ? f->n3 : f->n2;
    int rc = TOPAY_OK;
    if (pos_sq) rc = tp_download(f->stream, pos_sq, f->sq_pos[which], n * 4);
    if (neg_sq && rc == TOPAY_OK) rc = tp_download(f->stream, neg_sq, f->sq_neg[which], n * 4);
    return rc;
}

extern "C" int topay_field_download_occupancy(topay_field* f, int which, int8_t* occ_out) {
    if (!f || !occ_out || which < 0 || which > 3 || which == TOPAY_MAP2D_INFLATE) return TOPAY_ERR_INVALID_ARG;
    cudaSetDevice(f->device);
    const int8_t* src = which == TOPAY_MAP3D ? f->occ3d : which == TOPAY_MAP2D_CRITICAL ? f->occ2d_crit : f->occ2d;
    const size_t n = which == TOPAY_MAP3D ? f->n3 : f->n2;
    return tp_download(f->stream, occ_out, src, n);
}
