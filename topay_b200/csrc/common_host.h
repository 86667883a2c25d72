// Host-side helpers shared by field.cu, edt.cu, rogfield.cu and solver.cu.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>

#include "hd.cuh"

void tp_set_error(const std::string& msg);
// TOPAY_OK when `device` is a usable CUDA device, else TOPAY_ERR_NO_DEVICE (the
// product path never falls back to the CPU).
int tp_require_device(int device);

int tp_field_device(const topay_field* f);
bool tp_field_ready(const topay_field* f);
void tp_field_grid(const topay_field* f, TpGrid* out);
int tp_rogfield_device(const topay_rogfield* f);
bool tp_rogfield_ready(const topay_rogfield* f);
void tp_rogfield_grid(const topay_rogfield* f, TpGrid* out);   // kind = 1
// what the probabilistic layer (probmap.cu) needs of the ESDF ring it feeds: geometry, the two counter arrays, its stream
struct TpRogCounters {
    TpRog view;
    int16_t *occ_cnt, *unk_cnt;
    cudaStream_t stream;
    int device;
    topay_rog_desc desc;
};
void tp_rogfield_counters(topay_rogfield* f, TpRogCounters* out);

// Optional sink of the EDT's last pass: instead of a dense esdf array the two distances go straight into
// the ROG ring buffers through the per-axis wrap rule (rogfield.cu; esdf_map.cpp:154-320).
struct TpRogSink {
    int enabled, dims3;          // dims3: box is [A][B][C] (x, y, z); else [B][C] (x, y)
    int lo[3], idl[3], mem_end[3], size[3];
    int B, C;                    // box extents of the two inner axes
    int fuse;                    // apply the sign combine on the spot (no wrap on any axis)
    double* dist;                // res * sqrt(positive transform)  (distance_buffer / 2-D map)
    double* neg;                 // res * sqrt(negative transform)  (tmp_buffer1_ / neg_buffer)
};

// Scratch of the separable exact EDT (edt.cu), shared by the dense and the ROG-ring field.
struct TpEdtScratch {
    cudaStream_t stream;
    int16_t* packed16;            // pass-1 output (sign-packed 1-D distances), A*B*C
    int32_t* packed32;            // pass-2 output (sign-packed squared distances), A*B*C (3-D only)
    bool keep_sq;                 // also store the integer squared distances
    double res;
    TpRogSink sink;               // enabled = 0 for the dense field
};
int tp_signed_edt(const TpEdtScratch& s, const int8_t* src, int A, int B, int C, double* esdf, int32_t* sqp,
                  int32_t* sqn);

// Per-call device scratch comes from the stream-ordered allocator: cudaFree synchronises the whole device, which
// stalls every other stream (concurrent solves of a scenario sweep, the plans of other host threads).
// tp_pool_keep keeps the default pool's memory across synchronisations (set once per device).
inline void tp_pool_keep(int device) {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
}

// cudaMalloc of `count` elements (at least one). On failure *p is null, the error text is set and the result is
// TOPAY_ERR_ALLOC.
template <typename T>
int tp_dev_malloc(T** p, size_t count) {
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) {
        tp_set_error(std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
        *p = nullptr;
        return TOPAY_ERR_ALLOC;
    }
    return TOPAY_OK;
}

// Raises `kernel`'s max dynamic shared memory to at least `bytes`. The attribute belongs to the kernel, not to one
// solver or field, and objects of different sizes coexist in a process (bench: 64-piece plans next to 16-piece latency
// plans), so it only ever grows: every call sets the largest size asked for that kernel so far.
inline cudaError_t tp_grow_dyn_smem(const void* kernel, size_t bytes) {
    static std::mutex mu;
    static std::map<const void*, size_t> high;
    std::lock_guard<std::mutex> lock(mu);
    size_t& h = high[kernel];
    h = std::max(h, bytes);
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h);
}

#define TP_CUDA_OK(call, cleanup)                                                              \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            tp_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                  \
            cleanup;                                                                           \
            return TOPAY_ERR_CUDA;                                                             \
        }                                                                                      \
    } while (0)
