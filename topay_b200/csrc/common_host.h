// Host-side helpers shared by the library's objects. Two of them carry every copy between host and device:
// TpStaging stages one batched call (per-call scratch from the stream-ordered allocator, copies in, copies back,
// one synchronise of the object's stream), and tp_download is a single download on the object's stream.
// TpDevBuffers owns an object's device buffers.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "hd.cuh"

void tp_set_error(const std::string& msg);
// TOPAY_OK when `device` is a usable CUDA device, else TOPAY_ERR_NO_DEVICE (the
// product path never falls back to the CPU).
int tp_require_device(int device);

int tp_field_device(const topay_field* f);
bool tp_field_ready(const topay_field* f);
// TOPAY_OK when the dense field has been rebuilt since its occupancy last changed, else TOPAY_ERR_NOT_READY with the
// error text set: the one readiness check of every entry point that reads the field.
int tp_field_require_ready(const topay_field* f);
void tp_field_grid(const topay_field* f, TpGrid* out);
int tp_rogfield_device(const topay_rogfield* f);
bool tp_rogfield_ready(const topay_rogfield* f);
void tp_rogfield_grid(const topay_rogfield* f, TpGrid* out);   // kind = 1
cudaStream_t tp_rogfield_stream(const topay_rogfield* f);     // the ring's own stream: every update runs on it
// Generation of dist3 / crit / flat: changes whenever one of them is written (topay_rogfield_update_esdf, which
// topay_probmap_update also runs). Slides and counter updates write only the counters.
uint64_t tp_rogfield_generation(const topay_rogfield* f);
// Copies dist3 [n3], crit and flat [n2 each] into caller memory on the ring's stream, then records `done` there: a
// reader on another stream waits on `done`, and later updates of the ring queue behind the copy.
int tp_rogfield_snapshot(topay_rogfield* f, double* dist3, double* crit, double* flat, cudaEvent_t done);
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

// The staging of one batched call on an object's stream. in() copies a host array to new device scratch, out()
// allocates scratch that finish() copies back, inout() does both; a null host pointer gives a null device pointer.
// The first failure is kept with its text (TOPAY_ERR_ALLOC for an allocation, TOPAY_ERR_CUDA for a copy) and every
// later step does nothing, so the caller launches only while ok(). The scratch is freed on the stream on every path.
class TpStaging {
  public:
    explicit TpStaging(cudaStream_t q) : q_(q) {}
    TpStaging(const TpStaging&) = delete;
    TpStaging& operator=(const TpStaging&) = delete;
    ~TpStaging() {
        for (const Buf& b : bufs_) cudaFreeAsync(b.dev, q_);
    }
    template <typename T>
    T* in(const T* host, size_t count) { return (T*)stage((void*)host, count * sizeof(T), true, false); }
    template <typename T>
    T* out(T* host, size_t count) { return (T*)stage(host, count * sizeof(T), false, true); }
    template <typename T>
    T* inout(T* host, size_t count) { return (T*)stage(host, count * sizeof(T), true, true); }
    bool ok() const { return rc_ == TOPAY_OK; }
    // Copies the outputs back, waits for the stream and collects a failed launch; returns the call's status.
    int finish() {
        for (const Buf& b : bufs_)
            if (b.back && rc_ == TOPAY_OK)
                fail(cudaMemcpyAsync(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost, q_), "copy back");
        const cudaError_t e = cudaStreamSynchronize(q_);
        if (rc_ == TOPAY_OK) fail(e, "cudaStreamSynchronize");
        const cudaError_t l = cudaGetLastError();
        if (rc_ == TOPAY_OK) fail(l, "kernel launch");
        return rc_;
    }

  private:
    struct Buf {
        void* dev;
        void* host;
        size_t bytes;
        bool back;
    };
    void* stage(void* host, size_t bytes, bool copy_in, bool back) {
        if (!host || rc_ != TOPAY_OK) return nullptr;
        void* dev = nullptr;
        const cudaError_t e = cudaMallocAsync(&dev, std::max<size_t>(bytes, 1), q_);
        if (e != cudaSuccess) {
            tp_set_error(std::string("cudaMallocAsync failed: ") + cudaGetErrorString(e));
            rc_ = TOPAY_ERR_ALLOC;
            return nullptr;
        }
        bufs_.push_back(Buf{dev, host, bytes, back});
        if (copy_in) fail(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, q_), "copy in");
        return rc_ == TOPAY_OK ? dev : nullptr;
    }
    void fail(cudaError_t e, const char* what) {
        if (e == cudaSuccess || rc_ != TOPAY_OK) return;
        tp_set_error(std::string(what) + ": " + cudaGetErrorString(e));
        rc_ = TOPAY_ERR_CUDA;
    }
    cudaStream_t q_;
    std::vector<Buf> bufs_;
    int rc_ = TOPAY_OK;
};

// Copies `bytes` from the device to the host on `q` and waits for `q`: the host reads `dst` on return.
inline int tp_download(cudaStream_t q, void* dst, const void* src, size_t bytes) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, q);
    if (e == cudaSuccess) e = cudaStreamSynchronize(q);
    if (e != cudaSuccess) {
        tp_set_error(std::string("download: ") + cudaGetErrorString(e));
        return TOPAY_ERR_CUDA;
    }
    return TOPAY_OK;
}

// The device buffers of one long-lived object (dense field, ROG ring, probability map, solver). alloc() gives
// `count` elements (at least one), zeroed on the object's stream; the first failure is kept with its text and later
// allocations do nothing, so a constructor checks status once. Every buffer is freed with the owner.
struct TpDevBuffers {
    cudaStream_t stream = nullptr;
    int status = TOPAY_OK;
    std::vector<void*> ptrs;
    TpDevBuffers() = default;
    TpDevBuffers(const TpDevBuffers&) = delete;
    TpDevBuffers& operator=(const TpDevBuffers&) = delete;
    ~TpDevBuffers() {
        for (void* p : ptrs) cudaFree(p);
    }
    template <typename T>
    int alloc(T** p, size_t count) {
        *p = nullptr;
        if (status != TOPAY_OK) return status;
        const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
        cudaError_t e = cudaMalloc((void**)p, bytes);
        if (e != cudaSuccess) {
            *p = nullptr;
            tp_set_error(std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
            return status = TOPAY_ERR_ALLOC;
        }
        ptrs.push_back(*p);
        if ((e = cudaMemsetAsync(*p, 0, bytes, stream)) != cudaSuccess) {
            tp_set_error(std::string("cudaMemsetAsync: ") + cudaGetErrorString(e));
            return status = TOPAY_ERR_CUDA;
        }
        return TOPAY_OK;
    }
};

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
