// The separable exact signed EDT shared by the dense field (field.cu) and the ROG ring (rogfield.cu).
//
// The distance transform is exact and integer: each separable pass computes
// min_v (q - v)^2 + f(v) over a line, which is what the reference's lower-envelope
// routine evaluates (its intermediates are exact integers in double, SURVEY.md A.4), so
// the squared-distance grids are bit-identical; the final `res * sqrt(v)` and the
// sign combine are evaluated with explicit round-to-nearest intrinsics (no FMA
// contraction) so the fp64 grids are bit-identical too.
//
// Pass 1 runs along the contiguous axis from the binary occupancy (warp scans, positive and
// negative transform together, one sign-packed int16 per cell); passes 2/3 run along a strided
// axis on tiles of 16 contiguous cells x the whole line staged in shared memory, each line
// answered by a divide and conquer over its queries (edt_line.cuh); every global access is a
// 64-128 B contiguous segment and a voxel moves 1 + 2 | 2 + 4 | 4 + 8 = 21 B through the passes.
#include <algorithm>
#include <cfloat>
#include <cstdlib>

#include "common_host.h"
#include "edt_line.cuh"

// ------------------------------------------------------------------ kernels

// Pass 1, along the contiguous axis: 1-D distance to the nearest source (pos) and to the nearest
// non-source (neg) cell of each line, sign-packed into one int16 (edt_line.cuh; TP_INF16 = none on this line). One warp
// per line, four consecutive cells per lane (one 4-byte load, one 8-byte store when C % 4 == 0): the index of
// the last source at or before a cell is a running max inside the lane, a warp max-scan across
// lanes and a carry across the 128-cell chunks; the next source at or after it is the mirror image.
// Lines of up to 128 cells (the z axis of the 3-D grid) take a single chunk, everything in
// registers; longer lines (the 2-D maps) make a forward and a backward pass over their chunks.
#define TP_NEG_BIG (-(1 << 28))
#define TP_POS_BIG (1 << 28)

__device__ __forceinline__ int tp_scan_max_excl(int v, int lane) {
    // exclusive max-scan over lower lanes; identity TP_NEG_BIG
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x = max(x, y);
    }
    const int e = __shfl_up_sync(0xffffffffu, x, 1);
    return lane == 0 ? TP_NEG_BIG : e;
}
__device__ __forceinline__ int tp_scan_min_excl_rev(int v, int lane) {
    // exclusive min-scan over higher lanes; identity TP_POS_BIG
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_down_sync(0xffffffffu, x, d);
        if (lane + d < 32) x = min(x, y);
    }
    const int e = __shfl_down_sync(0xffffffffu, x, 1);
    return lane == 31 ? TP_POS_BIG : e;
}

template <bool VEC>
__global__ void __launch_bounds__(256)
k_edt_contig(const int8_t* __restrict__ src, int16_t* __restrict__ out, int64_t n_lines, int C) {
    const int lane = threadIdx.x & 31;
    const int64_t line = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (line >= n_lines) return;
    const int8_t* in = src + line * C;
    int16_t* o = out + line * C;
    const int nchunk = (C + 127) >> 7;
    auto load4 = [&](int c0, bool occ[4]) {
        if (VEC) {
            uchar4 v = make_uchar4(0, 0, 0, 0);
            if (c0 < C) v = *reinterpret_cast<const uchar4*>(in + c0);
            occ[0] = v.x == 1; occ[1] = v.y == 1; occ[2] = v.z == 1; occ[3] = v.w == 1;
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) occ[k] = (c0 + k < C) && in[c0 + k] == 1;
        }
    };
    // forward: last source / last free cell at or before each cell
    int carry_p = TP_NEG_BIG, carry_n = TP_NEG_BIG;
    int fp[4], fn[4];           // kept for the single-chunk case
    for (int ch = 0; ch < nchunk; ch++) {
        const int c0 = (ch << 7) + lane * 4;
        bool occ[4];
        load4(c0, occ);
        int lp = TP_NEG_BIG, ln = TP_NEG_BIG, lastp[4], lastn[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const bool in_line = c0 + k < C;
            if (in_line && occ[k]) lp = c0 + k;
            if (in_line && !occ[k]) ln = c0 + k;
            lastp[k] = lp;
            lastn[k] = ln;
        }
        const int ep = max(tp_scan_max_excl(lp, lane), carry_p);
        const int en = max(tp_scan_max_excl(ln, lane), carry_n);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int c = c0 + k;
            const int a = max(lastp[k], ep), b = max(lastn[k], en);
            fp[k] = a < 0 ? TP_INF16 : min(c - a, TP_INF16);
            fn[k] = b < 0 ? TP_INF16 : min(c - b, TP_INF16);
        }
        carry_p = max(carry_p, __shfl_sync(0xffffffffu, max(lp, ep), 31));
        carry_n = max(carry_n, __shfl_sync(0xffffffffu, max(ln, en), 31));
        if (nchunk > 1) {   // the forward result of the transform the cell is not a source of, sign-packed
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (c0 + k < C) o[c0 + k] = (int16_t)(occ[k] ? -fn[k] : fp[k]);
        }
    }
    // backward: next source / next free cell at or after each cell, min with the forward result
    carry_p = TP_POS_BIG;
    carry_n = TP_POS_BIG;
    for (int ch = nchunk - 1; ch >= 0; ch--) {
        const int c0 = (ch << 7) + lane * 4;
        bool occ[4];
        load4(c0, occ);
        int np_ = TP_POS_BIG, nn_ = TP_POS_BIG, nextp[4], nextn[4];
#pragma unroll
        for (int k = 3; k >= 0; k--) {
            const bool in_line = c0 + k < C;
            if (in_line && occ[k]) np_ = c0 + k;
            if (in_line && !occ[k]) nn_ = c0 + k;
            nextp[k] = np_;
            nextn[k] = nn_;
        }
        const int ep = min(tp_scan_min_excl_rev(np_, lane), carry_p);
        const int en = min(tp_scan_min_excl_rev(nn_, lane), carry_n);
        int16_t res[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int c = c0 + k;
            const int a = min(nextp[k], ep), b = min(nextn[k], en);
            int bp = a >= TP_POS_BIG ? TP_INF16 : min(a - c, TP_INF16);
            int bn = b >= TP_POS_BIG ? TP_INF16 : min(b - c, TP_INF16);
            if (nchunk > 1) {
                if (c < C) {
                    const int f = o[c];
                    if (occ[k]) bn = min(bn, -f);
                    else bp = min(bp, f);
                }
            } else {
                bp = min(bp, fp[k]);
                bn = min(bn, fn[k]);
            }
            res[k] = (int16_t)(occ[k] ? -bn : bp);   // sign-packed (edt_line.cuh)
        }
        carry_p = min(carry_p, __shfl_sync(0xffffffffu, min(np_, ep), 0));
        carry_n = min(carry_n, __shfl_sync(0xffffffffu, min(nn_, en), 0));
        if (VEC) {
            if (c0 < C) *reinterpret_cast<uint2*>(o + c0) = make_uint2((uint16_t)res[0] | ((uint32_t)(uint16_t)res[1] << 16),
                                                                       (uint16_t)res[2] | ((uint32_t)(uint16_t)res[3] << 16));
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (c0 + k < C) o[c0 + k] = res[k];
        }
    }
}

__device__ __forceinline__ void tp_edt_store(bool FINAL, int bp, int bn, size_t idx, double res,
                                             int32_t* __restrict__ out_pos, int32_t* __restrict__ out_neg,
                                             double* __restrict__ esdf, const TpRogSink& rs, int c_line, int c_outer,
                                             int c_inner) {
    if (bp >= TP_INF32) bp = FINAL ? INT32_MAX : TP_INF32;
    if (bn >= TP_INF32) bn = FINAL ? INT32_MAX : TP_INF32;
    if (FINAL) {
        // grid_map.cpp:457, 503, 515-517 — round-to-nearest, no FMA contraction
        // exactly one of the two transforms is non-zero at a cell (it is a source of the other one): one square root
        const bool occ = bn > 0;
        const int x = occ ? bn : bp;
        const double r = __dmul_rn(res, __dsqrt_rn(x == INT32_MAX ? DBL_MAX : (double)x));
        const double dp = occ ? 0.0 : r;        // res * sqrt(0) = +0
        const double dn = occ ? r : 0.0;
        if (rs.enabled) {
            // ROG ring: box coordinates -> ring memory, q > mem_end ? q + id_l - S : q + id_l per axis
            size_t m;
            if (rs.dims3) {
                // last 3-D pass: line axis = x, outer = y, inner = z
                const int qx = c_line + rs.lo[0], qy = c_outer + rs.lo[1], qz = c_inner + rs.lo[2];
                const int mx = qx > rs.mem_end[0] ? qx + rs.idl[0] - rs.size[0] : qx + rs.idl[0];
                const int my = qy > rs.mem_end[1] ? qy + rs.idl[1] - rs.size[1] : qy + rs.idl[1];
                const int mz = qz > rs.mem_end[2] ? qz + rs.idl[2] - rs.size[2] : qz + rs.idl[2];
                m = ((size_t)mx * rs.size[1] + my) * rs.size[2] + mz;
            } else {
                // last 2-D pass: line axis = x, inner = y
                const int qx = c_line + rs.lo[0], qy = c_inner + rs.lo[1];
                const int mx = qx > rs.mem_end[0] ? qx + rs.idl[0] - rs.size[0] : qx + rs.idl[0];
                const int my = qy > rs.mem_end[1] ? qy + rs.idl[1] - rs.size[1] : qy + rs.idl[1];
                m = (size_t)mx * rs.size[1] + my;
            }
            double d = dp;
            if (rs.fuse && dn > 0.0) d = __dadd_rn(d, __dadd_rn(-dn, res));
            rs.dist[m] = d;
            rs.neg[m] = dn;
            return;
        }
        double d = dp;
        if (dn > 0.0) d = __dadd_rn(d, __dadd_rn(-dn, res));
        if (esdf) esdf[idx] = d;
        if (out_pos) {
            out_pos[idx] = bp;
            out_neg[idx] = bn;
        }
    } else {
        out_pos[idx] = bp;
        out_neg[idx] = bn;
    }
}

// Passes 2 and 3 (and the last pass of the 2-D maps), along a strided axis. Block = one outer index x TZ
// contiguous inner cells; the whole line of the tile is staged in shared memory as sign-packed squared distances
// (edt_line.cuh), TZ x 2-4 B contiguous per row on the way in, TZ x 4 B (intermediate) or TZ x 8 B (ESDF) on the
// way out. Thread (x, y): column x of the tile, chunk y (y + TY, ...) of TP_EDT_CHUNK consecutive cells.
//   1. runs of "no source" cells get their skip distances (two walks over the thread's own chunk, the carries of
//      the neighbouring chunks through first / last tables);
//   2. the chunk boundaries are answered against the whole line (window cut-off + skips);
//   3. every thread answers the inside of its chunk by halving between known minimisers — no barrier, the
//      minimisers (int16) of a chunk are private to its thread.
// The negative transform of each cell is the short outward search; both results leave the block the moment they
// are known. The 16 threads of a row write 64 / 128 contiguous bytes.
// IN16: input = pass 1's sign-packed int16 1-D distances, else pass 2's sign-packed int32 squared distances.
template <bool IN16, bool FINAL, int TZ>
__global__ void k_edt_line(const void* __restrict__ in_, int32_t* __restrict__ out32, int32_t* __restrict__ out_pos,
                           int32_t* __restrict__ out_neg, double* __restrict__ esdf, int n_line, size_t line_stride,
                           size_t outer_stride, int n_inner, int tiles, int CH, double res,
                           const __grid_constant__ TpRogSink sink) {
    extern __shared__ __align__(16) int sm_i[];
    const int TY = blockDim.y, tx = threadIdx.x, ty = threadIdx.y;
    const int nseg = (n_line + CH - 1) / CH, nb = tp_edt_boundaries(n_line, CH);
    int* s_f = sm_i;                                                        // [n_line][TZ]
    short* s_arg = reinterpret_cast<short*>(s_f + n_line * TZ);     // [n_line][TZ]
    short* s_first = s_arg + n_line * TZ;                           // [nseg][TZ]
    short* s_last = s_first + nseg * TZ;                            // [nseg][TZ]
    const int outer = blockIdx.x / tiles, tile = blockIdx.x % tiles;
    const int c = tile * TZ + tx;
    const bool cvalid = c < n_inner;
    const size_t base = (size_t)outer * outer_stride + c;
    for (int l = ty; l < n_line; l += TY) {
        int v = TP_INF32;
        if (cvalid) {
            const size_t idx = base + (size_t)l * line_stride;
            v = IN16 ? tp_sq16(static_cast<const int16_t*>(in_)[idx]) : static_cast<const int32_t*>(in_)[idx];
        }
        s_f[l * TZ + tx] = v;
    }
    __syncthreads();
    int* col = s_f + tx;
    // 1. skip distances of the "no source" runs
    uint32_t has_run = 0u;      // bit i: the i-th chunk of this thread holds a "no source" cell
    if (cvalid) {
        int it = 0;
        for (int sg = ty; sg < nseg; sg += TY, it++) {
            const int v0 = sg * CH, v1 = min(v0 + CH, n_line);
            int first = -1, last = -1, cnt = 0;
            for (int v = v0; v < v1; v++)
                if (col[v * TZ] < TP_INF32) {
                    if (first < 0) first = v;
                    last = v;
                    cnt++;
                }
            s_first[sg * TZ + tx] = (short)first;
            s_last[sg * TZ + tx] = (short)last;
            if (cnt != v1 - v0 || it >= 32) has_run |= 1u << (it & 31);
        }
    }
    __syncthreads();
    if (cvalid && has_run != 0u) {
        int it = 0;
        for (int sg = ty; sg < nseg; sg += TY, it++) {
            if (!((has_run >> (it & 31)) & 1u)) continue;
            const int v0 = sg * CH, v1 = min(v0 + CH, n_line);
            int lastc = -1, nextc = n_line;     // nearest cell with a value before / after the chunk
            for (int k = sg - 1; k >= 0 && lastc < 0; k--) lastc = s_last[k * TZ + tx];
            for (int k = sg + 1; k < nseg && nextc >= n_line; k++) {
                const int fk = s_first[k * TZ + tx];
                if (fk >= 0) nextc = fk;
            }
            for (int v = v1 - 1; v >= v0; v--) {
                if (col[v * TZ] < TP_INF32) nextc = v;
                else col[v * TZ] = tp_skip_make(0, nextc - v);
            }
            for (int v = v0; v < v1; v++) {
                const int fv = col[v * TZ];
                if (fv < TP_INF32) lastc = v;
                else col[v * TZ] = fv | ((v - lastc) << TP_SKIP_BITS);
            }
        }
    }
    __syncthreads();
    auto emit = [&](int l, int bp) {
        const int bn = tp_neg_search<TZ>(col, n_line, l);
        const size_t idx = base + (size_t)l * line_stride;
        if (FINAL) {
            tp_edt_store(true, bp, bn, idx, res, out_pos, out_neg, esdf, sink, l, outer, c);
        } else {
            // exactly one of the two is non-zero (the cell is a source of the other transform)
            out32[idx] = bn > 0 ? -(bn >= TP_INF32 ? TP_INF32 : bn) : (bp >= TP_INF32 ? TP_INF32 : bp);
        }
    };
    // 2. chunk boundaries, each against the whole line
    if (cvalid)
        for (int b = ty; b < nb; b += TY) {
            const int q = tp_edt_boundary(b, n_line, CH);
            int arg;
            const int bp = tp_dc_query<TZ>(col, q, 0, n_line - 1, arg);
            s_arg[q * TZ + tx] = (short)arg;
            emit(q, bp);
        }
    __syncthreads();
    // 3. the inside of the chunks, one thread per chunk
    if (cvalid)
        for (int ch = ty; ch < nb - 1; ch += TY) {
            const int lo = tp_edt_boundary(ch, n_line, CH), hi = tp_edt_boundary(ch + 1, n_line, CH);
            for (int h = tp_dc_top(hi - lo) >> 1; h >= 1; h >>= 1)
                for (int q = lo + h; q < hi; q += 2 * h) {
                    const int qr = q + h < hi ? q + h : hi;
                    const int a_lo = s_arg[(q - h) * TZ + tx], a_hi = s_arg[qr * TZ + tx];
                    int arg;
                    const int bp = tp_dc_query<TZ>(col, q, a_lo, a_hi, arg);
                    s_arg[q * TZ + tx] = (short)arg;
                    emit(q, bp);
                }
        }
}

// Pass 1 on large grids with short contiguous lines (the z axis of the 3-D grid: C = 16 NV <= 128 cells): one THREAD
// per line — 16-byte loads of the occupancy, folded into a 128-bit occupancy mask; the nearest cell of the other kind
// before a cell is a running index, the nearest one after it a find-first-set on the shifted mask; 16-byte stores of
// the sign-packed int16 distances. A warp per line (k_edt_contig) spends two 5-step warp scans on an 80-cell line.
template <int NV>
__global__ void __launch_bounds__(128)
k_edt_contig_thread(const int8_t* __restrict__ src, int16_t* __restrict__ out, int64_t n_lines) {
    constexpr int C = 16 * NV;
    const int64_t line = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= n_lines) return;
    const uint4* in = reinterpret_cast<const uint4*>(src + line * C);
    unsigned long long occ_lo = 0ull, occ_hi = 0ull;
#pragma unroll
    for (int k = 0; k < NV; k++) {
        const uint4 v = in[k];
        const uint32_t ww[4] = {v.x, v.y, v.z, v.w};
        unsigned long long bits = 0ull;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            // byte == 1 -> 0xff (per-byte compare), its top bits gathered into a nibble
            const uint32_t eq = __vcmpeq4(ww[j], 0x01010101u) & 0x80808080u;
            bits |= (unsigned long long)((eq * 0x00204081u) >> 28) << (4 * j);
        }
        if (k < 4) occ_lo |= bits << (16 * k);
        else occ_hi |= bits << (16 * (k - 4));
    }
    constexpr unsigned long long V_LO = C >= 64 ? ~0ull : (1ull << (C & 63)) - 1ull;
    constexpr unsigned long long V_HI = C <= 64 ? 0ull : (C >= 128 ? ~0ull : (1ull << ((C - 64) & 63)) - 1ull);
    const unsigned long long free_lo = ~occ_lo & V_LO, free_hi = ~occ_hi & V_HI;
    uint4* dst = reinterpret_cast<uint4*>(out + line * C);
    int lastp = -2 * TP_INF16, lastn = -2 * TP_INF16;
    uint32_t o[4];
#pragma unroll
    for (int c = 0; c < C; c++) {
        const bool occ = c < 64 ? (occ_lo >> c) & 1ull : (occ_hi >> (c - 64)) & 1ull;
        if (occ) lastp = c; else lastn = c;
        // the other kind: free cells for an occupied cell, occupied ones for a free cell
        const unsigned long long lo = occ ? free_lo : occ_lo, hi = occ ? free_hi : occ_hi;
        int nxt = 2 * TP_INF16 + C;
        if (c < 64) {
            const unsigned long long x = lo >> c;
            if (x) nxt = c + __ffsll((long long)x) - 1;
            else if (C > 64 && hi) nxt = 64 + __ffsll((long long)hi) - 1;
        } else {
            const unsigned long long x = hi >> (c - 64);
            if (x) nxt = c + __ffsll((long long)x) - 1;
        }
        const int m = min(min(c - (occ ? lastn : lastp), nxt - c), TP_INF16);
        const uint32_t v = (uint32_t)(uint16_t)(int16_t)(occ ? -m : m);      // sign-packed (edt_line.cuh)
        if (c & 1) o[(c >> 1) & 3] |= v << 16; else o[(c >> 1) & 3] = v;
        if ((c & 7) == 7) dst[c >> 3] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// Passes 2 and 3 on large grids: the reference's own O(n) lower-envelope sweep in its integer two-scan form
// (edt_line.cuh, tp_env_*), NS threads per line. Block = 32 adjacent lines (lanes = consecutive inner cells, so every
// global access of a warp is one contiguous 64-256 B segment) x NS warps; warp j owns the sources of segment j of the
// line (L = ceil(n / NS) rounded up to 32 cells).
//   1. each thread builds the envelope of ITS segment's sources over the whole line (forward scan of L cells, input
//      fetched 16 cells ahead of the stack work; the stack is a per-thread local array of L entries, lane-interleaved by
//      the hardware) and records the segment's occupancy bits in shared memory;
//   2. the line is swept from its far end in chunks of 32 cells: every thread reads its envelope off at the chunk's
//      cells into shared memory, then the block's threads share the chunk's 32 x 32 outputs: minimum over the NS
//      envelopes = the positive transform of a free cell; an occupied cell takes the short outward search of the
//      negative transform instead (its sources, the free cells, are dense). Results leave the block at once.
// One thread per line would do with a fifth of the instructions per cell of the divide and conquer (k_edt_line), but an
// 800-cell line is then a 50 k-instruction dependency chain on 14 warps per SM; NS = 4 cuts the chain to a third and
// quadruples the warps.
__device__ __forceinline__ void tp_touch(const void* p) {
    unsigned a, b;
    asm volatile("ld.v2.u32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
}

template <bool IN16, bool FINAL, int NS, int MAXSEG>
__global__ void __launch_bounds__(32 * NS)
k_edt_scan(const void* __restrict__ in_, int32_t* __restrict__ out32, int32_t* __restrict__ out_pos,
           int32_t* __restrict__ out_neg, double* __restrict__ esdf, int n_line, int L, size_t line_stride,
           size_t outer_stride, int n_inner, int64_t n_lines, double res, const __grid_constant__ TpRogSink sink) {
    extern __shared__ __align__(16) int sm_scan[];
    const int lane = threadIdx.x, j = threadIdx.y;
    const int nw = (n_line + 31) >> 5;
    int* s_val = sm_scan;                                              // [NS][32 cells][32 lanes]
    unsigned* s_occ = reinterpret_cast<unsigned*>(sm_scan + NS * 1024);   // [nw][32 lanes]
    int64_t t = (int64_t)blockIdx.x * 32 + lane;
    const bool valid = t < n_lines;
    if (!valid) t = n_lines - 1;        // a lane beyond the grid repeats the last line and writes nothing
    const int outer = (int)(t / n_inner), c = (int)(t % n_inner);
    const size_t base = (size_t)outer * outer_stride + c;
    TpEnvEntry stk[MAXSEG];
    // raw cell of the line, index clamped (no predicate on the load: the fetches of a chunk issue back to back and are
    // converted only when the scan reaches them)
    auto raw = [&](int u) -> int {
        const size_t idx = base + (size_t)min(max(u, 0), n_line - 1) * line_stride;
        return IN16 ? (int)static_cast<const int16_t*>(in_)[idx] : static_cast<const int32_t*>(in_)[idx];
    };
    auto cvt = [&](int r) -> int { return IN16 ? tp_sq16(r) : r; };
    constexpr int PF = 16;
    // ---- 1. envelope of the segment's sources
    const int s0 = j * L, s1 = min(s0 + L, n_line);
    TpEnv e{-1, 0, 0, 0};
    if (s0 < s1) {
        int nx[PF], nn[PF];
        int prev = s0 > 0 ? tp_env_val<false>(cvt(raw(s0 - 1))) : 1;
#pragma unroll
        for (int k = 0; k < PF; k++) nx[k] = raw(s0 + k);
        int cur_raw = cvt(nx[0]);
        unsigned bits = 0u;
        for (int u0 = s0; u0 < s1; u0 += PF) {
#pragma unroll
            for (int k = 0; k < PF; k++) nn[k] = raw(u0 + PF + k);
#pragma unroll
            for (int k = 0; k < PF; k++) {
                const int u = u0 + k;
                if (u < s1) {
                    bits |= (cur_raw < 0 ? 1u : 0u) << (u & 31);
                    const int next_raw = cvt(k + 1 < PF ? nx[k + 1] : nn[0]);
                    const int nxt = u + 1 < n_line ? tp_env_val<false>(next_raw) : 1;
                    const int cur = tp_env_val<false>(cur_raw);
                    tp_env_push(e, stk, n_line, u, cur, prev, nxt);
                    prev = cur;
                    cur_raw = next_raw;
                }
            }
            if (((u0 + PF) & 31) == 0 || u0 + PF >= s1) {
                s_occ[(u0 >> 5) * 32 + lane] = bits;
                bits = 0u;
            }
#pragma unroll
            for (int k = 0; k < PF; k++) nx[k] = nn[k];
        }
    }
#pragma unroll
    for (int k = 1; k <= 8; k++) tp_touch(&stk[max(e.q - k, 0)]);
    __syncthreads();
    // ---- 2. sweep from the far end, 32 cells at a time
    const double r_inf = __dmul_rn(res, __dsqrt_rn(DBL_MAX));      // "no obstacle anywhere" (fillESDF's DBL_MAX)
    if (e.q < 0) {          // no source in the segment: a sentinel entry that never pops and never wins
        e.sv = 0;
        e.gv = TP_INF32;
        e.tv = -1;
    }
    for (int ub = (nw - 1) << 5; ub >= 0; ub -= 32) {
        int* sv_out = s_val + (j * 32 + 31) * 32 + lane;
#pragma unroll 8
        for (int u = ub + 31; u >= ub; u--, sv_out -= 32) {
            const int d = u - e.sv;
            *sv_out = d * d + e.gv;         // < 2^28 + 2^29; cells past the line's end are never read
            if (u == e.tv && e.q > 0) {     // the bottom entry (t = 0) stays
                e.q--;
                tp_env_load(e, stk);
                tp_touch(&stk[max(e.q - 8, 0)]);
            }
        }
        __syncthreads();
        const unsigned occ = s_occ[(ub >> 5) * 32 + lane];
        for (int k = j; k < 32; k += NS) {
            const int u = ub + k;
            if (u >= n_line || !valid) continue;
            int bp = s_val[k * 32 + lane], bn = 0;
#pragma unroll
            for (int jj = 1; jj < NS; jj++) bp = min(bp, s_val[(jj * 32 + k) * 32 + lane]);
            bp = min(bp, TP_INF32);
            if ((occ >> k) & 1u) {
                // negative transform: outward search, nearest cells first, ended by the window cut-off d^2 >= best
                bp = 0;
                bn = tp_env_val<true>(cvt(raw(u)));
                for (int d = 1; d < n_line; d++) {
                    const int dd = d * d;
                    if (dd >= bn) break;
                    if (u - d >= 0) bn = min(bn, dd + tp_env_val<true>(cvt(raw(u - d))));
                    if (u + d < n_line) bn = min(bn, dd + tp_env_val<true>(cvt(raw(u + d))));
                }
            }
            const size_t idx = base + (size_t)u * line_stride;
            if (!FINAL) {
                out32[idx] = bn > 0 ? -bn : bp;
            } else if (sink.enabled) {
                tp_edt_store(true, bp, bn, idx, res, out_pos, out_neg, esdf, sink, u, outer, c);
            } else {
                // the dense field's store (tp_edt_store without the ring sink): one square root per cell, rounded
                // products and sums (grid_map.cpp:457, 503, 515-517)
                const bool oc = bn > 0;
                const int x = oc ? bn : bp;
                const double r = x >= TP_INF32 ? r_inf : __dmul_rn(res, __dsqrt_rn((double)x));
                if (esdf) esdf[idx] = oc ? __dadd_rn(-r, res) : r;
                if (out_pos) {
                    out_pos[idx] = bp >= TP_INF32 ? INT32_MAX : bp;
                    out_neg[idx] = bn >= TP_INF32 ? INT32_MAX : bn;
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ host

namespace {

// A strided pass reads pass 1's int16 output and either ends the transform (2-D) or feeds pass 3 (3-D), or it is the
// 3-D pass 3 over pass 2's int32 output.
enum TpStridedPass { TP_PASS_2D, TP_PASS_2_OF_3D, TP_PASS_3_OF_3D };

using ContigThreadKernel = decltype(&k_edt_contig_thread<1>);
using ScanKernel = decltype(&k_edt_scan<true, true, 4, 256>);
using LineKernel = decltype(&k_edt_line<true, true, 16>);

// k_edt_contig_thread<NV> for lines of 16 NV cells, NV = 1..8
const ContigThreadKernel k_contig_thread_of[8] = {
    k_edt_contig_thread<1>, k_edt_contig_thread<2>, k_edt_contig_thread<3>, k_edt_contig_thread<4>,
    k_edt_contig_thread<5>, k_edt_contig_thread<6>, k_edt_contig_thread<7>, k_edt_contig_thread<8>};
// [pass]
const ScanKernel k_scan_of[3] = {k_edt_scan<true, true, 4, 256>, k_edt_scan<true, false, 4, 256>,
                                 k_edt_scan<false, true, 4, 256>};
// [pass][tile width 16, 8, 4]
const LineKernel k_line_of[3][3] = {
    {k_edt_line<true, true, 16>, k_edt_line<true, true, 8>, k_edt_line<true, true, 4>},
    {k_edt_line<true, false, 16>, k_edt_line<true, false, 8>, k_edt_line<true, false, 4>},
    {k_edt_line<false, true, 16>, k_edt_line<false, true, 8>, k_edt_line<false, true, 4>}};

// One strided pass over n_outer x n_inner lines of n_line cells. scan_mode: TOPAY_EDT_SCAN (-1 = by grid size).
int strided_pass(const TpEdtScratch& s, TpStridedPass pass, int scan_mode, int n_line, size_t line_stride,
                 int n_outer, size_t outer_stride, int n_inner, double* esdf, int32_t* sqp, int32_t* sqn) {
    cudaStream_t q = s.stream;
    const bool in16 = pass != TP_PASS_3_OF_3D, fin = pass != TP_PASS_2_OF_3D;
    const void* in = in16 ? (const void*)s.packed16 : (const void*)s.packed32;
    int32_t* out32 = fin ? nullptr : s.packed32;
    int32_t* op = fin && s.keep_sq ? sqp : nullptr;
    int32_t* on = fin && s.keep_sq ? sqn : nullptr;
    if (!fin) esdf = nullptr;
    const int64_t nl = (int64_t)n_outer * n_inner;
    // Measured on 800 x 800 x 80 (B200): pass 3 (every cell of a line carries a value) 0.84 ms by the envelope scan
    // against 1.07 ms by the divide and conquer; pass 2 (values only under obstacles) 0.61 against 0.46 ms.
    if (n_line <= 1024 && (scan_mode >= 0 ? scan_mode != 0 : (!in16 && nl >= 16384))) {
        constexpr int NS = 4;                                       // segment threads per line
        const int L = (((n_line + NS - 1) / NS) + 31) & ~31;       // <= 256
        const unsigned blocks = (unsigned)((nl + 31) / 32);
        const size_t smem = (size_t)NS * 1024 * 4 + (size_t)((n_line + 31) / 32) * 32 * 4;
        k_scan_of[pass]<<<blocks, dim3(32, NS), smem, q>>>(in, out32, op, on, esdf, n_line, L, line_stride,
                                                          outer_stride, n_inner, nl, s.res, s.sink);
        return TOPAY_OK;
    }
    // Chunk length: 32 queries per thread on large grids; small grids (the 2-D maps, the default 200 x 200 x 16
    // field) take shorter chunks so that the chunk threads of the whole grid still fill the machine.
    int CH = 32;
    while (CH > 4 && (long long)n_outer * n_inner * ((n_line + CH - 1) / CH) < 148 * 1024) CH >>= 1;
    // staged line (int32) + the minimisers (int16) + first / last tables of the chunks (int16)
    const int nseg = (n_line + CH - 1) / CH, nb = tp_edt_boundaries(n_line, CH);
    auto smem_of = [&](int tz) -> size_t {
        return (size_t)n_line * tz * 4 + (size_t)n_line * tz * 2 + (size_t)2 * nseg * tz * 2 + 16;
    };
    // Tile width: 16 cells (64 B rows in, 128 B rows of ESDF out) while at least two blocks fit an SM
    int TZ = 16;
    while (TZ > 4 && smem_of(TZ) > (size_t)100 * 1024) TZ >>= 1;
    // small grids: narrower tiles so that the blocks cover all SMs
    while (TZ > 4 && (long long)n_outer * ((n_inner + TZ - 1) / TZ) < 296) TZ >>= 1;
    const size_t smem = smem_of(TZ);
    if (smem > 200 * 1024) {
        tp_set_error("grid line too long for the strided-pass staging buffer");
        return TOPAY_ERR_TOO_LARGE;
    }
    int TY = std::max(1, std::min(1024 / TZ, nb));    // one thread per chunk boundary
    while ((TZ * TY) % 32 != 0 && TY < 1024 / TZ) TY++;     // whole warps
    const int tiles = (n_inner + TZ - 1) / TZ;
    const LineKernel kern = k_line_of[pass][TZ == 16 ? 0 : (TZ == 8 ? 1 : 2)];
    TP_CUDA_OK(tp_grow_dyn_smem((const void*)kern, smem), {});
    kern<<<(unsigned)n_outer * tiles, dim3(TZ, TY), smem, q>>>(in, out32, op, on, esdf, n_line, line_stride,
                                                               outer_stride, n_inner, tiles, CH, s.res, s.sink);
    return TOPAY_OK;
}

}  // namespace

// One signed transform over a [A][B][C] array (C contiguous): pass 1 along C, pass 2 along B and, when A > 1, pass 3
// along A. The last pass writes `esdf` (+ the integer grids when keep_sq is set). esdf may be NULL (integer grids
// only, keep_sq must then be set).
int tp_signed_edt(const TpEdtScratch& s, const int8_t* src, int A, int B, int C, double* esdf, int32_t* sqp,
                  int32_t* sqn) {
    cudaStream_t q = s.stream;
    const int64_t n_lines = (int64_t)A * B;
    // Large grids take the thread-per-line kernels (k_edt_contig_thread, k_edt_scan): their lines alone fill the
    // machine. Small ones (the 2-D maps, the default 200 x 200 x 16 field) keep the kernels that parallelise inside a
    // line. Both are exact, so the choice never shows in the result. TOPAY_EDT_SCAN = 0 / 1 forces it (tests).
    const char* env_scan = getenv("TOPAY_EDT_SCAN");
    const int scan_mode = env_scan ? atoi(env_scan) : -1;
    // pass 1
    if (C % 16 == 0 && C <= 128 && (scan_mode >= 0 ? scan_mode != 0 : n_lines >= 16384)) {
        k_contig_thread_of[C / 16 - 1]<<<(unsigned)((n_lines + 127) / 128), 128, 0, q>>>(src, s.packed16, n_lines);
    } else {
        const int wpb = 8;
        const unsigned blocks = (unsigned)((n_lines + wpb - 1) / wpb);
        if (C % 4 == 0)
            k_edt_contig<true><<<blocks, wpb * 32, 0, q>>>(src, s.packed16, n_lines, C);
        else
            k_edt_contig<false><<<blocks, wpb * 32, 0, q>>>(src, s.packed16, n_lines, C);
    }
    if (A == 1) return strided_pass(s, TP_PASS_2D, scan_mode, B, (size_t)C, 1, 0, C, esdf, sqp, sqn);
    const int rc = strided_pass(s, TP_PASS_2_OF_3D, scan_mode, B, (size_t)C, A, (size_t)B * C, C, esdf, sqp, sqn);
    if (rc != TOPAY_OK) return rc;
    return strided_pass(s, TP_PASS_3_OF_3D, scan_mode, A, (size_t)B * C, B, (size_t)C, C, esdf, sqp, sqn);
}
