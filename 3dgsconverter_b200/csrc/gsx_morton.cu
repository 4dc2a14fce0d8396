// gsx_morton.cu -- Morton ordering as a shared primitive (SURVEY 8(f) item 3) for sm_100a.
//
//   gsx_morton_order   formats/compressed_ply.py:252-297 (_sort_morton_order): 3 x 10-bit Morton code of the position
//                      normalised to the bounding box of the group, argsort, and RECURSION into every run of equal
//                      codes longer than 256 (re-normalised to the run's own box) until the run is small or has no
//                      extent.  Here: level by level over the whole array -- per level the active runs are
//                      compacted, their boxes reduced (warp-aggregated atomics), the keys (run id << 30 | code)
//                      sorted by our stable radix sort, and the next level's runs found by a flag/scan pass.
//                      The reference uses np.argsort's default (unstable) kind: the order of equal codes inside a
//                      finished run is unspecified there; we return the stable one (lowest original index first).
//   gsx_chunk_minmax   compressed_ply.py:206-246 (per-256-splat chunk min/max) and ksplat.py:426-441
//                      (np.minimum/maximum.reduceat over buckets): min and max of `ncol` columns of a row-major
//                      float32 matrix over consecutive chunks of the (optionally permuted) rows.
// Float arithmetic of the codes follows NumPy-2 float32 semantics: (c - min) * (1024.0 / len), clip to [0,1023],
// truncation to uint32.
#include "../../include/gsx.h"
#include "gsx_common.cuh"
#include "gsx_morton.cuh"
#include "gsx_radix.cuh"
#include "gsx_sor.cuh"

#include <algorithm>
#include <vector>

namespace gsx {

#define GSX_FULL 0xffffffffu

__device__ __forceinline__ uint32_t part1by2(uint32_t n) {
    n &= 0x000003ffu;
    n = (n ^ (n << 16)) & 0xff0000ffu;
    n = (n ^ (n << 8)) & 0x0300f00fu;
    n = (n ^ (n << 4)) & 0x030c30c3u;
    n = (n ^ (n << 2)) & 0x09249249u;
    return n;
}

// order-preserving float <-> uint mapping for atomicMin/Max
__device__ __forceinline__ uint32_t f2o(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float o2f(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

// segment of the e-th active element: largest s with seg_off[s] <= e
__device__ __forceinline__ int seg_of(const int* __restrict__ seg_off, int nseg, int64_t e) {
    int lo = 0, hi = nseg - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (seg_off[mid] <= e) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void k_mo_init_bounds(uint32_t* __restrict__ bounds, int nseg) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    for (int a = 0; a < 3; ++a) {
        bounds[6 * s + a] = 0xffffffffu;   // min slots start at +max
        bounds[6 * s + 3 + a] = 0u;        // max slots start at -max
    }
}

// per-run bounding boxes: warp-aggregated when the whole warp sits in one run (the common case)
__global__ void __launch_bounds__(256) k_mo_bounds(const float* __restrict__ xyz, const int32_t* __restrict__ order,
                                                   const int* __restrict__ seg_start, const int* __restrict__ seg_off,
                                                   int nseg, int64_t m, uint32_t* __restrict__ bounds) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = e < m;
    int s = 0;
    float p[3] = {0.f, 0.f, 0.f};
    if (act) {
        s = seg_of(seg_off, nseg, e);
        const int idx = order[seg_start[s] + (int)(e - seg_off[s])];
        p[0] = xyz[3 * (size_t)idx], p[1] = xyz[3 * (size_t)idx + 1], p[2] = xyz[3 * (size_t)idx + 2];
    }
    const int s0 = __shfl_sync(GSX_FULL, s, 0);
    const bool uniform = __all_sync(GSX_FULL, act && s == s0);
    if (uniform) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            float lo = p[a], hi = p[a];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(GSX_FULL, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(GSX_FULL, hi, o));
            }
            if ((threadIdx.x & 31) == 0) {
                atomicMin(bounds + 6 * s + a, f2o(lo));
                atomicMax(bounds + 6 * s + 3 + a, f2o(hi));
            }
        }
    } else if (act) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicMin(bounds + 6 * s + a, f2o(p[a]));
            atomicMax(bounds + 6 * s + 3 + a, f2o(p[a]));
        }
    }
}

// compressed_ply.py:266-283: codes relative to the run's box; key = run id << 30 | code; dead[s] = no extent
__global__ void __launch_bounds__(256) k_mo_keys(const float* __restrict__ xyz, const int32_t* __restrict__ order,
                                                 const int* __restrict__ seg_start, const int* __restrict__ seg_off,
                                                 int nseg, int64_t m, const uint32_t* __restrict__ bounds,
                                                 uint64_t* __restrict__ keys, int32_t* __restrict__ vals,
                                                 int* __restrict__ dead) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int s = seg_of(seg_off, nseg, e);
    const int idx = order[seg_start[s] + (int)(e - seg_off[s])];
    uint32_t q[3];
    bool flat = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float mn = o2f(bounds[6 * s + a]), mx = o2f(bounds[6 * s + 3 + a]);
        const float len = __fsub_rn(mx, mn);
        const float mul = len > 0.f ? __fdiv_rn(1024.0f, len) : 0.f;
        if (len != 0.f) flat = false;
        float v = __fmul_rn(__fsub_rn(xyz[3 * (size_t)idx + a], mn), mul);
        v = fminf(fmaxf(v, 0.f), 1023.f);
        q[a] = (uint32_t)v;
    }
    const uint32_t code = (part1by2(q[2]) << 2) | (part1by2(q[1]) << 1) | part1by2(q[0]);
    keys[e] = ((uint64_t)s << 30) | (uint64_t)code;
    vals[e] = idx;
    if (flat && e == seg_off[s]) dead[s] = 1;
}

__global__ void __launch_bounds__(256) k_mo_writeback(const int32_t* __restrict__ vals, const int* __restrict__ seg_start,
                                                      const int* __restrict__ seg_off, int nseg, int64_t m,
                                                      int32_t* __restrict__ order) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int s = seg_of(seg_off, nseg, e);
    order[seg_start[s] + (int)(e - seg_off[s])] = vals[e];
}

// run starts among the sorted keys (flag = 1 where a new (run id, code) group begins)
__global__ void __launch_bounds__(256) k_mo_flags(const uint64_t* __restrict__ keys, int64_t m,
                                                  uint32_t* __restrict__ flags) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e > m) return;
    flags[e] = e < m ? (uint32_t)(e == 0 || keys[e] != keys[e - 1]) : 0u;   // flags[m] is the scan's total slot
}

__global__ void __launch_bounds__(256) k_mo_starts(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ rank,
                                                   int64_t m, int* __restrict__ starts) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    if (e == 0 || keys[e] != keys[e - 1]) starts[rank[e]] = (int)e;
}

// next level's runs: groups longer than `limit` whose parent run still has extent
__global__ void __launch_bounds__(256) k_mo_pick(const int* __restrict__ starts, int nrun, int64_t m,
                                                 const uint64_t* __restrict__ keys, const int* __restrict__ dead,
                                                 const int* __restrict__ seg_start, const int* __restrict__ seg_off,
                                                 int limit, int* __restrict__ counter, int2* __restrict__ picked) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrun) return;
    const int b = starts[r], e = r + 1 < nrun ? starts[r + 1] : (int)m;
    if (e - b <= limit) return;
    const int s = (int)(keys[b] >> 30);
    if (dead[s]) return;
    const int pos = seg_start[s] + (b - seg_off[s]);
    picked[atomicAdd(counter, 1)] = make_int2(pos, e - b);
}

__global__ void k_mo_iota(int32_t* __restrict__ order, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) order[i] = (int32_t)i;
}

int64_t morton_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    size_t b = 2 * align_up((size_t)n * 8, 256) + 2 * align_up((size_t)n * 4, 256) + radix_ws_bytes(n);
    b += align_up((size_t)(n + 1) * 4, 256) + scan_workspace_bytes(n + 1) + align_up((size_t)n * 4, 256);  // flags, starts
    const size_t maxseg = (size_t)n / 257 + 2;
    b += 4 * align_up(maxseg * 8, 256) + align_up(maxseg * 24, 256) + 4096;
    return (int64_t)b;
}

int morton_order(const float* xyz, int64_t n, int32_t* order, int limit, int max_levels, int* levels_out, void* ws,
                 int64_t ws_bytes, cudaStream_t st) {
    GSX_NVTX("gsx::morton_order");
    GSX_REQUIRE(n >= 0 && n < GSX_N_LIMIT, GSX_ERR_ARG, "morton: n out of range");
    if (levels_out) *levels_out = 0;
    if (n == 0) return GSX_OK;
    GSX_REQUIRE(limit >= 1, GSX_ERR_ARG, "morton: limit must be >= 1");
    GSX_REQUIRE(ws_bytes >= morton_workspace_bytes(n), GSX_ERR_WORKSPACE, "morton: workspace too small");
    Carver c(ws, (size_t)ws_bytes);
    uint64_t* k0 = c.take<uint64_t>((size_t)n);
    uint64_t* k1 = c.take<uint64_t>((size_t)n);
    int32_t* v0 = c.take<int32_t>((size_t)n);
    int32_t* v1 = c.take<int32_t>((size_t)n);
    char* rws = c.take<char>(radix_ws_bytes(n));
    uint32_t* flags = c.take<uint32_t>((size_t)n + 1);
    uint32_t* sws = c.take<uint32_t>(scan_workspace_bytes(n + 1) / 4 + 1);
    int* starts = c.take<int>((size_t)n);
    const size_t maxseg = (size_t)n / 257 + 2;
    int* seg_start = c.take<int>(maxseg);
    int* seg_off = c.take<int>(maxseg + 1);
    int* dead = c.take<int>(maxseg);
    int2* picked = c.take<int2>(maxseg);
    uint32_t* bounds = c.take<uint32_t>(6 * maxseg);
    int* counter = c.take<int>(8);
    GSX_REQUIRE(c.ok(), GSX_ERR_WORKSPACE, "morton: workspace too small");

    k_mo_iota<<<(int)((n + 255) / 256), 256, 0, st>>>(order, n);
    GSX_KERNEL_CHECK();
    if (n == 1) return GSX_OK;
    std::vector<int> h_start{0}, h_len{(int)n};
    int level = 0;
    while (!h_start.empty() && level < max_levels) {
        const int nseg = (int)h_start.size();
        std::vector<int> h_off(nseg + 1, 0);
        for (int s = 0; s < nseg; ++s) h_off[s + 1] = h_off[s] + h_len[s];
        const int64_t m = h_off[nseg];
        GSX_CUDA_CHECK(cudaMemcpyAsync(seg_start, h_start.data(), (size_t)nseg * 4, cudaMemcpyHostToDevice, st));
        GSX_CUDA_CHECK(cudaMemcpyAsync(seg_off, h_off.data(), (size_t)(nseg + 1) * 4, cudaMemcpyHostToDevice, st));
        GSX_CUDA_CHECK(cudaMemsetAsync(dead, 0, (size_t)nseg * 4, st));
        GSX_CUDA_CHECK(cudaMemsetAsync(counter, 0, 32, st));
        GSX_CUDA_CHECK(cudaStreamSynchronize(st));  // the host vectors are reused below
        const int mb = (int)((m + 255) / 256);
        k_mo_init_bounds<<<(nseg + 255) / 256, 256, 0, st>>>(bounds, nseg);
        GSX_KERNEL_CHECK();
        k_mo_bounds<<<mb, 256, 0, st>>>(xyz, order, seg_start, seg_off, nseg, m, bounds);
        GSX_KERNEL_CHECK();
        k_mo_keys<<<mb, 256, 0, st>>>(xyz, order, seg_start, seg_off, nseg, m, bounds, k0, v0, dead);
        GSX_KERNEL_CHECK();
        int seg_bits = 1;
        while ((1ll << seg_bits) < nseg) ++seg_bits;
        uint64_t* ks = nullptr;
        int32_t* vs = nullptr;
        int rc = radix_sort_pairs(k0, k1, v0, v1, m, 0, 30 + (nseg > 1 ? seg_bits : 0), rws, radix_ws_bytes(n), &ks, &vs, st);
        if (rc) return rc;
        k_mo_writeback<<<mb, 256, 0, st>>>(vs, seg_start, seg_off, nseg, m, order);
        GSX_KERNEL_CHECK();
        // runs of equal (run id, code) longer than `limit` become the next level's runs
        k_mo_flags<<<(int)((m + 1 + 255) / 256), 256, 0, st>>>(ks, m, flags);
        GSX_KERNEL_CHECK();
        rc = exclusive_scan_u32_ws(flags, m + 1, sws, st);   // flags[e] -> rank of the group that starts at e
        if (rc) return rc;
        uint32_t nrun = 0;
        GSX_CUDA_CHECK(cudaMemcpyAsync(&nrun, flags + m, 4, cudaMemcpyDeviceToHost, st));
        k_mo_starts<<<mb, 256, 0, st>>>(ks, flags, m, starts);
        GSX_KERNEL_CHECK();
        GSX_CUDA_CHECK(cudaStreamSynchronize(st));
        k_mo_pick<<<(int)((nrun + 255) / 256), 256, 0, st>>>(starts, (int)nrun, m, ks, dead, seg_start, seg_off, limit, counter,
                                                            picked);
        GSX_KERNEL_CHECK();
        int npick = 0;
        GSX_CUDA_CHECK(cudaMemcpyAsync(&npick, counter, 4, cudaMemcpyDeviceToHost, st));
        GSX_CUDA_CHECK(cudaStreamSynchronize(st));
        std::vector<int2> hp((size_t)npick);
        if (npick) {
            GSX_CUDA_CHECK(cudaMemcpyAsync(hp.data(), picked, (size_t)npick * sizeof(int2), cudaMemcpyDeviceToHost, st));
            GSX_CUDA_CHECK(cudaStreamSynchronize(st));
        }
        std::sort(hp.begin(), hp.end(), [](const int2& a, const int2& b) { return a.x < b.x; });  // atomics: any order
        h_start.resize((size_t)npick);
        h_len.resize((size_t)npick);
        for (int i = 0; i < npick; ++i) h_start[i] = hp[i].x, h_len[i] = hp[i].y;
        ++level;
    }
    if (levels_out) *levels_out = level;
    return GSX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// chunk min/max: one block per chunk, `ncol` (<= 8) columns of a row-major [n, F] matrix, rows optionally permuted
__global__ void __launch_bounds__(256) k_chunk_minmax(const float* __restrict__ rows, int F, const int32_t* __restrict__ order,
                                                      int64_t n, int chunk, int ncol, const int* __restrict__ cols,
                                                      float clip_lo, float clip_hi, float* __restrict__ lo_out,
                                                      float* __restrict__ hi_out) {
    const int64_t c0 = (int64_t)blockIdx.x * chunk;
    const int64_t c1 = c0 + chunk < n ? c0 + chunk : n;
    float lo[8], hi[8];
#pragma unroll
    for (int a = 0; a < 8; ++a) lo[a] = INFINITY, hi[a] = -INFINITY;
    for (int64_t j = c0 + threadIdx.x; j < c1; j += blockDim.x) {
        const float* r = rows + (size_t)(order ? order[j] : j) * F;
#pragma unroll
        for (int a = 0; a < 8; ++a)
            if (a < ncol) {
                float v = __ldg(r + cols[a]);
                v = fminf(fmaxf(v, clip_lo), clip_hi);
                lo[a] = fminf(lo[a], v);
                hi[a] = fmaxf(hi[a], v);
            }
    }
    __shared__ float slo[8][8], shi[8][8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(GSX_FULL, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(GSX_FULL, hi[a], o));
        }
        if (lane == 0) slo[a][w] = lo[a], shi[a][w] = hi[a];
    }
    __syncthreads();
    if (threadIdx.x < ncol) {
        float l = slo[threadIdx.x][0], h = shi[threadIdx.x][0];
        for (int k = 1; k < 8; ++k) l = fminf(l, slo[threadIdx.x][k]), h = fmaxf(h, shi[threadIdx.x][k]);
        lo_out[(size_t)blockIdx.x * ncol + threadIdx.x] = l;
        hi_out[(size_t)blockIdx.x * ncol + threadIdx.x] = h;
    }
}

int chunk_minmax(const float* rows, int64_t n, int F, const int32_t* order, int chunk, const int* cols_host, int ncol,
                 float clip_lo, float clip_hi, float* lo_out, float* hi_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
    if (n == 0) return GSX_OK;
    GSX_REQUIRE(ncol >= 1 && ncol <= 8 && chunk >= 1 && F >= 1, GSX_ERR_ARG, "chunk_minmax: bad shape");
    GSX_REQUIRE(ws_bytes >= 64, GSX_ERR_WORKSPACE, "chunk_minmax: needs 64 bytes of scratch");
    for (int a = 0; a < ncol; ++a) GSX_REQUIRE(cols_host[a] >= 0 && cols_host[a] < F, GSX_ERR_ARG, "chunk_minmax: bad column");
    GSX_CUDA_CHECK(cudaMemcpyAsync(ws, cols_host, (size_t)ncol * 4, cudaMemcpyHostToDevice, st));
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    const int64_t nchunk = (n + chunk - 1) / chunk;
    k_chunk_minmax<<<(int)nchunk, 256, 0, st>>>(rows, F, order, n, chunk, ncol, (const int*)ws, clip_lo, clip_hi, lo_out, hi_out);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

}  // namespace gsx
