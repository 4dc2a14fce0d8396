// gsx_compact.cu -- stream compaction of the per-point working set between filters.
//
// Replaces the host-side `vertices[mask]` round trips of the filter chain (data_processor.py:114,149,
// 209,217-224 as driven by converter.py:194-236) for the columns the filters need: xyz (12 B/pt),
// opacity (4 B/pt) and the original row index (4 B/pt).  The 248-byte records stay on the host and
// are gathered ONCE, with the surviving indices, when the caller reads `DataProcessor.data`.
// Stable (order-preserving), like NumPy boolean indexing.  Two forms, A/B in profiles/r02_stream_kernels_probe.json
// (64 M rows, 50 % survivors): count -> multi-level scan -> scatter (0.72 ms) and the shipped single pass with
// decoupled look-back over per-tile survivor counts (k_cmp_onepass, 0.66 ms).  A first single-pass version that staged
// the survivors' DATA in 40 KiB of shared memory per block was slower than both (0.85 ms: occupancy).
#include "../../include/gsx.h"
#include "gsx_common.cuh"
#include "gsx_compact.cuh"
#include "gsx_radix.cuh"

namespace gsx {

#define GSX_FULL 0xffffffffu
constexpr int kCmpBlock = 1024;

__global__ void __launch_bounds__(kCmpBlock) k_cmp_count(const uint8_t* __restrict__ mask, int64_t n,
                                                         uint32_t* __restrict__ counts) {
    int64_t i = (int64_t)blockIdx.x * kCmpBlock + threadIdx.x;
    bool keep = i < n && mask[i] != 0;
    unsigned b = __ballot_sync(GSX_FULL, keep);
    __shared__ uint32_t wc[32];
    if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t v = wc[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GSX_FULL, v, o);
        if (threadIdx.x == 0) counts[blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(kCmpBlock)
    k_cmp_scatter(const uint8_t* __restrict__ mask, int64_t n, const uint32_t* __restrict__ block_off,
                  const float* __restrict__ xyz, const float* __restrict__ opacity, const int32_t* __restrict__ idx,
                  float* __restrict__ xyz_out, float* __restrict__ opacity_out, int32_t* __restrict__ idx_out) {
    int64_t i = (int64_t)blockIdx.x * kCmpBlock + threadIdx.x;
    bool keep = i < n && mask[i] != 0;
    unsigned b = __ballot_sync(GSX_FULL, keep);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __shared__ uint32_t wc[32];
    if (lane == 0) wc[w] = __popc(b);
    __syncthreads();
    if (threadIdx.x < 32) {  // exclusive scan of the 32 warp counts
        uint32_t v = wc[threadIdx.x], x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
            if (lane >= o) x += y;
        }
        wc[threadIdx.x] = x - v;
    }
    __syncthreads();
    if (!keep) return;
    const uint32_t pos = block_off[blockIdx.x] + wc[w] + __popc(b & ((1u << lane) - 1u));
    xyz_out[3 * (size_t)pos] = xyz[3 * i];
    xyz_out[3 * (size_t)pos + 1] = xyz[3 * i + 1];
    xyz_out[3 * (size_t)pos + 2] = xyz[3 * i + 2];
    if (opacity) opacity_out[pos] = opacity[i];
    idx_out[pos] = idx ? idx[i] : (int32_t)i;
}

#ifndef GSX_COMPACT_ONEPASS
#define GSX_COMPACT_ONEPASS 1   // single pass with decoupled look-back; 0 = the count -> scan -> scatter form (A/B)
#endif
// The single pass handles n < GSX_COMPACT_ONEPASS_MAX_N: its look-back words carry the running survivor count in 30
// bits, so from 2^30 rows on (2^30 survivors are possible) the count -> scan -> scatter form runs, whose 32-bit block
// offsets hold any n < 2^31.  A smaller value (a test build) runs that form at small n.
#ifndef GSX_COMPACT_ONEPASS_MAX_N
#define GSX_COMPACT_ONEPASS_MAX_N (1ll << 30)
#endif
static_assert(GSX_COMPACT_ONEPASS_MAX_N >= 1 && GSX_COMPACT_ONEPASS_MAX_N <= (1ll << 30),
              "look-back words hold 30-bit survivor counts");
#if GSX_COMPACT_ONEPASS
constexpr int kOpThreads = 256, kOpPer = 8, kOpTile = kOpThreads * kOpPer;   // 2048 rows per tile
constexpr uint32_t kLbAgg = 1u << 30, kLbInc = 1u << 31, kLbVal = (1u << 30) - 1u;

// tile id from an atomic counter (lower tiles are resident), survivor counts chained by decoupled look-back (one warp
// reads 32 predecessors' count|flag words at a time), the survivors' LOCAL ROW NUMBERS staged in 4 KiB of shared memory,
// then the block copies the surviving rows out in order (gather inside the tile's window, contiguous writes).
__global__ void __launch_bounds__(kOpThreads)
    k_cmp_onepass(const uint8_t* __restrict__ mask, int64_t n, int64_t ntiles, const float* __restrict__ xyz,
                  const float* __restrict__ opacity, const int32_t* __restrict__ idx, float* __restrict__ xyz_out,
                  float* __restrict__ opacity_out, int32_t* __restrict__ idx_out, uint32_t* lookback,
                  unsigned int* tile_counter, uint32_t* __restrict__ total_out) {
    __shared__ uint16_t s_src[kOpTile];
    __shared__ uint32_t s_wsum[8];
    __shared__ unsigned int s_tile;
    __shared__ uint32_t s_excl;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
    __syncthreads();
    const int64_t tile = s_tile;
    const int l0 = threadIdx.x * kOpPer;
    const int64_t i0 = tile * kOpTile + l0;
    unsigned keepbits = 0;
    if (i0 + kOpPer <= n && ((reinterpret_cast<uintptr_t>(mask) + (uintptr_t)i0) & 7) == 0) {
        const uint2 m8 = *reinterpret_cast<const uint2*>(mask + i0);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if ((m8.x >> (8 * e)) & 0xffu) keepbits |= 1u << e;
            if ((m8.y >> (8 * e)) & 0xffu) keepbits |= 1u << (4 + e);
        }
    } else {
#pragma unroll
        for (int e = 0; e < kOpPer; ++e)
            if (i0 + e < n && mask[i0 + e] != 0) keepbits |= 1u << e;
    }
    const uint32_t mine = __popc(keepbits);
    uint32_t x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_wsum[w] = x;
    __syncthreads();
    uint32_t woff = 0, tile_cnt = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t c = s_wsum[k];
        if (k < w) woff += c;
        tile_cnt += c;
    }
    uint32_t lrank = woff + x - mine;
    if (w == 0) {
        volatile uint32_t* lb = lookback;
        if (lane == 0) lb[tile] = tile_cnt | (tile == 0 ? kLbInc : kLbAgg);
        uint32_t excl = 0;
        int64_t t = tile - 1;
        const long long t0 = clock64();
        while (t >= 0) {
            const int64_t id = t - lane;
            uint32_t v = (uint32_t)(1u << 31);   // before the first tile: an inclusive prefix of 0
            if (id >= 0) v = lb[id];
            const unsigned inc = __ballot_sync(GSX_FULL, (v & (1u << 31)) != 0u);
            const unsigned notready = __ballot_sync(GSX_FULL, (v & (3u << 30)) == 0u);
            const int li = inc ? __ffs(inc) - 1 : 31;
            const unsigned need = li == 31 ? 0xffffffffu : ((1u << (li + 1)) - 1u);
            if (notready & need) {
                if (clock64() - t0 > (1ll << 31)) __trap();   // ~1 s: cannot happen (lower tiles are resident)
                continue;
            }
            uint32_t part = lane <= li ? (v & kLbVal) : 0u;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(GSX_FULL, part, o);
            excl += part;
            if (inc) break;
            t -= 32;
        }
        if (lane == 0) {
            if (tile != 0) lb[tile] = (excl + tile_cnt) | kLbInc;
            s_excl = excl;
            if (tile == ntiles - 1) *total_out = excl + tile_cnt;
        }
    }
#pragma unroll
    for (int e = 0; e < kOpPer; ++e)
        if ((keepbits >> e) & 1u) s_src[lrank++] = (uint16_t)(l0 + e);
    __syncthreads();
    const size_t obase = s_excl;
    const int64_t tbase = tile * kOpTile;
    for (uint32_t t = threadIdx.x; t < tile_cnt; t += kOpThreads) {
        const int64_t src = tbase + s_src[t];
        if (opacity) opacity_out[obase + t] = __ldg(opacity + src);
        idx_out[obase + t] = idx ? __ldg(idx + src) : (int32_t)src;
    }
    for (uint32_t t3 = threadIdx.x; t3 < 3 * tile_cnt; t3 += kOpThreads) {
        const uint32_t t = t3 / 3, c = t3 - 3 * t;
        xyz_out[3 * obase + t3] = __ldg(xyz + 3 * (tbase + s_src[t]) + c);
    }
}
#endif

int64_t compact_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    int64_t blocks = (n + kCmpBlock - 1) / kCmpBlock;
    return (int64_t)((size_t)(blocks + 64) * 4 + scan_workspace_bytes(blocks) + 1024);
}

int compact_points(const uint8_t* mask, int64_t n, const float* xyz, const float* opacity, const int32_t* idx,
                   float* xyz_out, float* opacity_out, int32_t* idx_out, int64_t* count_host, void* ws,
                   int64_t ws_bytes, cudaStream_t st) {
    GSX_NVTX("gsx::compact_points");
    GSX_REQUIRE(n >= 0 && n < GSX_N_LIMIT, GSX_ERR_ARG, "compact: n=%lld out of range [0, 2^31-64)", (long long)n);
    if (n == 0) {
        *count_host = 0;
        return GSX_OK;
    }
    GSX_REQUIRE(ws_bytes >= compact_workspace_bytes(n), GSX_ERR_WORKSPACE, "compact: workspace too small");
    GSX_REQUIRE((opacity == nullptr) == (opacity_out == nullptr), GSX_ERR_ARG, "compact: opacity in/out mismatch");
#if GSX_COMPACT_ONEPASS
    if (n < GSX_COMPACT_ONEPASS_MAX_N) {
        const int64_t tiles = (n + kOpTile - 1) / kOpTile;   // (fits the two-pass workspace: fewer tiles than blocks)
        uint32_t* words = (uint32_t*)ws;                      // [0] tile counter, [1] total, [16 ..] look-back words
        GSX_CUDA_CHECK(cudaMemsetAsync(words, 0, (size_t)(tiles + 16) * 4, st));
        k_cmp_onepass<<<(unsigned)tiles, kOpThreads, 0, st>>>(mask, n, tiles, xyz, opacity, idx, xyz_out, opacity_out,
                                                             idx_out, words + 16, words, words + 1);
        GSX_KERNEL_CHECK();
        uint32_t total1 = 0;
        GSX_CUDA_CHECK(cudaMemcpyAsync(&total1, words + 1, 4, cudaMemcpyDeviceToHost, st));
        GSX_CUDA_CHECK(cudaStreamSynchronize(st));
        *count_host = (int64_t)total1;
        return GSX_OK;
    }
#endif
    const int64_t blocks = (n + kCmpBlock - 1) / kCmpBlock;
    uint32_t* counts = (uint32_t*)ws;          // blocks + 1 (total in the extra slot after the scan)
    uint32_t* sws = counts + blocks + 64;
    GSX_CUDA_CHECK(cudaMemsetAsync(counts + blocks, 0, 4, st));
    k_cmp_count<<<(unsigned)blocks, kCmpBlock, 0, st>>>(mask, n, counts);
    GSX_KERNEL_CHECK();
    int rc = exclusive_scan_u32_ws(counts, blocks + 1, sws, st);  // counts[blocks] becomes the total
    if (rc) return rc;
    k_cmp_scatter<<<(unsigned)blocks, kCmpBlock, 0, st>>>(mask, n, counts, xyz, opacity, idx, xyz_out, opacity_out,
                                                          idx_out);
    GSX_KERNEL_CHECK();
    uint32_t total = 0;
    GSX_CUDA_CHECK(cudaMemcpyAsync(&total, counts + blocks, 4, cudaMemcpyDeviceToHost, st));
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    *count_host = (int64_t)total;
    return GSX_OK;
}

}  // namespace gsx
