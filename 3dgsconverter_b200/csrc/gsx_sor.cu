// gsx_sor.cu -- Statistical Outlier Removal, Taichi semantics, for sm_100a.
//
// Replaces /root/reference/gsconverter/processing/gpu_ops.py:193-263 (host driver
// filter_sor_gpu) and :98-176 (Taichi kernel sor_compute_mean_dists).  Normative
// arithmetic: SURVEY.md Appendix A.1.
//
// Design (B200-first, not a translation of the Taichi kernel):
//   * grid build entirely on device: min/max reduce -> 64-bit key (bucket hash << 15 |
//     5+5+5-bit Morton code of the position inside the cell) -> radix sort -> float4
//     gather (w carries the original index, so the "unsort" is fused into the query
//     kernel) -> {start,end} bucket table -> bounding boxes of every aligned run of 32
//     ("chunk") and 1024 ("super") sorted points.
//   * query kernel: one warp per query, persistent CTAs with a dynamic batch counter.
//     Lane p<27 evaluates probe p's hash and loads its bucket entry ({start,end}, and the 32-byte box if non-empty);
//     the probes are visited nearest box first (redux.min on the lower bound) and dropped once
//     lb >= tau; candidates are streamed 32 at a time with one coalesced float4 load per lane;
//     the K best d^2 live one per lane in a register (two for K>32) and are maintained with
//     ballot + shfl insertion or a bitonic merge.
//   * EXACT pruning: the reference's result only depends on the multiset of the K
//     smallest distances among the probed buckets' contents (A.1 step 7).  A chunk whose
//     box lower bound -- evaluated with the same monotone float32 op sequence as d^2 --
//     is >= the current K-th best can never contribute, so it is skipped.  Big buckets
//     (the clustered part of the cloud, where the reference visits 10^4..10^5 candidates
//     per point) are walked super -> chunk -> points, nearest box first (redux.min).
//     Selection is done on d^2 and sqrt is taken of the K winners only (sqrt is
//     monotone, so the K smallest d are the sqrt of the K smallest d^2).
//   * reference quirks kept on purpose: hash buckets (not cells), a bucket reached by two
//     probes is scanned twice, int32-wrapping probe hash (GSX_HASH_I32WRAP), self/duplicate
//     skip by d^2 > 1e-12, K capped at 50, 1e10 "empty" sentinel and the < 0.9e10 validity
//     test, mean = 0 when no candidate was found.
#include "gsx_common.cuh"
#include "gsx_sor.cuh"

#include "gsx_radix.cuh"
#include <math.h>

namespace gsx {

// smallest float32 whose sqrt is >= 1e10f: d is inserted by the reference iff sqrt(d2) < 1e10f
#define GSX_D2LIM_BITS 0x60ad78ebu
#define GSX_FULL 0xffffffffu

#ifndef GSX_MORTON_BITS
#define GSX_MORTON_BITS 15
#endif
constexpr int kMortonBits = GSX_MORTON_BITS;       // in-cell Morton code: kMortonBits/3 bits per axis
constexpr float kMortonScale = (float)(1 << (GSX_MORTON_BITS / 3));
constexpr float kMortonMax = kMortonScale - 1.f;
#ifndef GSX_SMALL_BUCKET
#define GSX_SMALL_BUCKET 64
#endif
constexpr int kSmallBucket = GSX_SMALL_BUCKET;  // buckets up to this size are scanned without box tests
#ifndef GSX_QUERY_BATCH
#define GSX_QUERY_BATCH 16
#endif
constexpr int kQueryBatch = GSX_QUERY_BATCH;   // consecutive queries grabbed per warp

// ------------------------------------------------------------------ workspace layout

SorWs sor_carve(void* ws, int64_t ws_bytes, int64_t n, size_t sort_ws_bytes) {
    // The GRID part (what the query kernel reads) comes first, so a blob of gsx_sor_grid_workspace_bytes(n) is a
    // valid workspace for build_from_sorted / mean_dists; the sort buffers (keys, values, radix scratch) follow.
    SorWs w;
    Carver c(ws, (size_t)ws_bytes);
    int64_t nchunk = (n + 31) / 32, nsuper = (nchunk + 31) / 32;
    w.n = n;
    w.spos = c.take<float4>(n);
    w.tab_se = c.take<int2>(n);
    w.tab_box = c.take<float4>(2 * n);
    w.startbits = c.take<uint32_t>(nchunk);
    w.cellbits = c.take<uint32_t>(nchunk);
    w.bigbits = c.take<uint32_t>(nchunk);
    w.startlist = c.take<uint32_t>(n / 8 + 1024);
    w.caabb = c.take<float4>(2 * nchunk);
    w.saabb = c.take<float4>(2 * nsuper);
    w.partial = c.take<float>(6 * 1024);
    w.minmax = c.take<float>(8);
    w.counters = c.take<unsigned int>(64);
    w.stats = c.take<unsigned long long>(8);
    w.meanstd = c.take<float>(8);
    w.ms_bytes = mean_std_ws_bytes(n);
    w.ms_ws = c.take<char>(w.ms_bytes);
    w.grid_total = align_up(c.off, 256);
    w.keys0 = c.take<uint64_t>(n);
    w.keys1 = c.take<uint64_t>(n);
    w.sort_ws_bytes = sort_ws_bytes;
    w.sort_ws = c.take<char>(sort_ws_bytes);
    w.total = align_up(c.off, 256);
    w.ok = c.ok();
    w.grid_ok = w.grid_total <= (size_t)(ws_bytes > 0 ? ws_bytes : 0);
    return w;
}

size_t sor_sort_ws_bytes(int64_t n) { return radix_ws_bytes(n) + 256; }  // scratch of the pair sort

int64_t sor_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    SorWs w = sor_carve(nullptr, 0, n, sor_sort_ws_bytes(n));
    return (int64_t)w.total + 1024;
}

int64_t sor_grid_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    SorWs w = sor_carve(nullptr, 0, n, sor_sort_ws_bytes(n));
    return (int64_t)w.grid_total;
}

// ------------------------------------------------------------------ min / max

__global__ void __launch_bounds__(256) k_minmax_partial(const float* __restrict__ xyz, int64_t n,
                                                        float* __restrict__ partial) {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            float v = xyz[3 * i + a];
            lo[a] = fminf(lo[a], v);
            hi[a] = fmaxf(hi[a], v);
        }
    }
    __shared__ float sm[6][8];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(GSX_FULL, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(GSX_FULL, hi[a], o));
        }
        if (lane_id() == 0) {
            sm[a][threadIdx.x >> 5] = lo[a];
            sm[3 + a][threadIdx.x >> 5] = hi[a];
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float r = sm[threadIdx.x][0];
        for (int w = 1; w < 8; ++w) r = threadIdx.x < 3 ? fminf(r, sm[threadIdx.x][w]) : fmaxf(r, sm[threadIdx.x][w]);
        partial[blockIdx.x * 6 + threadIdx.x] = r;
    }
}

__global__ void k_minmax_final(const float* __restrict__ partial, int nblocks, float* __restrict__ out) {
    // 6 warps, warp a reduces component a over the block partials
    const int a = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (a >= 6) return;
    float r = a < 3 ? INFINITY : -INFINITY;
    for (int b = lane; b < nblocks; b += 32) r = a < 3 ? fminf(r, partial[b * 6 + a]) : fmaxf(r, partial[b * 6 + a]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float t = __shfl_xor_sync(GSX_FULL, r, o);
        r = a < 3 ? fminf(r, t) : fmaxf(r, t);
    }
    if (lane == 0) out[a] = r;
}

int sor_minmax(const float* xyz, int64_t n, float* minmax_dev, float* partial, cudaStream_t st) {
    int blocks = (int)((n + 255) / 256);
    int cap = sm_count() * 4;
    if (blocks > cap) blocks = cap;
    if (blocks > 1024) blocks = 1024;
    if (blocks < 1) blocks = 1;
    k_minmax_partial<<<blocks, 256, 0, st>>>(xyz, n, partial);
    GSX_KERNEL_CHECK();
    k_minmax_final<<<1, 192, 0, st>>>(partial, blocks, minmax_dev);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

// ------------------------------------------------------------------ keys

__device__ __forceinline__ uint32_t spread6(uint32_t v) {  // 6 bits -> every third bit
    v &= 63u;
    v = (v | (v << 8)) & 0x0000300Fu;   // ..xx........xxxx
    v = (v | (v << 4)) & 0x000030C3u;   // ..xx....xx....xx
    v = (v | (v << 2)) & 0x00009249u;   // x..x..x..x..x..x
    return v;
}

// gpu_ops.py:216-224: gi = floor((p - min)/cell) (float32 ops), int64 hash mod n (the modulo by multiply-high:
// M64 = floor((2^64-1)/n), q in {true q - 2 .. true q}).  *fx.. return the cell-relative coordinates.
__device__ __forceinline__ uint32_t bucket_hash(float x, float y, float z, float bx, float by, float bz, float cell,
                                                int64_t n, uint64_t M64, float& fx, float& fy, float& fz, float& flx,
                                                float& fly, float& flz) {
    fx = __fdiv_rn(__fsub_rn(x, bx), cell);
    fy = __fdiv_rn(__fsub_rn(y, by), cell);
    fz = __fdiv_rn(__fsub_rn(z, bz), cell);
    flx = floorf(fx), fly = floorf(fy), flz = floorf(fz);
    int64_t gx = (int64_t)(int32_t)flx, gy = (int64_t)(int32_t)fly, gz = (int64_t)(int32_t)flz;
    int64_t hx = (gx * 73856093LL) ^ (gy * 19349663LL) ^ (gz * 83492791LL);
    int64_t h;
    if (hx >= 0) {  // always, since gi >= 0 for points inside the bounding box
        uint64_t q = __umul64hi((uint64_t)hx, M64);
        uint64_t r = (uint64_t)hx - q * (uint64_t)n;
        while (r >= (uint64_t)n) r -= (uint64_t)n;
        h = (int64_t)r;
    } else {
        h = hx % n;
        if (h < 0) h += n;
    }
    return (uint32_t)h;
}

__device__ __forceinline__ uint32_t bucket_of(float x, float y, float z, float bx, float by, float bz, float cell,
                                              int64_t n, uint64_t M64) {
    float a, b, c, d, e, f;
    return bucket_hash(x, y, z, bx, by, bz, cell, n, M64, a, b, c, d, e, f);
}

// sort key: bucket hash << kMortonBits | Morton code of the position inside the cell (ordering only -- the
// in-bucket order never affects results)
__device__ __forceinline__ uint64_t bucket_key(float x, float y, float z, float bx, float by, float bz, float cell,
                                               int64_t n, uint64_t M64) {
    float fx, fy, fz, flx, fly, flz;
    const uint32_t h = bucket_hash(x, y, z, bx, by, bz, cell, n, M64, fx, fy, fz, flx, fly, flz);
    uint32_t sx = (uint32_t)fminf(kMortonMax, fmaxf(0.f, (fx - flx) * kMortonScale));
    uint32_t sy = (uint32_t)fminf(kMortonMax, fmaxf(0.f, (fy - fly) * kMortonScale));
    uint32_t sz = (uint32_t)fminf(kMortonMax, fmaxf(0.f, (fz - flz) * kMortonScale));
    uint32_t mort = (spread6(sx) << 2) | (spread6(sy) << 1) | spread6(sz);
    return ((uint64_t)h << kMortonBits) | (uint64_t)mort;
}

// The sort works on ONE 64-bit word per point: [ bucket | Morton (top mort_bits of the kMortonBits code) | index ].
// Only the bits above the index are sorted (stable LSD passes => equal keys stay in index order, as with a separate
// payload), and a pass moves 8 bytes per point instead of 12.  The Morton field takes what is left of the 64 bits
// after the bucket and the index (15 bits up to 16.7 M points, 9 at 80 M, 3 at 1 B): it only orders points INSIDE a
// bucket, which never changes a result.
struct PackFmt {
    int idx_bits, mort_bits, bucket_bits;
    __host__ __device__ int key_shift() const { return idx_bits + mort_bits; }     // word >> key_shift = bucket
    __host__ __device__ uint64_t idx_mask() const { return (1ull << idx_bits) - 1ull; }
    __host__ __device__ int sort_begin() const { return idx_bits; }
    __host__ __device__ int sort_end() const { return idx_bits + mort_bits + bucket_bits; }
};

static int bits_for(int64_t n) {   // smallest b with 2^b >= n (at least 1)
    int b = 1;
    while (((int64_t)1 << b) < n) ++b;
    return b;
}

static PackFmt pack_fmt(int64_t n_items, int64_t n_buckets) {
    PackFmt f;
    f.idx_bits = bits_for(n_items);
    f.bucket_bits = bits_for(n_buckets);
    int avail = 64 - f.idx_bits - f.bucket_bits;
    if (avail > kMortonBits) avail = kMortonBits;
    f.mort_bits = avail < 0 ? 0 : avail - avail % 3;
    return f;
}

__device__ __forceinline__ uint64_t pack_word(uint64_t key /* bucket << kMortonBits | morton */, uint64_t bucket_sub,
                                              int64_t idx, PackFmt f) {
    const uint64_t bucket = (key >> kMortonBits) - bucket_sub;
    const uint64_t mort = (key & ((1ull << kMortonBits) - 1ull)) >> (kMortonBits - f.mort_bits);
    return (((bucket << f.mort_bits) | mort) << f.idx_bits) | (uint64_t)idx;
}

__global__ void __launch_bounds__(256) k_sor_keys(const float* __restrict__ xyz, int64_t n, float bx, float by,
                                                  float bz, float cell, uint64_t M64, PackFmt f,
                                                  uint64_t* __restrict__ keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = pack_word(bucket_key(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], bx, by, bz, cell, n, M64), 0, i, f);
}

// gpu_ops.py:228-237 in one pass over the hash-sorted order.  One block = 1024 sorted points = one "super", one
// warp = one "chunk" of 32.  GATHER: sorted_pos = pos[sort_order] (float4, w = original index) is produced here
// and the bucket of a position comes from its sort key; otherwise spos is given (distributed build) and the
// bucket is re-hashed from the position.  Outputs: {start,end} of every occupied bucket (tab_se pre-zeroed:
// start == end == 0 <=> the reference's cell_start == -1), one bit per sorted position that starts a bucket,
// and the bounding boxes of every chunk and super.
// order-preserving float <-> uint32 (for redux.sync min/max); +/-inf map to the extremes, -0 < +0
__device__ __forceinline__ uint32_t float_to_ord(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_to_float(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

template <bool GATHER>
__device__ __forceinline__ void
    sor_finish_tile(const int64_t tile, const float* __restrict__ xyz, const uint64_t* __restrict__ keys, PackFmt fmt,
                    float4* __restrict__ spos, int64_t n, float bx, float by, float bz, float cell, uint64_t M64,
                    int2* __restrict__ tab_se, uint32_t* __restrict__ startbits, uint32_t* __restrict__ cellbits,
                    float4* __restrict__ caabb, float4* __restrict__ saabb) {
    const int64_t j = tile * 1024 + threadIdx.x;
    const int lane = lane_id();
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    uint32_t h = 0xffffffffu;
    auto hash_at = [&](int64_t t) -> uint32_t {
        if (GATHER) return (uint32_t)(keys[t] >> fmt.key_shift());
        const float4 q = spos[t];
        return bucket_of(q.x, q.y, q.z, bx, by, bz, cell, n, M64);
    };
    int gcx = 0x7fffffff, gcy = 0, gcz = 0;   // grid cell of this position (gpu_ops.py:113-115 arithmetic)
    if (j < n) {
        float x, y, z;
        if (GATHER) {
            const uint64_t word = keys[j];
            const int32_t idx = (int32_t)(word & fmt.idx_mask());
            x = xyz[3 * (int64_t)idx], y = xyz[3 * (int64_t)idx + 1], z = xyz[3 * (int64_t)idx + 2];
            spos[j] = make_float4(x, y, z, __int_as_float(idx));
            h = (uint32_t)(word >> fmt.key_shift());
        } else {
            const float4 p = spos[j];
            x = p.x, y = p.y, z = p.z;
            h = bucket_of(x, y, z, bx, by, bz, cell, n, M64);
        }
        gcx = (int)floorf(__fdiv_rn(__fsub_rn(x, bx), cell));
        gcy = (int)floorf(__fdiv_rn(__fsub_rn(y, by), cell));
        gcz = (int)floorf(__fdiv_rn(__fsub_rn(z, bz), cell));
        lo[0] = hi[0] = x;
        lo[1] = hi[1] = y;
        lo[2] = hi[2] = z;
    }
    // neighbouring hashes: through shared memory inside the block (invalid threads hold the sentinel 0xffffffff, which
    // no real bucket has: h < n < 2^31); only the two block-edge threads look at global memory
    __shared__ uint32_t sh_h[1024];
    sh_h[threadIdx.x] = h;
    __syncthreads();
    uint32_t hprev = threadIdx.x > 0 ? sh_h[threadIdx.x - 1] : 0xffffffffu;
    uint32_t hnext = threadIdx.x < 1023 ? sh_h[threadIdx.x + 1] : 0xffffffffu;
    if (j < n) {
        if (threadIdx.x == 0 && j > 0) hprev = hash_at(j - 1);
        if (threadIdx.x == 1023 && j + 1 < n) hnext = hash_at(j + 1);
    }
    // "the query at this sorted position has another grid cell than the one before it": lets k_sor_knn skip the three
    // divisions + vote per query.  Exact compare of the three cell indices (block edges are conservatively "new").
    __shared__ int sh_c[3][1024];
    sh_c[0][threadIdx.x] = gcx, sh_c[1][threadIdx.x] = gcy, sh_c[2][threadIdx.x] = gcz;
    __syncthreads();
    const bool newcell = j < n && (threadIdx.x == 0 || sh_c[0][threadIdx.x - 1] != gcx ||
                                   sh_c[1][threadIdx.x - 1] != gcy || sh_c[2][threadIdx.x - 1] != gcz);
    const unsigned cb = __ballot_sync(GSX_FULL, newcell);
    const bool start = j < n && (j == 0 || h != hprev);
    const bool end = j < n && (j == n - 1 || h != hnext);
    if (start) tab_se[h].x = (int)j;
    if (end) tab_se[h].y = (int)(j + 1);
    const unsigned sb = __ballot_sync(GSX_FULL, start);
    // chunk boxes: one redux.sync per component on order-preserving integer keys (exact: min/max only select)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        lo[a] = ord_to_float(__reduce_min_sync(GSX_FULL, float_to_ord(lo[a])));
        hi[a] = ord_to_float(__reduce_max_sync(GSX_FULL, float_to_ord(hi[a])));
    }
    __shared__ float sm[6][32];
    const int w = threadIdx.x >> 5;
    const int64_t chunk = tile * 32 + w;
    if (lane == 0) {
        if (chunk * 32 < n) {
            startbits[chunk] = sb;
            cellbits[chunk] = cb;
            caabb[2 * chunk] = make_float4(lo[0], lo[1], lo[2], hi[0]);
            caabb[2 * chunk + 1] = make_float4(hi[1], hi[2], 0.f, 0.f);
        }
        for (int a = 0; a < 3; ++a) {
            sm[a][w] = lo[a];
            sm[3 + a][w] = hi[a];
        }
    }
    __syncthreads();
    if (w == 0) {
        float v[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            v[a] = sm[a][lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                float t = __shfl_xor_sync(GSX_FULL, v[a], o);
                v[a] = a < 3 ? fminf(v[a], t) : fmaxf(v[a], t);
            }
        }
        if (lane == 0) {
            saabb[2 * tile] = make_float4(v[0], v[1], v[2], v[3]);
            saabb[2 * tile + 1] = make_float4(v[4], v[5], 0.f, 0.f);
        }
    }
}

template <bool GATHER>
__global__ void __launch_bounds__(1024)
    k_sor_finish(const float* __restrict__ xyz, const uint64_t* __restrict__ keys, PackFmt fmt,
                 float4* __restrict__ spos, int64_t n, float bx, float by, float bz, float cell, uint64_t M64,
                 int2* __restrict__ tab_se, uint32_t* __restrict__ startbits, uint32_t* __restrict__ cellbits,
                 float4* __restrict__ caabb, float4* __restrict__ saabb) {
    sor_finish_tile<GATHER>(blockIdx.x, xyz, keys, fmt, spos, n, bx, by, bz, cell, M64, tab_se, startbits, cellbits, caabb,
                            saabb);
}

// the same pass as the fallback of the flag-driven stage C: a resident-size grid that returns at once unless the start
// list overflowed (a grid of n/1024 empty blocks would itself cost ~0.1 ms at 80 M points)
__global__ void __launch_bounds__(1024)
    k_sor_finish_gated(float4* __restrict__ spos, int64_t n, float bx, float by, float bz, float cell, uint64_t M64,
                       int2* __restrict__ tab_se, uint32_t* __restrict__ startbits, uint32_t* __restrict__ cellbits,
                       float4* __restrict__ caabb, float4* __restrict__ saabb, const unsigned int* __restrict__ gate) {
    if (!*gate) return;
    const int64_t tiles = (n + 1023) / 1024;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        sor_finish_tile<false>(t, nullptr, nullptr, PackFmt{}, spos, n, bx, by, bz, cell, M64, tab_se, startbits, cellbits,
                               caabb, saabb);
        __syncthreads();
    }
}

// Bounding box of every occupied bucket (exact over its points): lets the query kernel skip whole buckets whose
// box is farther than the current K-th best, and visit the 27 probes nearest first.  Each warp takes the bucket
// starts among its 32 sorted positions (startbits) and reduces each bucket cooperatively (stride 32 over the
// bucket's range; chunks that lie entirely inside the bucket contribute their box instead of their points).
// tab_box[2h] = {lo.xyz, -}, tab_box[2h+1] = {hi.xyz, -}: 32 bytes = one DRAM sector per occupied bucket.
__device__ __forceinline__ void
    bucket_boxes_chunk(const int64_t chunk, const uint32_t* __restrict__ startbits, const float4* __restrict__ spos,
                       const float4* __restrict__ caabb, const int2* __restrict__ tab_se, int64_t n, float bx,
                       float by, float bz, float cell, uint64_t M64, float4* __restrict__ tab_box) {
    const int lane = lane_id();
    if (chunk * 32 >= n) return;
    unsigned m = startbits[chunk];
    // the hash and the end of every bucket that starts in this chunk: one lane per start, in parallel
    uint32_t my_h = 0;
    int my_end = 0;
    if ((m >> lane) & 1u) {
        const float4 p0 = spos[chunk * 32 + lane];
        my_h = bucket_of(p0.x, p0.y, p0.z, bx, by, bz, cell, n, M64);
        my_end = tab_se[my_h].y;
    }
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const int64_t s = chunk * 32 + src;
        const uint32_t hb = __shfl_sync(GSX_FULL, my_h, src);
        const int64_t end = __shfl_sync(GSX_FULL, my_end, src);
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        int64_t cf = (s + 31) >> 5, cl = end >> 5;  // full chunks [cf, cl)
        int64_t head_end = cf * 32, tail_begin = cl * 32;
        if (cf > cl) {  // the bucket lies inside one chunk: reduce it point by point
            head_end = end;
            tail_begin = end;
            cf = cl = 0;
        }
        for (int64_t t = s + lane; t < head_end; t += 32) {
            float4 p = spos[t];
            lo[0] = fminf(lo[0], p.x), lo[1] = fminf(lo[1], p.y), lo[2] = fminf(lo[2], p.z);
            hi[0] = fmaxf(hi[0], p.x), hi[1] = fmaxf(hi[1], p.y), hi[2] = fmaxf(hi[2], p.z);
        }
        for (int64_t c = cf + lane; c < cl; c += 32) {
            float4 a = caabb[2 * c], b = caabb[2 * c + 1];
            lo[0] = fminf(lo[0], a.x), lo[1] = fminf(lo[1], a.y), lo[2] = fminf(lo[2], a.z);
            hi[0] = fmaxf(hi[0], a.w), hi[1] = fmaxf(hi[1], b.x), hi[2] = fmaxf(hi[2], b.y);
        }
        for (int64_t t = tail_begin + lane; t < end; t += 32) {
            float4 p = spos[t];
            lo[0] = fminf(lo[0], p.x), lo[1] = fminf(lo[1], p.y), lo[2] = fminf(lo[2], p.z);
            hi[0] = fmaxf(hi[0], p.x), hi[1] = fmaxf(hi[1], p.y), hi[2] = fmaxf(hi[2], p.z);
        }
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo[a] = fminf(lo[a], __shfl_xor_sync(GSX_FULL, lo[a], o));
                hi[a] = fmaxf(hi[a], __shfl_xor_sync(GSX_FULL, hi[a], o));
            }
        if (lane == 0) {
            tab_box[2 * (size_t)hb] = make_float4(lo[0], lo[1], lo[2], 0.f);
            tab_box[2 * (size_t)hb + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
        }
    }
}

__global__ void __launch_bounds__(256)
    k_sor_bucket_boxes(const uint32_t* __restrict__ startbits, const float4* __restrict__ spos,
                       const float4* __restrict__ caabb, const int2* __restrict__ tab_se, int64_t n, float bx,
                       float by, float bz, float cell, uint64_t M64, float4* __restrict__ tab_box) {
    bucket_boxes_chunk(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, startbits, spos, caabb, tab_se, n, bx, by, bz,
                       cell, M64, tab_box);
}

__global__ void __launch_bounds__(256)
    k_sor_bucket_boxes_gated(const uint32_t* __restrict__ startbits, const float4* __restrict__ spos,
                             const float4* __restrict__ caabb, const int2* __restrict__ tab_se, int64_t n, float bx,
                             float by, float bz, float cell, uint64_t M64, float4* __restrict__ tab_box,
                             const unsigned int* __restrict__ gate) {
    if (!*gate) return;
    const int64_t nchunk = (n + 31) >> 5, step = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < nchunk; c += step)
        bucket_boxes_chunk(c, startbits, spos, caabb, tab_se, n, bx, by, bz, cell, M64, tab_box);
}

// Stage C when the owners shipped per-point flags (bit 0 bucket start, bit 1 cell change).  Three kernels, none of
// which hashes every point (the replicated re-hash was ~130 of ~250 instructions per point) and none of which leaves
// a block waiting on a serial tail:
//   k_sor_finish_flags  one pass over the sorted order: chunk / super boxes, the start and cell bit masks, and the
//                       positions of the bucket starts compacted into ONE global list (a block reserves its slice
//                       with a single atomicAdd);
//   k_sor_bucket_tail   one THREAD per listed bucket start (perfectly compacted, ~1/32 of the points): hash of that
//                       one point, then a serial walk over the bucket's contiguous points (scanning the start flags
//                       for its end) -> {start,end} entry and the exact box of every bucket of <= kSmallBucket points;
//                       longer buckets only get their start written and a bit in `bigbits`;
//   k_sor_big_buckets   one warp per 32 positions, only for the few long buckets: end found by scanning the start
//                       bit mask, box from the chunk boxes (complete after the first kernel).
// The list has room for n/8 + 1024 starts (average bucket >= 8 points); if it overflows, a device-side flag makes
// the last two kernels return and the re-hashing kernels (k_sor_finish<false>, k_sor_bucket_boxes) take over --
// no host round trip either way.
struct StartList {
    unsigned int* count;      // [0] entries reserved, [1] overflow flag
    unsigned int* pos;        // start positions
    unsigned int capacity;
};

__global__ void __launch_bounds__(1024)
    k_sor_finish_flags(const float4* __restrict__ spos, const uint8_t* __restrict__ flags, int64_t n,
                       uint32_t* __restrict__ startbits, uint32_t* __restrict__ cellbits, float4* __restrict__ caabb,
                       float4* __restrict__ saabb, StartList sl) {
    const int64_t j = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    const int lane = lane_id();
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    bool start = false, newcell = false;
    if (j < n) {
        const float4 p = spos[j];
        lo[0] = hi[0] = p.x;
        lo[1] = hi[1] = p.y;
        lo[2] = hi[2] = p.z;
        const uint8_t f = flags[j];
        start = (f & 1) != 0;
        newcell = (f & 2) != 0;
    }
    const unsigned sb = __ballot_sync(GSX_FULL, start), cb = __ballot_sync(GSX_FULL, newcell);
    __shared__ unsigned s_wcnt[32], s_base;
    const int w = threadIdx.x >> 5;
    if (lane == 0) s_wcnt[w] = __popc(sb);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        lo[a] = ord_to_float(__reduce_min_sync(GSX_FULL, float_to_ord(lo[a])));
        hi[a] = ord_to_float(__reduce_max_sync(GSX_FULL, float_to_ord(hi[a])));
    }
    __shared__ float sm[6][32];
    const int64_t chunk = (int64_t)blockIdx.x * 32 + w;
    if (lane == 0) {
        if (chunk * 32 < n) {
            startbits[chunk] = sb;
            cellbits[chunk] = cb;
            caabb[2 * chunk] = make_float4(lo[0], lo[1], lo[2], hi[0]);
            caabb[2 * chunk + 1] = make_float4(hi[1], hi[2], 0.f, 0.f);
        }
        for (int a = 0; a < 3; ++a) {
            sm[a][w] = lo[a];
            sm[3 + a][w] = hi[a];
        }
    }
    __syncthreads();
    if (w == 0) {
        // exclusive prefix of the 32 warp counts, one global reservation for the whole block
        unsigned v = s_wcnt[lane], x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned y = __shfl_up_sync(GSX_FULL, x, o);
            if (lane >= o) x += y;
        }
        s_wcnt[lane] = x - v;
        if (lane == 31) {
            unsigned base = 0;
            if (x) {
                base = atomicAdd(sl.count, x);
                if (base + x > sl.capacity) {
                    atomicExch(sl.count + 1, 1u);
                    base = 0xffffffffu;
                }
            }
            s_base = base;
        }
        float vb[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            vb[a] = sm[a][lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                float t = __shfl_xor_sync(GSX_FULL, vb[a], o);
                vb[a] = a < 3 ? fminf(vb[a], t) : fmaxf(vb[a], t);
            }
        }
        if (lane == 0) {
            saabb[2 * (int64_t)blockIdx.x] = make_float4(vb[0], vb[1], vb[2], vb[3]);
            saabb[2 * (int64_t)blockIdx.x + 1] = make_float4(vb[4], vb[5], 0.f, 0.f);
        }
    }
    __syncthreads();
    if (start && s_base != 0xffffffffu)
        sl.pos[s_base + s_wcnt[w] + __popc(sb & ((1u << lane) - 1u))] = (unsigned)j;
}

__global__ void __launch_bounds__(256)
    k_sor_bucket_tail(const float4* __restrict__ spos, const uint8_t* __restrict__ flags, int64_t n, float bx, float by,
                      float bz, float cell, uint64_t M64, int2* __restrict__ tab_se, float4* __restrict__ tab_box,
                      uint32_t* __restrict__ bigbits, StartList sl) {
    if (sl.count[1]) return;   // list overflow: the re-hashing path handles everything
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= sl.count[0]) return;
    const int64_t pj = sl.pos[t];
    const float4 p = spos[pj];
    const uint32_t h = bucket_of(p.x, p.y, p.z, bx, by, bz, cell, n, M64);
    float blo[3] = {p.x, p.y, p.z}, bhi[3] = {p.x, p.y, p.z};
    int64_t u = pj + 1;
    const int64_t lim = pj + kSmallBucket < n ? pj + kSmallBucket : n;
    for (; u < lim; ++u) {
        if (flags[u] & 1) break;
        const float4 c = spos[u];
        blo[0] = fminf(blo[0], c.x), blo[1] = fminf(blo[1], c.y), blo[2] = fminf(blo[2], c.z);
        bhi[0] = fmaxf(bhi[0], c.x), bhi[1] = fmaxf(bhi[1], c.y), bhi[2] = fmaxf(bhi[2], c.z);
    }
    const bool closed = u == n || (flags[u] & 1);
    if (closed) {
        tab_se[h] = make_int2((int)pj, (int)u);
        tab_box[2 * (size_t)h] = make_float4(blo[0], blo[1], blo[2], 0.f);
        tab_box[2 * (size_t)h + 1] = make_float4(bhi[0], bhi[1], bhi[2], 0.f);
    } else {
        tab_se[h].x = (int)pj;   // the end comes from k_sor_big_buckets
        atomicOr(bigbits + (pj >> 5), 1u << (pj & 31));
    }
}

// the few buckets longer than kSmallBucket: one warp per chunk that holds such a start
__global__ void __launch_bounds__(256)
    k_sor_big_buckets(const uint32_t* __restrict__ bigbits, const uint32_t* __restrict__ startbits,
                      const float4* __restrict__ spos, const float4* __restrict__ caabb, int64_t n, float bx, float by,
                      float bz, float cell, uint64_t M64, int2* __restrict__ tab_se, float4* __restrict__ tab_box,
                      StartList sl) {
    if (sl.count[1]) return;
    const int lane = lane_id();
    const int64_t nchunk = (n + 31) >> 5;
    // a resident-size grid sweeps the (almost empty) bit mask 32 words per warp step; the warp then handles the
    // words that have a bit, one after the other
    const int64_t wstep = (((int64_t)gridDim.x * blockDim.x) >> 5) * 32;
    for (int64_t c0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; c0 < nchunk; c0 += wstep) {
    const uint32_t myword = c0 + lane < nchunk ? bigbits[c0 + lane] : 0u;
    unsigned wordmask = __ballot_sync(GSX_FULL, myword != 0u);
    while (wordmask) {
    const int wl = __ffs(wordmask) - 1;
    wordmask &= wordmask - 1;
    const int64_t chunk = c0 + wl;
    unsigned m = __shfl_sync(GSX_FULL, myword, wl);
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const int64_t s = chunk * 32 + src;
        // end = next bucket start after s: first in this chunk's word, then 32 words at a time
        int64_t end = n;
        {
            const unsigned rest = src == 31 ? 0u : (startbits[chunk] & (0xffffffffu << (src + 1)));
            if (rest) {
                end = chunk * 32 + __ffs(rest) - 1;
            } else {
                for (int64_t d0 = chunk + 1; d0 < nchunk; d0 += 32) {
                    const int64_t c = d0 + lane;
                    const unsigned wv = c < nchunk ? startbits[c] : 0u;
                    const unsigned any = __ballot_sync(GSX_FULL, wv != 0u);
                    if (any) {
                        const int l = __ffs(any) - 1;
                        const unsigned word = __shfl_sync(GSX_FULL, wv, l);
                        end = (d0 + l) * 32 + __ffs(word) - 1;
                        break;
                    }
                }
            }
        }
        const float4 p0 = spos[s];
        const uint32_t hb = bucket_of(p0.x, p0.y, p0.z, bx, by, bz, cell, n, M64);
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        int64_t cf = (s + 31) >> 5, cl = end >> 5;  // full chunks [cf, cl)
        int64_t head_end = cf * 32, tail_begin = cl * 32;
        if (cf > cl) {
            head_end = end;
            tail_begin = end;
            cf = cl = 0;
        }
        for (int64_t t = s + lane; t < head_end; t += 32) {
            float4 p = spos[t];
            lo[0] = fminf(lo[0], p.x), lo[1] = fminf(lo[1], p.y), lo[2] = fminf(lo[2], p.z);
            hi[0] = fmaxf(hi[0], p.x), hi[1] = fmaxf(hi[1], p.y), hi[2] = fmaxf(hi[2], p.z);
        }
        for (int64_t c = cf + lane; c < cl; c += 32) {
            float4 a = caabb[2 * c], b = caabb[2 * c + 1];
            lo[0] = fminf(lo[0], a.x), lo[1] = fminf(lo[1], a.y), lo[2] = fminf(lo[2], a.z);
            hi[0] = fmaxf(hi[0], a.w), hi[1] = fmaxf(hi[1], b.x), hi[2] = fmaxf(hi[2], b.y);
        }
        for (int64_t t = tail_begin + lane; t < end; t += 32) {
            float4 p = spos[t];
            lo[0] = fminf(lo[0], p.x), lo[1] = fminf(lo[1], p.y), lo[2] = fminf(lo[2], p.z);
            hi[0] = fmaxf(hi[0], p.x), hi[1] = fmaxf(hi[1], p.y), hi[2] = fmaxf(hi[2], p.z);
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = ord_to_float(__reduce_min_sync(GSX_FULL, float_to_ord(lo[a])));
            hi[a] = ord_to_float(__reduce_max_sync(GSX_FULL, float_to_ord(hi[a])));
        }
        if (lane == 0) {
            tab_se[hb].y = (int)end;
            tab_box[2 * (size_t)hb] = make_float4(lo[0], lo[1], lo[2], 0.f);
            tab_box[2 * (size_t)hb + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
        }
    }
    }
    }
}

template <bool GATHER>
static int sor_finish(const float* xyz, int64_t n, const float* bmin, float cell, SorWs& w, PackFmt fmt, cudaStream_t st) {
    const uint64_t M64 = 0xFFFFFFFFFFFFFFFFull / (uint64_t)n;
    GSX_CUDA_CHECK(cudaMemsetAsync(w.tab_se, 0, (size_t)n * sizeof(int2), st));
    k_sor_finish<GATHER><<<(int)((n + 1023) / 1024), 1024, 0, st>>>(xyz, w.keys_sorted, fmt, w.spos, n, bmin[0],
                                                                    bmin[1], bmin[2], cell, M64, w.tab_se, w.startbits,
                                                                    w.cellbits, w.caabb, w.saabb);
    GSX_KERNEL_CHECK();
    k_sor_bucket_boxes<<<(int)((n + 255) / 256), 256, 0, st>>>(w.startbits, w.spos, w.caabb, w.tab_se, n, bmin[0],
                                                               bmin[1], bmin[2], cell, M64, w.tab_box);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

int sor_build(const float* xyz, int64_t n, const float* bmin, float cell, SorWs& w, cudaStream_t st) {
    GSX_NVTX("gsx::sor_build");
    int blocks = (int)((n + 255) / 256);
    const PackFmt fmt = pack_fmt(n, n);
    k_sor_keys<<<blocks, 256, 0, st>>>(xyz, n, bmin[0], bmin[1], bmin[2], cell, 0xFFFFFFFFFFFFFFFFull / (uint64_t)n,
                                       fmt, w.keys0);
    GSX_KERNEL_CHECK();
    {
        int rc = radix_sort_keys(w.keys0, w.keys1, n, fmt.sort_begin(), fmt.sort_end(), w.sort_ws, w.sort_ws_bytes,
                                 &w.keys_sorted, st);
        if (rc) return rc;
    }
    return sor_finish<true>(xyz, n, bmin, cell, w, fmt, st);
}

// ------------------------------------------------------------------ distributed build (one process per GPU)
// Bucket-range ownership: rank o owns the buckets [ceil(o*N/G), ceil((o+1)*N/G)).  Every rank sorts its own
// slab by the GLOBAL bucket key, the runs are exchanged by owner (all-to-all, host side: gsx/dist.py), each
// owner sorts what it received, the sorted float4 segments are all-gathered, and every rank fills its table,
// boxes and bucket boxes from the (now identical) sorted array.  The sort work per rank drops from N to 2N/G.

// stage A: owner rank of every slab point (owner o holds the buckets [ceil(o*N/G), ceil((o+1)*N/G)))
__global__ void __launch_bounds__(256) k_sor_owner_keys(const float* __restrict__ xyz, int64_t n, int64_t n_global,
                                                        int world, float bx, float by, float bz, float cell,
                                                        uint64_t M64, int idx_bits, uint64_t* __restrict__ keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t h = bucket_key(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], bx, by, bz, cell, n_global, M64) >> kMortonBits;
    // o = floor(h*G/N) satisfies ceil(o*N/G) <= h; it is the owner unless h < ceil(o*N/G) can happen -- it cannot:
    // o*N/G <= h  =>  ceil(o*N/G) <= h because h is an integer.
    keys[i] = (((h * (uint64_t)world) / (uint64_t)n_global) << idx_bits) | (uint64_t)i;   // owner | slab index
}

__global__ void __launch_bounds__(256) k_sor_gather_slab(const float* __restrict__ xyz,
                                                         const uint64_t* __restrict__ words, uint64_t idx_mask, int64_t n,
                                                         int64_t idx_base, float4* __restrict__ pos4) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int32_t idx = (int32_t)(words[j] & idx_mask);
    pos4[j] = make_float4(xyz[3 * (int64_t)idx], xyz[3 * (int64_t)idx + 1], xyz[3 * (int64_t)idx + 2],
                          __int_as_float((int)(idx_base + idx)));
}

__global__ void k_sor_owner_counts(const uint64_t* __restrict__ owners_sorted, int idx_bits, int64_t n, int world,
                                   long long* __restrict__ cuts) {
    // cuts[o] = first sorted position whose owner is >= o (o = 0..world); one thread per boundary, binary search
    int o = threadIdx.x;
    if (o > world) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if ((owners_sorted[mid] >> idx_bits) < (uint64_t)o) lo = mid + 1; else hi = mid;
    }
    cuts[o] = lo;
}

int sor_dist_local_run(const float* xyz, int64_t n_local, int64_t idx_base, int64_t n_global, int world,
                       const float* bmin, float cell, float4* pos4_out, long long* cuts_dev, SorWs& w,
                       cudaStream_t st) {
    GSX_NVTX("gsx::sor_dist_local_run");
    GSX_REQUIRE(world >= 1 && world <= 255, GSX_ERR_ARG, "sor: world size must be in [1,255]");
    if (n_local == 0) {
        GSX_CUDA_CHECK(cudaMemsetAsync(cuts_dev, 0, (size_t)(world + 1) * sizeof(long long), st));
        return GSX_OK;
    }
    int blocks = (int)((n_local + 255) / 256);
    const int idx_bits = bits_for(n_local);
    k_sor_owner_keys<<<blocks, 256, 0, st>>>(xyz, n_local, n_global, world, bmin[0], bmin[1], bmin[2], cell,
                                             0xFFFFFFFFFFFFFFFFull / (uint64_t)n_global, idx_bits, w.keys0);
    GSX_KERNEL_CHECK();
    uint64_t* ks = nullptr;
    int rc = radix_sort_keys(w.keys0, w.keys1, n_local, idx_bits, idx_bits + 8, w.sort_ws, w.sort_ws_bytes, &ks,
                             st);  // one stable pass: a partition by owner
    if (rc) return rc;
    k_sor_gather_slab<<<blocks, 256, 0, st>>>(xyz, ks, (1ull << idx_bits) - 1ull, n_local, idx_base, pos4_out);
    GSX_KERNEL_CHECK();
    k_sor_owner_counts<<<1, 256, 0, st>>>(ks, idx_bits, n_local, world, cuts_dev);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

// stage B: order the received runs of this rank's bucket range
__global__ void __launch_bounds__(256) k_gather4(const float4* __restrict__ in, const uint64_t* __restrict__ words,
                                                 uint64_t idx_mask, int64_t n, float4* __restrict__ out) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) out[j] = in[words[j] & idx_mask];
}

// sort key of the owner's points: the bucket RELATIVE to the first bucket of the owner's range (the high log2(G) bits
// of the absolute bucket are constant inside a range: one radix pass less from 8 ranks on)
__global__ void __launch_bounds__(256) k_sor_keys_pos4(const float4* __restrict__ pos4, int64_t n, int64_t n_global,
                                                       float bx, float by, float bz, float cell, uint64_t M64,
                                                       uint64_t bucket_lo, PackFmt f, uint64_t* __restrict__ keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = pos4[i];
    keys[i] = pack_word(bucket_key(p.x, p.y, p.z, bx, by, bz, cell, n_global, M64), bucket_lo, i, f);
}

// stage B output with per-point flags for stage C: bit 0 = this sorted point starts a bucket, bit 1 = its grid cell
// differs from the previous sorted point's (first point of a segment: both).  The owner knows the sorted keys, so
// the ranks that receive the segment do not have to re-hash every point (their stage C is replicated work).
__global__ void __launch_bounds__(256)
    k_owner_gather_flags(const float4* __restrict__ in, const uint64_t* __restrict__ keys_sorted, PackFmt fmt, int64_t m, float bx, float by, float bz, float cell,
                         float4* __restrict__ out, uint8_t* __restrict__ flags) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ int sh_c[3][256];
    int gx = 0x7fffffff, gy = 0, gz = 0;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < m) {
        p = in[keys_sorted[j] & fmt.idx_mask()];
        out[j] = p;
        gx = (int)floorf(__fdiv_rn(__fsub_rn(p.x, bx), cell));
        gy = (int)floorf(__fdiv_rn(__fsub_rn(p.y, by), cell));
        gz = (int)floorf(__fdiv_rn(__fsub_rn(p.z, bz), cell));
    }
    sh_c[0][threadIdx.x] = gx, sh_c[1][threadIdx.x] = gy, sh_c[2][threadIdx.x] = gz;
    __syncthreads();
    if (j >= m) return;
    const bool start = j == 0 || (keys_sorted[j] >> fmt.key_shift()) != (keys_sorted[j - 1] >> fmt.key_shift());
    bool newcell = threadIdx.x == 0 || sh_c[0][threadIdx.x - 1] != gx || sh_c[1][threadIdx.x - 1] != gy ||
                   sh_c[2][threadIdx.x - 1] != gz;   // block edges: conservatively "new"
    flags[j] = (uint8_t)((start ? 1 : 0) | ((newcell || start) ? 2 : 0));
}

int sor_dist_merge(const float4* pos4_in, int64_t m, int64_t n_global, int64_t bucket_lo, int64_t bucket_hi,
                   const float* bmin, float cell, float4* pos4_out, uint8_t* flags_out, SorWs& w, cudaStream_t st) {
    GSX_NVTX("gsx::sor_dist_merge");
    if (m == 0) return GSX_OK;
    GSX_REQUIRE(bucket_lo >= 0 && bucket_lo < bucket_hi && bucket_hi <= n_global, GSX_ERR_ARG, "sor: bad bucket range");
    int blocks = (int)((m + 255) / 256);
    const PackFmt fmt = pack_fmt(m, bucket_hi - bucket_lo);
    k_sor_keys_pos4<<<blocks, 256, 0, st>>>(pos4_in, m, n_global, bmin[0], bmin[1], bmin[2], cell,
                                            0xFFFFFFFFFFFFFFFFull / (uint64_t)n_global, (uint64_t)bucket_lo, fmt, w.keys0);
    GSX_KERNEL_CHECK();
    uint64_t* ks = nullptr;
    int rc = radix_sort_keys(w.keys0, w.keys1, m, fmt.sort_begin(), fmt.sort_end(), w.sort_ws, w.sort_ws_bytes, &ks, st);
    if (rc) return rc;
    if (flags_out)
        k_owner_gather_flags<<<blocks, 256, 0, st>>>(pos4_in, ks, fmt, m, bmin[0], bmin[1], bmin[2], cell, pos4_out,
                                                     flags_out);
    else
        k_gather4<<<blocks, 256, 0, st>>>(pos4_in, ks, fmt.idx_mask(), m, pos4_out);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

// stage C: everything gsx_sor_build produces, from an already hash-sorted float4 array
int sor_build_from_sorted(const float4* spos_in, const uint8_t* flags, int64_t n, const float* bmin, float cell, SorWs& w,
                          cudaStream_t st) {
    GSX_NVTX("gsx::sor_build_from_sorted");
    if (spos_in != w.spos)
        GSX_CUDA_CHECK(cudaMemcpyAsync(w.spos, spos_in, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, st));
    w.keys_sorted = nullptr;
    if (!flags) return sor_finish<false>(nullptr, n, bmin, cell, w, PackFmt{}, st);
    const uint64_t M64 = 0xFFFFFFFFFFFFFFFFull / (uint64_t)n;
    const int64_t nchunk = (n + 31) / 32;
    StartList sl;
    sl.count = w.counters + 8;                       // [8] count, [9] overflow
    sl.pos = reinterpret_cast<unsigned int*>(w.startlist);
    sl.capacity = (unsigned)(n / 8 + 1024);
    GSX_CUDA_CHECK(cudaMemsetAsync(w.tab_se, 0, (size_t)n * sizeof(int2), st));
    GSX_CUDA_CHECK(cudaMemsetAsync(w.bigbits, 0, (size_t)nchunk * sizeof(uint32_t), st));
    GSX_CUDA_CHECK(cudaMemsetAsync(sl.count, 0, 2 * sizeof(unsigned int), st));
    k_sor_finish_flags<<<(int)((n + 1023) / 1024), 1024, 0, st>>>(w.spos, flags, n, w.startbits, w.cellbits, w.caabb,
                                                                  w.saabb, sl);
    GSX_KERNEL_CHECK();
    const unsigned tail_blocks = (sl.capacity + 255) / 256;   // upper bound of the list length (threads beyond it exit)
    k_sor_bucket_tail<<<tail_blocks, 256, 0, st>>>(w.spos, flags, n, bmin[0], bmin[1], bmin[2], cell, M64, w.tab_se,
                                                   w.tab_box, w.bigbits, sl);
    GSX_KERNEL_CHECK();
    k_sor_big_buckets<<<sm_count() * 8, 256, 0, st>>>(w.bigbits, w.startbits, w.spos, w.caabb, n, bmin[0], bmin[1], bmin[2],
                                                      cell, M64, w.tab_se, w.tab_box, sl);
    GSX_KERNEL_CHECK();
    // overflow fallback (average bucket < 8 points): the re-hashing pair, gated on the device-side flag
    const int resident = sm_count() * 2;
    k_sor_finish_gated<<<resident, 1024, 0, st>>>(w.spos, n, bmin[0], bmin[1], bmin[2], cell, M64, w.tab_se, w.startbits,
                                                  w.cellbits, w.caabb, w.saabb, sl.count + 1);
    GSX_KERNEL_CHECK();
    k_sor_bucket_boxes_gated<<<resident * 4, 256, 0, st>>>(w.startbits, w.spos, w.caabb, w.tab_se, n, bmin[0], bmin[1],
                                                           bmin[2], cell, M64, w.tab_box, sl.count + 1);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

// ------------------------------------------------------------------ query kernel

// gpu_ops.py:130-132 probe hash.  mode 0: int32 wrapping products (Taichi default_ip), Python-style
// modulo via Lemire fastmod; mode 1: int64 products.
__device__ __forceinline__ uint32_t probe_hash(int nx, int ny, int nz, uint32_t n, uint64_t M, int mode) {
    if (mode == GSX_HASH_MODE_I32WRAP) {
        int32_t h = (int32_t)((uint32_t)nx * 73856093u) ^ (int32_t)((uint32_t)ny * 19349663u) ^
                    (int32_t)((uint32_t)nz * 83492791u);
        uint32_t a = h < 0 ? (uint32_t)(-(int64_t)h) : (uint32_t)h;
        uint32_t r = fastmod_u32(a, M, n);
        return h < 0 ? (r ? n - r : 0u) : r;
    } else {
        int64_t h = ((int64_t)nx * 73856093LL) ^ ((int64_t)ny * 19349663LL) ^ ((int64_t)nz * 83492791LL);
        int64_t r = h % (int64_t)n;
        if (r < 0) r += n;
        return (uint32_t)r;
    }
}

// Lower bound of the float32 d^2 the scan would compute for any point inside the box: same op
// sequence (sub, mul, add -- no fma), every op monotone, so lb <= d2(point) exactly.
__device__ __forceinline__ float box_lb(const float4* __restrict__ aabb, int64_t id, float qx, float qy, float qz) {
    float4 a = __ldg(aabb + 2 * id), b = __ldg(aabb + 2 * id + 1);
    float dx = fmaxf(fmaxf(__fsub_rn(a.x, qx), __fsub_rn(qx, a.w)), 0.f);
    float dy = fmaxf(fmaxf(__fsub_rn(a.y, qy), __fsub_rn(qy, b.x)), 0.f);
    float dz = fmaxf(fmaxf(__fsub_rn(a.z, qz), __fsub_rn(qz, b.y)), 0.f);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// one compare-exchange stage of a 32-lane bitonic network: lanes whose `take_min` is set keep the
// smaller of (own, partner), the others the larger
__device__ __forceinline__ float cmpx(float v, int j, bool take_min) {
    float o = __shfl_xor_sync(GSX_FULL, v, j);
    return take_min ? fminf(v, o) : fmaxf(v, o);
}

// ascending bitonic sort of one value per lane (15 stages)
__device__ __forceinline__ float warp_sort32(float v, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) v = cmpx(v, j, ((lane & k) == 0) == ((lane & j) == 0));
    }
    return v;
}

#ifndef GSX_KNN_FIRST_SORT
#define GSX_KNN_FIRST_SORT 1
#endif
// long buckets that span fewer than this many supers (1024 points each) skip the super-box level (0: never).
// A/B (profiles/r02c_knn_variants.log): 8 -> -1.4 % on the mixed cloud (within ~1 % run-to-run noise), 32 -> +6 %.
#ifndef GSX_KNN_FLAT_SUPERS
#define GSX_KNN_FLAT_SUPERS 8
#endif
// Epilogue of a query (gpu_ops.py:163-174: serial float32 sum of the valid distances, mean) -- batched: every query
// of a batch parks its K ascending distances and its row number in shared memory, and after the batch lane q sums
// query q (16 serial sums run side by side instead of one shuffle + add per rank on lane 0 of every query).
#ifndef GSX_KNN_EPI_SMEM
#define GSX_KNN_EPI_SMEM 1
#endif
template <int NREG>
struct TopK {
    float v0, v1;  // lane l holds rank l (v0) and rank 32+l (v1) of the ascending d^2 list
    float tau;     // current K-th smallest (rank K-1), warp-uniform
    int K;
    __device__ __forceinline__ void init(int k) {
        K = k;
        v0 = v1 = tau = __uint_as_float(GSX_D2LIM_BITS);
    }
    __device__ __forceinline__ void refresh_tau() {
        tau = (NREG == 2 && K > 32) ? __shfl_sync(GSX_FULL, v1, K - 33) : __shfl_sync(GSX_FULL, v0, K - 1);
    }
    // insert warp-uniform x (< tau), gpu_ops.py:154-160 in the d^2 domain
    __device__ __forceinline__ void insert(float x, int lane) {
        float up0 = __shfl_up_sync(GSX_FULL, v0, 1);
        if (NREG == 2) {
            float top0 = __shfl_sync(GSX_FULL, v0, 31);
            float up1 = __shfl_up_sync(GSX_FULL, v1, 1);
            if (lane == 0) up1 = top0;
            if (v1 > x) v1 = fmaxf(up1, x);
        }
        if (lane == 0) up0 = 0.f;
        if (v0 > x) v0 = fmaxf(up0, x);
        refresh_tau();
    }
    // NREG==1 only: merge one candidate per lane (nv; lanes without a candidate pass the sentinel) into
    // the list.  sort(nv) ascending, reverse it, lane-wise min with the ascending list = the 32 smallest
    // of the union as a bitonic sequence, 5 merge stages sort it.  Lanes >= K only ever hold values
    // >= rank K-1, so they never change the K smallest (only the multiset of values matters, A.1-7).
    __device__ __forceinline__ void merge32(float nv, int lane) {
        nv = warp_sort32(nv, lane);
#if GSX_KNN_FIRST_SORT
        // the first merge of a query meets an empty list (32 sentinels): the sorted candidates ARE the merged list --
        // skips the reversal and the 5 merge stages (the sentinel is the largest value either side can hold)
        if (__all_sync(GSX_FULL, v0 == __uint_as_float(GSX_D2LIM_BITS))) {
            v0 = nv;
            refresh_tau();
            return;
        }
#endif
        float r = __shfl_sync(GSX_FULL, nv, 31 - lane);
        float m = fminf(v0, r);
#pragma unroll
        for (int j = 16; j > 0; j >>= 1) m = cmpx(m, j, (lane & j) == 0);
        v0 = m;
        refresh_tau();
    }
};

// positions in the hash-sorted order fit 31 bits (n < 2^31 - 64): 32-bit index arithmetic in the scan loops
#ifndef GSX_KNN_I32
#define GSX_KNN_I32 1
#endif
#if GSX_KNN_I32
typedef int pos_t;
#else
typedef int64_t pos_t;
#endif
// A/B variant named by BASELINE.json's north_star: stage the query's centre bucket (<= 64 points = 1 KiB) into shared
// memory with a 1-D TMA bulk copy (cp.async.bulk + mbarrier) once per cell change, and scan it from there.
#ifndef GSX_KNN_TMA
#define GSX_KNN_TMA 0
#endif

#ifndef GSX_MERGE_THRESHOLD
#define GSX_MERGE_THRESHOLD 9
#endif
constexpr int kMergeThreshold = GSX_MERGE_THRESHOLD;  // serial insert ~11 instr each vs ~95 for a full merge

// distance of the query to candidate j and ballot/shfl insertion of the lanes that beat tau
template <int NREG, bool STATS>
__device__ __forceinline__ void scan32(const float4* __restrict__ spos, pos_t j, bool valid, float qx, float qy,
                                       float qz, TopK<NREG>& tk, int lane, unsigned long long& n_scanned,
                                       const float4* sbuf = nullptr) {
    float d2 = INFINITY;
    if (valid) {
        float4 c = sbuf ? sbuf[lane] : __ldg(spos + j);
        float ax = __fsub_rn(qx, c.x), ay = __fsub_rn(qy, c.y), az = __fsub_rn(qz, c.z);
        d2 = __fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az));
    }
    if (STATS) n_scanned += __popc(__ballot_sync(GSX_FULL, valid));
    bool pass = valid && d2 > 1.0e-12f && d2 < tk.tau;
    unsigned m = __ballot_sync(GSX_FULL, pass);
    if (NREG == 1 && __popc(m) >= kMergeThreshold) {
        tk.merge32(pass ? d2 : __uint_as_float(GSX_D2LIM_BITS), lane);
        return;
    }
    while (m) {
        int src = __ffs(m) - 1;
        m &= m - 1;
        float x = __shfl_sync(GSX_FULL, d2, src);
        if (x < tk.tau) tk.insert(x, lane);
    }
}

#ifndef GSX_KNN_MINBLOCKS
#define GSX_KNN_MINBLOCKS 8
#endif
// Group path (K <= 32, batched epilogue): a batch whose positions all lie in one grid cell, inside the long bucket that
// the centre probe reaches, walks the probes / super boxes / chunk boxes ONCE for the whole batch.  The walk prunes
// with the box-to-box bound lb(B, box) (B = bounding box of the batch) against tau_G = the largest seed tau of the
// batch, and lists what survives; each query then tests only the listed boxes with its own bound.  Exact: for every q
// in B, lb(B, box) <= box_lb(q, box) (same monotone op sequence), and tau_G >= every member's tau, so a box left out
// satisfies lb(q) >= tau_seed(q) -- the same rule as the per-query walk (DESIGN §4.2).  A seed list that is not full,
// or a list longer than GSX_KNN_GROUP_LIST entries, sends the batch to the per-query path.
#ifndef GSX_KNN_GROUP
#define GSX_KNN_GROUP 1
#endif
#ifndef GSX_KNN_GROUP_LIST
#define GSX_KNN_GROUP_LIST 256
#endif
// A/B (profiles/r03_knn_variants.log, 10 M mixed): 32 / 64 entries slower than no group path, 128 -3.6 %, 256 -4.5 %,
// 512 -2.2 % (the shared memory starts to cost L1)
constexpr int kGroupList = GSX_KNN_GROUP_LIST;   // list entries per warp (shared memory)
// Diagnostic build (scripts/knn_class_profile.py): with stats, lane 0 of every batch adds the batch's clock64 cycles
// and query count to one of 4 classes by the size of the centre probe's bucket (<= 64, <= 1024, <= 16384, larger):
// stats[8 + c] cycles, stats[12 + c] queries.  Never shipped.
#ifndef GSX_KNN_PROFILE
#define GSX_KNN_PROFILE 0
#endif
#ifndef GSX_KNN_CELLBITS
#define GSX_KNN_CELLBITS 1
#endif

// shared memory of k_sor_knn: the epilogue rows, then (group path) one list per warp
template <int NREG, int ES>
__host__ __device__ constexpr bool knn_group_on() { return GSX_KNN_GROUP && GSX_KNN_CELLBITS && NREG == 1 && ES > 0; }
template <int NREG, int ES>
constexpr size_t knn_smem_bytes() {
    return (size_t)8 * kQueryBatch * ES * sizeof(float) +
           (knn_group_on<NREG, ES>() ? (size_t)8 * (kGroupList + 32) * sizeof(unsigned) : 0);
}

template <int NREG, bool STATS, int ES>
__global__ void __launch_bounds__(256, GSX_KNN_MINBLOCKS)
    k_sor_knn(const float4* __restrict__ spos, const int2* __restrict__ tab_se, const float4* __restrict__ tab_box,
              const uint32_t* __restrict__ cellbits, const float4* __restrict__ caabb,
              const float4* __restrict__ saabb, float* __restrict__ final_means, unsigned int* __restrict__ work,
              int64_t q_begin, int64_t q_end, int q_stride, int q_phase, int K, int hash_mode, float bx, float by,
              float bz, float cell,
              uint32_t n, uint64_t M, unsigned long long* __restrict__ stats) {
    const int lane = lane_id();
    unsigned long long st_visits = 0, st_scanned = 0, st_boxes = 0, st_queries = 0, st_group = 0;
    static_assert(ES >= 0 && ES <= 33, "a row holds at most the 32 ranks of one register + the row number");
    // batched epilogue (ES > 0): [8 warps][kQueryBatch][ES] floats, a row = ES-1 ranks (>= K) + the row number; ES is
    // odd so that the lanes of the final pass (one query each) read distinct banks
    extern __shared__ float s_epi[];
    float* const epi = s_epi + (threadIdx.x >> 5) * (kQueryBatch * (ES > 0 ? ES : 1));
    // group path, per warp: the list (entry = chunk id << 5 | probe; chunk ids < 2^26), then the bucket hash of probe
    // p at glist[kGroupList + p], so that the group code can reload the probe boxes instead of keeping them live
    constexpr bool GROUP = knn_group_on<NREG, ES>();
    unsigned* const glist =
        reinterpret_cast<unsigned*>(s_epi + 8 * kQueryBatch * ES) + (threadIdx.x >> 5) * (kGroupList + 32);
    auto probe_box = [&](float& lx, float& ly, float& lz, float& hx, float& hy, float& hz) {   // lane < 27, pc > 0
        const size_t h = glist[kGroupList + lane];
        const float4 b0 = __ldg(tab_box + 2 * h), b1 = __ldg(tab_box + 2 * h + 1);
        lx = b0.x, ly = b0.y, lz = b0.z, hx = b1.x, hy = b1.y, hz = b1.z;
    };
#if GSX_KNN_TMA
    __shared__ __align__(128) float4 s_stage[8][kSmallBucket];
    __shared__ __align__(8) unsigned long long s_bar[8];
    float4* wbuf = s_stage[threadIdx.x >> 5];
    const uint32_t bar_addr = (uint32_t)__cvta_generic_to_shared(&s_bar[threadIdx.x >> 5]);
    uint32_t bar_phase = 0;
    int staged_s = -1, staged_c = 0;
    if (lane == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr) : "memory");
    __syncwarp();
#endif

    for (;;) {
#if GSX_KNN_PROFILE
        const long long prof_t0 = clock64();
        int prof_cls = 0;
#endif
        unsigned int b0 = 0;
        if (lane == 0) b0 = atomicAdd(work, (unsigned)kQueryBatch);
        b0 = __shfl_sync(GSX_FULL, b0, 0);
        // batch number b0/16 of THIS launch is global batch (b0/16)*q_stride + q_phase: with q_stride = number of ranks the
        // batches are dealt round-robin, so every rank samples the whole hash range (cost-balanced, see dist.py)
        int64_t qb = q_begin + ((int64_t)(b0 / kQueryBatch) * q_stride + q_phase) * kQueryBatch;
        if (qb >= q_end) break;
        int64_t qe = qb + kQueryBatch < q_end ? qb + kQueryBatch : q_end;
        // the 27 probes of a query depend only on its cell: consecutive hash-sorted queries mostly share
        // it, so the hashes and table entries are recomputed only when the cell changes
#if GSX_KNN_CELLBITS
        // one bit per sorted position (k_sor_finish): "another grid cell than the position before".  A batch is 16
        // consecutive positions inside one 32-bit word (kQueryBatch divides 32, batches are aligned to q_begin).
        const uint32_t cellword = __ldg(cellbits + (qb >> 5));
#else
        int cgx = 0x7fffffff, cgy = 0, cgz = 0;
#endif
        int ps = 0, pc = 0;                                  // lane p: bucket range of probe p
        float blx = 0.f, bly = 0.f, blz = 0.f, bhx = 0.f, bhy = 0.f, bhz = 0.f;  // and its bounding box
        const pos_t qb_p = (pos_t)qb, qe_p = (pos_t)qe;      // positions fit 31 bits (pos_t): 32-bit loop bookkeeping
#pragma unroll 1
        for (pos_t i = qb_p; i < qe_p; ++i) {
            float4 q = __ldg(spos + i);
#if GSX_KNN_CELLBITS
            const uint32_t w_i = (i >> 5) == (qb_p >> 5) ? cellword : __ldg(cellbits + (i >> 5));
            if (i == qb_p || ((w_i >> (i & 31)) & 1u)) {   // warp-uniform by construction
                const int gx = (int)floorf(__fdiv_rn(__fsub_rn(q.x, bx), cell));
                const int gy = (int)floorf(__fdiv_rn(__fsub_rn(q.y, by), cell));
                const int gz = (int)floorf(__fdiv_rn(__fsub_rn(q.z, bz), cell));
#else
            const int gx = (int)floorf(__fdiv_rn(__fsub_rn(q.x, bx), cell));
            const int gy = (int)floorf(__fdiv_rn(__fsub_rn(q.y, by), cell));
            const int gz = (int)floorf(__fdiv_rn(__fsub_rn(q.z, bz), cell));
#ifndef GSX_CELL_REUSE
#define GSX_CELL_REUSE 1
#endif
            // (vote makes the predicate provably warp-uniform: no reconvergence code in the loop below)
            if (!GSX_CELL_REUSE || __any_sync(GSX_FULL, gx != cgx || gy != cgy || gz != cgz)) {
                cgx = gx, cgy = gy, cgz = gz;
#endif
                ps = 0, pc = 0;
                if (lane < 27) {
                    // probe offsets of lane p<27 in the reference's loop order (dx outer, dz inner), computed here
                    // rather than held in registers through the query
                    unsigned pl;
                    asm volatile("mov.u32 %0, %%laneid;" : "=r"(pl));   // volatile: not hoisted out of the loop
                    const int pdx = (int)pl / 9 - 1, pdy = ((int)pl / 3) % 3 - 1, pdz = (int)pl % 3 - 1;
                    uint32_t h = probe_hash(gx + pdx, gy + pdy, gz + pdz, n, M, hash_mode);
                    if (GROUP) glist[kGroupList + lane] = h;
                    const int2 se = __ldg(tab_se + h);
                    ps = se.x;
                    pc = se.y - se.x;
                    if (pc > 0) {  // the box of an empty bucket is never written (and never read)
                        const float4 b0 = __ldg(tab_box + 2 * (size_t)h), b1 = __ldg(tab_box + 2 * (size_t)h + 1);
                        blx = b0.x, bly = b0.y, blz = b0.z, bhx = b1.x, bhy = b1.y, bhz = b1.z;
                    }
                }
#if GSX_KNN_TMA
                {   // stage the centre bucket of the new cell (if it is a small one) for the queries that share it
                    const int s13 = __shfl_sync(GSX_FULL, ps, 13), c13 = __shfl_sync(GSX_FULL, pc, 13);
                    staged_c = 0;
                    if (c13 > 0 && c13 <= kSmallBucket) {
                        __syncwarp();   // every lane is done with the previous contents of wbuf
                        if (lane == 0) {
                            const uint32_t bytes = (uint32_t)c13 * 16u;
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
                            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                             (uint32_t)__cvta_generic_to_shared(wbuf)),
                                         "l"(spos + s13), "r"(bytes), "r"(bar_addr)
                                         : "memory");
                        }
                        uint32_t ok = 0;
                        for (unsigned spin = 0; !ok && spin < (1u << 24); ++spin) {   // bounded: never hang the GPU
                            asm volatile(
                                "{\n\t.reg .pred p;\n\t"
                                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                                "selp.u32 %0, 1, 0, p;\n\t}"
                                : "=r"(ok)
                                : "r"(bar_addr), "r"(bar_phase)
                                : "memory");
                        }
                        bar_phase ^= 1u;
                        if (__all_sync(GSX_FULL, ok != 0)) {
                            staged_s = s13;
                            staged_c = c13;
                        }
                    }
                }
#endif
            }
#if GSX_KNN_PROFILE
            if (i == qb_p) {
                const int c13 = __shfl_sync(GSX_FULL, pc, 13);
                prof_cls = c13 <= kSmallBucket ? 0 : c13 <= 1024 ? 1 : c13 <= 16384 ? 2 : 3;
            }
#endif
#if GSX_KNN_CELLBITS
            if constexpr (GROUP) if (i == qb_p) {
                const int s13 = __shfl_sync(GSX_FULL, ps, 13), c13 = __shfl_sync(GSX_FULL, pc, 13);
                const pos_t ql = qe_p - 1;
                // positions qb+1 .. qe-1 of the cell word: a set bit = another cell than the position before
                const uint32_t later = ((2u << (ql & 31)) - 1u) & ~((2u << (qb_p & 31)) - 1u);
                if (c13 > kSmallBucket && qb_p >= s13 && qe_p <= (pos_t)s13 + c13 && (ql >> 5) == (qb_p >> 5) &&
                    (cellword & later) == 0u) {
                    // phase A: the seed list of every query (its own chunk, as the per-query path does), parked in
                    // the query's epilogue row; B = box of the batch, tau_G = largest seed tau
                    const int skip_chunk = (int)(qb_p >> 5);
                    const pos_t js = ((pos_t)skip_chunk << 5) + lane;
                    const bool jv = js >= s13 && js < (pos_t)s13 + c13;
                    float tau_g = 0.f;
                    float Blx = INFINITY, Bly = INFINITY, Blz = INFINITY, Bhx = -INFINITY, Bhy = -INFINITY,
                          Bhz = -INFINITY;
                    bool full = true;
#pragma unroll 1
                    for (pos_t t = qb_p; t < qe_p; ++t) {
                        const float4 qt = __ldg(spos + t);
                        TopK<NREG> tk;
                        tk.init(K);
                        scan32<NREG, STATS>(spos, js, jv, qt.x, qt.y, qt.z, tk, lane, st_scanned);
                        if (!(tk.tau < __uint_as_float(GSX_D2LIM_BITS))) {   // fewer than K candidates in the chunk
                            full = false;
                            break;
                        }
                        tau_g = fmaxf(tau_g, tk.tau);
                        Blx = fminf(Blx, qt.x), Bly = fminf(Bly, qt.y), Blz = fminf(Blz, qt.z);
                        Bhx = fmaxf(Bhx, qt.x), Bhy = fmaxf(Bhy, qt.y), Bhz = fmaxf(Bhz, qt.z);
                        if (lane < ES - 1) epi[(int)(t - qb_p) * ES + lane] = tk.v0;
                    }
                    // phase B: one walk for the batch.  The bound per axis is max(lo_box - hi_B, lo_B - hi_box, 0),
                    // then the op sequence of box_lb: <= box_lb(q, box) for every q in B.
                    auto lb_b = [&](float lx, float ly, float lz, float hx, float hy, float hz) {
                        const float dx = fmaxf(fmaxf(__fsub_rn(lx, Bhx), __fsub_rn(Blx, hx)), 0.f);
                        const float dy = fmaxf(fmaxf(__fsub_rn(ly, Bhy), __fsub_rn(Bly, hy)), 0.f);
                        const float dz = fmaxf(fmaxf(__fsub_rn(lz, Bhz), __fsub_rn(Blz, hz)), 0.f);
                        return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                    };
                    int cnt = 0;
                    auto append = [&](bool take, unsigned entry) {   // ballot compaction into the warp's list
                        const unsigned m = __ballot_sync(GSX_FULL, take);
                        const int at = cnt + __popc(m & ((1u << lane) - 1u));
                        if (take && at < kGroupList) glist[at] = entry;
                        cnt += __popc(m);
                    };
                    unsigned small = 0;   // probes whose (small) bucket passed the group bound
                    if (full) {
                        // a bucket reached by two probes is listed (and later scanned) twice, as in the per-query path
                        bool pt = false;
                        if (pc > 0) {
                            float lx, ly, lz, hx, hy, hz;
                            probe_box(lx, ly, lz, hx, hy, hz);
                            pt = lb_b(lx, ly, lz, hx, hy, hz) < tau_g;
                        }
                        small = __ballot_sync(GSX_FULL, pt && pc <= kSmallBucket);
                        unsigned lm = __ballot_sync(GSX_FULL, pt && pc > kSmallBucket);
                        while (lm && cnt <= kGroupList) {
                            const int p = __ffs(lm) - 1;
                            lm &= lm - 1;
                            const int s = __shfl_sync(GSX_FULL, ps, p), c = __shfl_sync(GSX_FULL, pc, p);
                            const int fc = s >> 5, lc = (s + c - 1) >> 5, fs = fc >> 5, ls = lc >> 5;
                            auto chunks = [&](const int cbase) {
                                const int cid = cbase + lane;
                                bool take = false;
                                if (cid >= fc && cid <= lc) {
                                    const float4 a = __ldg(caabb + 2 * cid), b = __ldg(caabb + 2 * cid + 1);
                                    take = lb_b(a.x, a.y, a.z, a.w, b.x, b.y) < tau_g;
                                }
                                if (STATS) st_boxes += __popc(__ballot_sync(GSX_FULL, cid >= fc && cid <= lc));
                                append(take, ((unsigned)cid << 5) | (unsigned)p);
                            };
                            if (GSX_KNN_FLAT_SUPERS > 0 && ls - fs < GSX_KNN_FLAT_SUPERS) {
                                for (int cb = fc; cb <= lc && cnt <= kGroupList; cb += 32) chunks(cb);
                                continue;
                            }
                            for (int sb = fs; sb <= ls && cnt <= kGroupList; sb += 32) {
                                const int sid = sb + lane;
                                bool take = false;
                                if (sid <= ls) {
                                    const float4 a = __ldg(saabb + 2 * sid), b = __ldg(saabb + 2 * sid + 1);
                                    take = lb_b(a.x, a.y, a.z, a.w, b.x, b.y) < tau_g;
                                }
                                if (STATS) st_boxes += __popc(__ballot_sync(GSX_FULL, sid <= ls));
                                unsigned sm = __ballot_sync(GSX_FULL, take);
                                while (sm && cnt <= kGroupList) {
                                    const int srcs = __ffs(sm) - 1;
                                    sm &= sm - 1;
                                    chunks((sb + srcs) * 32);
                                }
                            }
                        }
                    }
                    if (full && cnt <= kGroupList) {
                        __syncwarp();   // the list is read by other lanes than the ones that wrote it
                        // phase C: per query, its seed list back, then the listed chunks and the small buckets, each
                        // nearest box first
#pragma unroll 1
                        for (pos_t t = qb_p; t < qe_p; ++t) {
                            const float4 qt = __ldg(spos + t);
                            TopK<NREG> tk;
                            tk.init(K);
                            // ranks >= ES-1 >= K are never read: the sentinel keeps the list ascending
                            if (lane < ES - 1) tk.v0 = epi[(int)(t - qb_p) * ES + lane];
                            tk.refresh_tau();
#pragma unroll 1
                            for (int g0 = 0; g0 < cnt; g0 += 32) {
                                const bool ev = g0 + lane < cnt;
                                const unsigned ent = ev ? glist[g0 + lane] : 0u;
                                unsigned key = 0xffffffffu;
                                if (ev && ent != (((unsigned)(qb_p >> 5) << 5) | 13u)) {   // not the seed chunk
                                    const float lb = box_lb(caabb, (int)(ent >> 5), qt.x, qt.y, qt.z);
                                    if (lb < tk.tau) key = __float_as_uint(lb);
                                }
                                if (STATS) st_boxes += __popc(__ballot_sync(GSX_FULL, ev));
                                for (;;) {
                                    const unsigned mc = __reduce_min_sync(GSX_FULL, key);
                                    if (mc == 0xffffffffu || !(__uint_as_float(mc) < tk.tau)) break;
                                    const int src = __ffs(__ballot_sync(GSX_FULL, key == mc)) - 1;
                                    if (lane == src) key = 0xffffffffu;
                                    const unsigned e_src = __shfl_sync(GSX_FULL, ent, src);
                                    const int pp = (int)(e_src & 31u);
                                    const int s = __shfl_sync(GSX_FULL, ps, pp), c = __shfl_sync(GSX_FULL, pc, pp);
                                    const pos_t j = ((pos_t)(e_src >> 5) << 5) + lane;
                                    scan32<NREG, STATS>(spos, j, j >= s && j < (pos_t)s + c, qt.x, qt.y, qt.z, tk, lane,
                                                        st_scanned);
                                }
                            }
                            unsigned pkey = 0xffffffffu;
                            if ((small >> lane) & 1u) {
                                float blx, bly, blz, bhx, bhy, bhz;
                                probe_box(blx, bly, blz, bhx, bhy, bhz);
                                const float dx = fmaxf(fmaxf(__fsub_rn(blx, qt.x), __fsub_rn(qt.x, bhx)), 0.f);
                                const float dy = fmaxf(fmaxf(__fsub_rn(bly, qt.y), __fsub_rn(qt.y, bhy)), 0.f);
                                const float dz = fmaxf(fmaxf(__fsub_rn(blz, qt.z), __fsub_rn(qt.z, bhz)), 0.f);
                                pkey = __float_as_uint(
                                    __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
                            }
#pragma unroll 1
                            for (;;) {
                                const unsigned mp = __reduce_min_sync(GSX_FULL, pkey);
                                if (mp == 0xffffffffu || !(__uint_as_float(mp) < tk.tau)) break;
                                const int p = __ffs(__ballot_sync(GSX_FULL, pkey == mp)) - 1;
                                if (lane == p) pkey = 0xffffffffu;
                                const int s = __shfl_sync(GSX_FULL, ps, p), c = __shfl_sync(GSX_FULL, pc, p);
                                const pos_t e = (pos_t)s + c;
#pragma unroll 1
                                for (pos_t base = s; base < e; base += 32)
                                    scan32<NREG, STATS>(spos, base + lane, base + lane < e, qt.x, qt.y, qt.z, tk, lane,
                                                        st_scanned);
                            }
                            const float d0 = __fsqrt_rn(tk.v0);
                            float* row = epi + (int)(t - qb_p) * ES;
                            if (ES <= 32) {
                                if (lane < ES) row[lane] = lane == ES - 1 ? qt.w : d0;
                            } else {
                                row[lane] = d0;
                                if (lane == 0) row[ES - 1] = qt.w;
                            }
                        }
                        if (STATS) {
                            int tot = pc;
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(GSX_FULL, tot, o);
                            st_visits += (unsigned long long)tot * (unsigned long long)(qe_p - qb_p);
                            st_queries += (unsigned long long)(qe_p - qb_p);
                            st_group += (unsigned long long)(qe_p - qb_p);
                        }
                        break;   // the batched epilogue below sums the rows
                    }
                    // fallback to the per-query path: q and the probe boxes are reloaded, so that they are not live
                    // through the group code
                    q = __ldg(spos + i);
                    blx = bly = blz = bhx = bhy = bhz = 0.f;
                    if (lane < 27 && pc > 0) probe_box(blx, bly, blz, bhx, bhy, bhz);
                }
            }
#endif
            if (STATS) {
                int tot = pc;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(GSX_FULL, tot, o);
                st_visits += (unsigned long long)tot;
                st_queries += 1;
            }
            TopK<NREG> tk;
            tk.init(K);

            // lower bound of d^2 to the bucket's box (same monotone op sequence as d^2 itself, see box_lb):
            // probes are visited nearest box first and dropped as soon as lb >= tau.  The query's own bucket
            // has lb == 0 and therefore comes first whenever the centre probe reaches it.
            unsigned pkey = 0xffffffffu;
            if (pc > 0) {
                float dx = fmaxf(fmaxf(__fsub_rn(blx, q.x), __fsub_rn(q.x, bhx)), 0.f);
                float dy = fmaxf(fmaxf(__fsub_rn(bly, q.y), __fsub_rn(q.y, bhy)), 0.f);
                float dz = fmaxf(fmaxf(__fsub_rn(blz, q.z), __fsub_rn(q.z, bhz)), 0.f);
                pkey = __float_as_uint(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
            }

            // seed from the chunk that holds the query itself when its own bucket is big: gives a
            // tight tau before the box walk.  Only legal if the centre probe really reaches the
            // query's bucket range (with the wrapped hash it may not, SURVEY F8).
            int skip_chunk = -1;
            {
                int s13 = __shfl_sync(GSX_FULL, ps, 13), c13 = __shfl_sync(GSX_FULL, pc, 13);
                if (c13 > kSmallBucket && i >= s13 && i < (pos_t)s13 + c13) {
                    skip_chunk = (int)(i >> 5);
                    const pos_t j = ((pos_t)skip_chunk << 5) + lane;
                    scan32<NREG, STATS>(spos, j, j >= s13 && j < (pos_t)s13 + c13, q.x, q.y, q.z, tk, lane,
                                        st_scanned);
                }
            }

#pragma unroll 1
            for (;;) {
                const unsigned mp = __reduce_min_sync(GSX_FULL, pkey);
                if (mp == 0xffffffffu || !(__uint_as_float(mp) < tk.tau)) break;
                const int p = __ffs(__ballot_sync(GSX_FULL, pkey == mp)) - 1;
                if (lane == p) pkey = 0xffffffffu;
                const int s = __shfl_sync(GSX_FULL, ps, p), c = __shfl_sync(GSX_FULL, pc, p);
                const pos_t e = (pos_t)s + c;
                if (c <= kSmallBucket) {
#if GSX_KNN_TMA
                    const bool from_smem = staged_c > 0 && s == staged_s;   // warp-uniform
#pragma unroll 1
                    for (pos_t base = s; base < e; base += 32)
                        scan32<NREG, STATS>(spos, base + lane, base + lane < e, q.x, q.y, q.z, tk, lane, st_scanned,
                                            from_smem ? wbuf + (base - s) : nullptr);
#else
#pragma unroll 1
                    for (pos_t base = s; base < e; base += 32)
                        scan32<NREG, STATS>(spos, base + lane, base + lane < e, q.x, q.y, q.z, tk, lane, st_scanned);
#endif
                    continue;
                }
                const int skip = p == 13 ? skip_chunk : -1;
                const int fc = s >> 5, lc = (int)((e - 1) >> 5);
                const int fs = fc >> 5, ls = lc >> 5;
                // the 32 chunks cbase .. cbase+31: box test per lane, then nearest box first while it can still improve
                auto chunk_group = [&](const int cbase) {
                    const int cid = cbase + lane;
                    const bool cv = cid >= fc && cid <= lc && cid != skip;
                    unsigned ckey = 0xffffffffu;
                    if (cv) {
                        float lb = box_lb(caabb, cid, q.x, q.y, q.z);
                        if (lb < tk.tau) ckey = __float_as_uint(lb);
                    }
                    if (STATS) st_boxes += __popc(__ballot_sync(GSX_FULL, cv));
                    for (;;) {
                        unsigned mc = __reduce_min_sync(GSX_FULL, ckey);
                        if (mc == 0xffffffffu || !(__uint_as_float(mc) < tk.tau)) break;
                        int srcc = __ffs(__ballot_sync(GSX_FULL, ckey == mc)) - 1;
                        if (lane == srcc) ckey = 0xffffffffu;
                        const pos_t j = ((pos_t)(cbase + srcc) << 5) + lane;
                        scan32<NREG, STATS>(spos, j, j >= s && j < e, q.x, q.y, q.z, tk, lane, st_scanned);
                    }
                };
#if GSX_KNN_FLAT_SUPERS > 0
                // a bucket of a few supers: every super box is near the query (it sits in or next to this bucket), so
                // the super level prunes nothing -- test the chunk boxes directly, 32 at a time (exact either way: a
                // chunk is skipped only when its lower bound is >= the current tau, and tau never grows)
                if (ls - fs < GSX_KNN_FLAT_SUPERS) {
                    for (int cb = fc; cb <= lc; cb += 32) chunk_group(cb);
                    continue;
                }
#endif
                for (int sb = fs; sb <= ls; sb += 32) {
                    const int sid = sb + lane;
                    unsigned skey = 0xffffffffu;
                    if (sid <= ls) {
                        float lb = box_lb(saabb, sid, q.x, q.y, q.z);
                        if (lb < tk.tau) skey = __float_as_uint(lb);
                    }
                    if (STATS) st_boxes += __popc(__ballot_sync(GSX_FULL, sid <= ls));
                    for (;;) {
                        unsigned ms = __reduce_min_sync(GSX_FULL, skey);
                        if (ms == 0xffffffffu || !(__uint_as_float(ms) < tk.tau)) break;
                        int srcs = __ffs(__ballot_sync(GSX_FULL, skey == ms)) - 1;
                        if (lane == srcs) skey = 0xffffffffu;
                        chunk_group((sb + srcs) * 32);
                    }
                }
            }

            // gpu_ops.py:163-174: ascending serial float32 sum of the valid (< 0.9e10) distances.  The
            // list is ascending, so the valid entries are a prefix of the first K ranks.
            const float d0 = __fsqrt_rn(tk.v0), d1 = NREG == 2 ? __fsqrt_rn(tk.v1) : 0.f;
            if (ES > 0) {   // park the list: ranks 0..ES-2 (>= K of them) and the row number in the last slot
                float* row = epi + (int)(i - qb_p) * ES;
                if (ES <= 32) {
                    if (lane < ES) row[lane] = lane == ES - 1 ? q.w : d0;
                } else {   // ES == 33: all 32 ranks, the row number by lane 0
                    row[lane] = d0;
                    if (lane == 0) row[ES - 1] = q.w;
                }
                continue;
            }
            int valid = __popc(__ballot_sync(GSX_FULL, lane < K && d0 < 0.9e10f));
            if (NREG == 2) valid += __popc(__ballot_sync(GSX_FULL, lane + 32 < K && d1 < 0.9e10f));
            float sum = 0.f;
            for (int r = 0; r < valid; ++r) {
                float x = (NREG == 2 && r >= 32) ? __shfl_sync(GSX_FULL, d1, r - 32) : __shfl_sync(GSX_FULL, d0, r);
                sum = __fadd_rn(sum, x);
            }
            if (lane == 0) final_means[__float_as_int(q.w)] = valid > 0 ? __fdiv_rn(sum, (float)valid) : 0.f;
        }
        if (ES > 0) {
            __syncwarp();
            if (lane < (int)(qe_p - qb_p)) {   // lane q: the serial sum of query q, rank order, exactly as above
                const float* row = epi + lane * ES;
                float sum = 0.f;
                int valid = 0;
                for (int r = 0; r < K; ++r) {
                    const float x = row[r];
                    if (x < 0.9e10f) {
                        sum = __fadd_rn(sum, x);
                        ++valid;
                    }
                }
                final_means[__float_as_int(row[ES - 1])] = valid > 0 ? __fdiv_rn(sum, (float)valid) : 0.f;
            }
            __syncwarp();   // the next batch overwrites the rows (and the group list)
        }
#if GSX_KNN_PROFILE
        if (STATS && lane == 0) {
            atomicAdd(stats + 8 + prof_cls, (unsigned long long)(clock64() - prof_t0));
            atomicAdd(stats + 12 + prof_cls, (unsigned long long)(qe_p - qb_p));
        }
#endif
    }
    if (STATS && lane == 0) {
        atomicAdd(stats + 0, st_visits);
        atomicAdd(stats + 1, st_scanned);
        atomicAdd(stats + 2, st_boxes);
        atomicAdd(stats + 3, st_queries);
        atomicAdd(stats + 4, st_group);
    }
}

#ifndef GSX_KNN16
#define GSX_KNN16 0   // 1: K <= 16 goes to the two-queries-per-warp kernel (gsx_sor_knn16.cuh) -- an A/B variant, it
                      // measured SLOWER than the warp-per-query kernel (profiles/r02_knn16_variants.log)
#endif
#include "gsx_sor_knn16.cuh"

__global__ void k_fill_f32(float* p, int64_t n, float v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

template <int NREG, bool STATS, int ES>
static int launch_knn(SorWs& w, int64_t q_begin, int64_t q_end, int q_stride, int q_phase, int K, int hash_mode,
                      const float* bmin, float cell,
                      float* final_means, unsigned long long* stats, uint64_t M, int64_t want, cudaStream_t st) {
    int per_sm = 0;
    const size_t smem = knn_smem_bytes<NREG, ES>();
    GSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sor_knn<NREG, STATS, ES>, 256, smem));
    int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 4);  // persistent: exactly the resident CTAs
    if (grid > want) grid = want;
    if (grid < 1) grid = 1;
    k_sor_knn<NREG, STATS, ES><<<(int)grid, 256, smem, st>>>(w.spos, w.tab_se, w.tab_box, w.cellbits, w.caabb, w.saabb, final_means, w.counters,
                                                      q_begin, q_end, q_stride, q_phase, K, hash_mode, bmin[0], bmin[1],
                                                      bmin[2], cell,
                                                      (uint32_t)w.n, M, stats);
    return GSX_OK;
}

template <bool STATS>
static int launch_knn16(SorWs& w, int64_t q_begin, int64_t q_end, int q_stride, int q_phase, int K, int hash_mode,
                        const float* bmin, float cell, float* final_means, unsigned long long* stats, uint64_t M,
                        int64_t want, cudaStream_t st) {
    int per_sm = 0;
    GSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sor_knn16<STATS>, 256, 0));
    int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 4);
    want = (want + 1) / 2;   // a block takes 16 batches at a time, not 8
    if (grid > want) grid = want;
    if (grid < 1) grid = 1;
    k_sor_knn16<STATS><<<(int)grid, 256, 0, st>>>(w.spos, w.tab_se, w.tab_box, w.cellbits, w.caabb, w.saabb, final_means,
                                                  w.counters, q_begin, q_end, q_stride, q_phase, K, hash_mode, bmin[0],
                                                  bmin[1], bmin[2], cell, (uint32_t)w.n, M, stats);
    return GSX_OK;
}

// compile-time configuration of the query kernel (A/B variants differ only here): recorded next to every ncu capture
// and checked by bench.py before it uses a capture's instruction count for the roofline
#define GSX_STR2(x) #x
#define GSX_STR(x) GSX_STR2(x)
#if GSX_KNN_FLAT_SUPERS > 0
#define GSX_FLAT_INFO ";flat_supers=" GSX_STR(GSX_KNN_FLAT_SUPERS)
#else
#define GSX_FLAT_INFO ""
#endif
const char* sor_build_info() {
    return "knn=r03"
           ";group=" GSX_STR(GSX_KNN_GROUP) ";group_list=" GSX_STR(GSX_KNN_GROUP_LIST) ";profile=" GSX_STR(GSX_KNN_PROFILE)
           ";epi_smem=" GSX_STR(GSX_KNN_EPI_SMEM) ";first_sort=" GSX_STR(GSX_KNN_FIRST_SORT)
           ";query_batch=" GSX_STR(GSX_QUERY_BATCH) ";minblocks=" GSX_STR(GSX_KNN_MINBLOCKS)
           ";merge_threshold=" GSX_STR(GSX_MERGE_THRESHOLD) ";small_bucket=" GSX_STR(GSX_SMALL_BUCKET)
           GSX_FLAT_INFO ";knn16=" GSX_STR(GSX_KNN16) ";tma=" GSX_STR(GSX_KNN_TMA) ";i32=" GSX_STR(GSX_KNN_I32);
}

int sor_mean_dists(SorWs& w, int64_t q_begin, int64_t q_end, int q_stride, int q_phase, int k, int hash_mode,
                   const float* bmin, float cell,
                   float* final_means, unsigned long long* stats, cudaStream_t st) {
    GSX_NVTX("gsx::sor_mean_dists(k_sor_knn)");
    int64_t n = w.n;
    GSX_REQUIRE(k >= 1, GSX_ERR_ARG, "sor: k must be >= 1 (got %d)", k);
    GSX_REQUIRE(hash_mode == 0 || hash_mode == 1, GSX_ERR_ARG, "sor: bad hash_mode %d", hash_mode);
    GSX_REQUIRE(q_begin >= 0 && q_end <= n && q_begin <= q_end, GSX_ERR_ARG, "sor: bad query range");
    GSX_REQUIRE(q_stride >= 1 && q_phase >= 0 && q_phase < q_stride, GSX_ERR_ARG, "sor: bad query stride/phase");
    int K = k < 50 ? k : 50;  // gpu_ops.py:244
    if (q_end == q_begin) return GSX_OK;
    if (!(cell > 1e-8f)) {  // gpu_ops.py:175-176 (unreachable through the driver: cell >= 1e-4)
        GSX_REQUIRE(q_begin == 0 && q_end == n, GSX_ERR_UNSUPPORTED, "sor: degenerate cell with a query range");
        k_fill_f32<<<(int)((n + 255) / 256), 256, 0, st>>>(final_means, n, 0.f);
        GSX_KERNEL_CHECK();
        return GSX_OK;
    }
    GSX_CUDA_CHECK(cudaMemsetAsync(w.counters, 0, sizeof(unsigned int), st));
    uint64_t M = 0xFFFFFFFFFFFFFFFFull / (uint64_t)n + 1ull;
    int64_t nq = (q_end - q_begin + q_stride - 1) / q_stride + kQueryBatch;   // this launch's share (upper bound)
    int64_t want = (nq + (int64_t)kQueryBatch * 8 - 1) / ((int64_t)kQueryBatch * 8);
    int rc;
    if (GSX_KNN16 && K <= 16)
        rc = stats ? launch_knn16<true>(w, q_begin, q_end, q_stride, q_phase, K, hash_mode, bmin, cell, final_means, stats, M, want, st)
                   : launch_knn16<false>(w, q_begin, q_end, q_stride, q_phase, K, hash_mode, bmin, cell, final_means, stats, M, want, st);
    else {
#define GSX_KNN_ARGS w, q_begin, q_end, q_stride, q_phase, K, hash_mode, bmin, cell, final_means, stats, M, want, st
        // ES = row stride of the batched shared-memory epilogue (0: per-query shuffle epilogue)
        constexpr int ES16 = GSX_KNN_EPI_SMEM ? 17 : 0, ES32 = GSX_KNN_EPI_SMEM ? 33 : 0;
        if (K <= 16) rc = stats ? launch_knn<1, true, ES16>(GSX_KNN_ARGS) : launch_knn<1, false, ES16>(GSX_KNN_ARGS);
        else if (K <= 32) rc = stats ? launch_knn<1, true, ES32>(GSX_KNN_ARGS) : launch_knn<1, false, ES32>(GSX_KNN_ARGS);
        else rc = stats ? launch_knn<2, true, 0>(GSX_KNN_ARGS) : launch_knn<2, false, 0>(GSX_KNN_ARGS);
#undef GSX_KNN_ARGS
    }
    if (rc) return rc;
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

}  // namespace gsx
