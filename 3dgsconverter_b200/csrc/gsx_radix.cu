// gsx_radix.cu -- stable LSD radix sort of (uint64 key, int32 value) pairs, hand-written for sm_100a.
//
// Serves the hash-grid build (gpu_ops.py:227 `np.argsort(hashed)`; word = bucket | Morton code | index, keys only)
// and, as (key, value) pairs, the Morton orderings of the exact-KNN path and of compressed_ply / ksplat and the SOG
// lexsort.  8-bit digits.  Two forms of a pass: the onesweep form further down is the one used (see there); the
// three-kernel form takes over from n = GSX_RADIX_ONESWEEP_MAX_N (2^30: the onesweep look-back words carry 30-bit
// counts) up to its own limit n < 2^32 (32-bit offsets), and is the A/B baseline (-DGSX_RADIX_ONESWEEP=0):
//   k_rs_hist    per-tile digit histogram (tile = 4096 keys, one CTA)  -> hist[digit][tile]
//   exclusive scan of the digit-major matrix (multi-level block scan)   -> global base of (digit, tile)
//   k_rs_scatter per-tile stable ranks: every warp owns 512 consecutive keys, ranks them 32 at a time
//                with match.any on the digit + per-warp shared-memory counters, warps are chained by a
//                per-digit prefix over the 8 warps; the pairs are first placed in shared memory in locally
//                sorted order so that the final global writes are coalesced runs per digit.
// Only the bits [begin_bit, end_bit) are sorted (the hash needs ceil(log2 N) bits, not 32).
// HBM traffic per pass: 8 B (hist) + 12 B read + 12 B written per pair.
#include "gsx_common.cuh"
#include "gsx_radix.cuh"

namespace gsx {

#define GSX_FULL 0xffffffffu
#ifndef GSX_RADIX_ONESWEEP
#define GSX_RADIX_ONESWEEP 1
#endif
// onesweep sorts n < GSX_RADIX_ONESWEEP_MAX_N, the three-kernel passes everything above.  2^30 is the most the 30-bit
// count field of a look-back word can hold; a smaller value (a test build) runs the three-kernel passes at small n.
#ifndef GSX_RADIX_ONESWEEP_MAX_N
#define GSX_RADIX_ONESWEEP_MAX_N (1ll << 30)
#endif
static_assert(GSX_RADIX_ONESWEEP_MAX_N >= 1 && GSX_RADIX_ONESWEEP_MAX_N <= (1ll << 30),
              "onesweep look-back words hold 30-bit counts");
constexpr int64_t kRsMaxN = 1ll << 32;   // three-kernel passes: 32-bit histogram entries and scatter offsets
constexpr int kRsThreads = 256;
constexpr int kRsPerThread = 16;
constexpr int kRsTile = kRsThreads * kRsPerThread;  // 4096
constexpr int kRsWarpKeys = 32 * kRsPerThread;      // 512 consecutive keys per warp
constexpr int kScanBlock = 2048;                    // elements per scan CTA (256 threads x 8)

// ------------------------------------------------------------------ exclusive scan (uint32, in place)
__global__ void __launch_bounds__(256) k_scan_block(uint32_t* __restrict__ data, int64_t n,
                                                    uint32_t* __restrict__ sums) {
    const int64_t base = (int64_t)blockIdx.x * kScanBlock + (int64_t)threadIdx.x * 8;
    uint32_t v[8];
    uint32_t tsum = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        v[e] = base + e < n ? data[base + e] : 0u;
        tsum += v[e];
    }
    // exclusive scan of the 256 thread sums
    uint32_t x = tsum;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
        if (lane >= o) x += y;
    }
    __shared__ uint32_t wsum[8];
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (i < w) woff += wsum[i];
    uint32_t run = woff + x - tsum;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        if (base + e < n) data[base + e] = run;
        run += v[e];
    }
    if (threadIdx.x == 255 && sums) sums[blockIdx.x] = run;
}

__global__ void __launch_bounds__(256) k_scan_add(uint32_t* __restrict__ data, int64_t n,
                                                  const uint32_t* __restrict__ sums) {
    const uint32_t add = sums[blockIdx.x];
    const int64_t base = (int64_t)blockIdx.x * kScanBlock + (int64_t)threadIdx.x * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e)
        if (base + e < n) data[base + e] += add;
}

static size_t scan_ws_elems(int64_t n) {
    size_t tot = 0;
    while (n > kScanBlock) {
        n = (n + kScanBlock - 1) / kScanBlock;
        tot += (size_t)n + 64;
    }
    return tot + 64;
}

static int exclusive_scan_u32(uint32_t* data, int64_t n, uint32_t* ws, cudaStream_t st) {
    int64_t blocks = (n + kScanBlock - 1) / kScanBlock;
    if (blocks <= 1) {
        k_scan_block<<<1, 256, 0, st>>>(data, n, nullptr);
        GSX_KERNEL_CHECK();
        return GSX_OK;
    }
    k_scan_block<<<(unsigned)blocks, 256, 0, st>>>(data, n, ws);
    GSX_KERNEL_CHECK();
    int rc = exclusive_scan_u32(ws, blocks, ws + blocks + 64, st);
    if (rc) return rc;
    k_scan_add<<<(unsigned)blocks, 256, 0, st>>>(data, n, ws);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

size_t scan_workspace_bytes(int64_t n) { return scan_ws_elems(n) * sizeof(uint32_t); }
int exclusive_scan_u32_ws(uint32_t* data, int64_t n, uint32_t* ws, cudaStream_t st) {
    return exclusive_scan_u32(data, n, ws, st);
}

// ------------------------------------------------------------------ radix passes
__global__ void __launch_bounds__(kRsThreads) k_rs_hist(const uint64_t* __restrict__ keys, int64_t n, int shift,
                                                        int64_t ntiles, uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kRsTile;
#pragma unroll 4
    for (int e = 0; e < kRsPerThread; ++e) {
        int64_t i = base + (int64_t)e * kRsThreads + threadIdx.x;
        if (i < n) atomicAdd(&sh[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * ntiles + blockIdx.x] = sh[threadIdx.x];
}

// dynamic shared memory of k_rs_scatter: the tile's pairs (PAIRS = false: bare keys) in locally sorted order + counters
template <bool PAIRS>
constexpr size_t rs_scatter_smem() {
    return (size_t)kRsTile * (PAIRS ? 12 : 8) + (size_t)8 * 256 * 4 + 2 * 256 * 4;
}

template <bool PAIRS>
__global__ void __launch_bounds__(kRsThreads)
    k_rs_scatter(const uint64_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                 uint64_t* __restrict__ keys_out, int32_t* __restrict__ vals_out, int64_t n, int shift,
                 int64_t ntiles, const uint32_t* __restrict__ base_off) {
    extern __shared__ __align__(16) unsigned char rs_smem[];
    uint64_t* skeys = reinterpret_cast<uint64_t*>(rs_smem);                      // [kRsTile]
    int32_t* svals = reinterpret_cast<int32_t*>(rs_smem + (size_t)kRsTile * 8);  // [kRsTile] (PAIRS only)
    constexpr size_t kPairBytes = (size_t)kRsTile * (PAIRS ? 12 : 8);
    uint32_t(*wcnt)[256] = reinterpret_cast<uint32_t(*)[256]>(rs_smem + kPairBytes);  // [8][256]
    uint32_t* dstart = reinterpret_cast<uint32_t*>(rs_smem + kPairBytes + 8 * 256 * 4);  // [256]
    uint32_t* gbase = dstart + 256;                                                       // [256]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int t = threadIdx.x; t < 8 * 256; t += kRsThreads) (&wcnt[0][0])[t] = 0;
    __syncthreads();
    const int64_t tbase = (int64_t)blockIdx.x * kRsTile;
    const int64_t wbase = tbase + (int64_t)w * kRsWarpKeys;
    uint64_t key[kRsPerThread];
    uint32_t rank[kRsPerThread];  // stable rank of the key among equal digits of this warp
    // phase A: ranks inside the warp (index order: step-major, lane-minor)
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        key[e] = i < n ? keys_in[i] : 0ull;
    }
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        const bool act = i < n;
        const uint32_t d = act ? ((uint32_t)(key[e] >> shift) & 255u) : (256u + lane);  // unique when inactive
        const unsigned peers = __match_any_sync(GSX_FULL, d);
        const uint32_t before = act ? wcnt[w][d] : 0u;
        rank[e] = before + __popc(peers & ((1u << lane) - 1u));
        __syncwarp();
        if (act && (peers & ((1u << lane) - 1u)) == 0u) wcnt[w][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // phase B: digit d = thread d: tile count, per-warp exclusive offsets, global base
    uint32_t dcount;
    {
        const int d = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) {
            uint32_t c = wcnt[ww][d];
            wcnt[ww][d] = run;
            run += c;
        }
        dcount = run;
        gbase[d] = base_off[(size_t)d * ntiles + blockIdx.x];
    }
    // exclusive scan of the 256 digit counts -> start of each digit in the locally sorted tile
    {
        uint32_t x = dcount;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
            if (lane >= o) x += y;
        }
        __shared__ uint32_t wtot[8];
        if (lane == 31) wtot[w] = x;
        __syncthreads();
        uint32_t woff = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < w) woff += wtot[i];
        dstart[threadIdx.x] = woff + x - dcount;
    }
    __syncthreads();
    // phase C: pairs into shared memory in locally sorted (digit-major, stable) order
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        if (i < n) {
            const uint32_t d = (uint32_t)(key[e] >> shift) & 255u;
            const uint32_t lp = dstart[d] + wcnt[w][d] + rank[e];
            skeys[lp] = key[e];
            if (PAIRS) svals[lp] = vals_in[i];
        }
    }
    __syncthreads();
    // phase D: coalesced write-out: consecutive threads hold consecutive elements of a digit run
    const int cnt = (int)(n - tbase < kRsTile ? n - tbase : kRsTile);
    for (int j = threadIdx.x; j < cnt; j += kRsThreads) {
        const uint64_t k = skeys[j];
        const uint32_t d = (uint32_t)(k >> shift) & 255u;
        const uint32_t pos = gbase[d] + ((uint32_t)j - dstart[d]);
        keys_out[pos] = k;
        if (PAIRS) vals_out[pos] = svals[j];
    }
}

// ------------------------------------------------------------------ onesweep passes (decoupled look-back)
// The three-kernel pass above reads every key twice (histogram, scatter) and round-trips a [256 x tiles] matrix
// through a multi-level scan.  The onesweep form reads the keys ONCE per pass:
//   k_os_hist   one pass over the keys: the GLOBAL digit histograms of all passes at once (shared-memory atomics,
//               then one global atomic per (pass, digit) per block);  k_os_scan makes them exclusive.
//   k_os_pass   a tile takes its id from an atomic counter (so every lower-numbered tile is already running),
//               ranks its 4096 keys exactly like k_rs_scatter, publishes its 256 digit counts and obtains the counts
//               of all lower tiles by looking back over the published words -- thread d follows digit d.
//               A word = count | flag (bit 30: tile aggregate, bit 31: inclusive prefix); it is a single 32-bit
//               store, so flag and payload cannot be seen apart.  The wait for a predecessor is bounded (trap).
// HBM traffic per pass: 8 (+4) B read + 8 (+4) B written per key (+ 8 B once for the histograms); the look-back
// words are 1 KiB per tile per pass.  PAIRS = false sorts bare 64-bit words (the grid build packs the point index
// into the low bits of its key).
constexpr uint32_t kOsAgg = 1u << 30, kOsInc = 1u << 31, kOsVal = (1u << 30) - 1u;
constexpr int kOsMaxPass = 8;
constexpr uint32_t kOsSpinLimit = 1u << 22;

__global__ void __launch_bounds__(256) k_os_hist(const uint64_t* __restrict__ keys, int64_t n, int begin_bit,
                                                  int npass, uint32_t* __restrict__ ghist) {
    __shared__ uint32_t sh[kOsMaxPass * 256];
    for (int t = threadIdx.x; t < npass * 256; t += 256) sh[t] = 0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const uint64_t k = keys[i] >> begin_bit;
        for (int p = 0; p < npass; ++p) atomicAdd(&sh[p * 256 + ((uint32_t)(k >> (8 * p)) & 255u)], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < npass * 256; t += 256)
        if (sh[t]) atomicAdd(&ghist[t], sh[t]);
}

// exclusive scan of each pass's 256 bins (block p = pass p)
__global__ void __launch_bounds__(256) k_os_scan(uint32_t* __restrict__ ghist) {
    uint32_t* h = ghist + blockIdx.x * 256;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t v = h[threadIdx.x];
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
        if (lane >= o) x += y;
    }
    __shared__ uint32_t wt[8];
    if (lane == 31) wt[w] = x;
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (i < w) woff += wt[i];
    h[threadIdx.x] = woff + x - v;
}

template <bool PAIRS>
constexpr size_t os_pass_smem() {
    return (size_t)kRsTile * (PAIRS ? 12 : 8) + (size_t)8 * 256 * 4 + 2 * 256 * 4;
}

template <bool PAIRS>
__global__ void __launch_bounds__(kRsThreads, PAIRS ? 3 : 4)
    k_os_pass(const uint64_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in, uint64_t* __restrict__ keys_out,
              int32_t* __restrict__ vals_out, int64_t n, int shift, const uint32_t* __restrict__ gbase_pass,
              uint32_t* lookback, unsigned int* tile_counter) {
    extern __shared__ __align__(16) unsigned char rs_smem[];
    uint64_t* skeys = reinterpret_cast<uint64_t*>(rs_smem);                      // [kRsTile]
    int32_t* svals = reinterpret_cast<int32_t*>(rs_smem + (size_t)kRsTile * 8);  // [kRsTile] (PAIRS only)
    constexpr size_t kPairBytes = (size_t)kRsTile * (PAIRS ? 12 : 8);
    uint32_t(*wcnt)[256] = reinterpret_cast<uint32_t(*)[256]>(rs_smem + kPairBytes);  // [8][256]
    uint32_t* dstart = reinterpret_cast<uint32_t*>(rs_smem + kPairBytes + 8 * 256 * 4);  // [256]
    uint32_t* gbase = dstart + 256;                                                       // [256]
    __shared__ unsigned int s_tile;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
    for (int t = threadIdx.x; t < 8 * 256; t += kRsThreads) (&wcnt[0][0])[t] = 0;
    __syncthreads();
    const unsigned int tile = s_tile;
    const int64_t tbase = (int64_t)tile * kRsTile;
    const int64_t wbase = tbase + (int64_t)w * kRsWarpKeys;
    uint64_t key[kRsPerThread];
    uint32_t rank2[kRsPerThread / 2];   // two 16-bit stable ranks per word (a rank is < 4096)
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        key[e] = i < n ? keys_in[i] : 0ull;
    }
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        const bool act = i < n;
        const uint32_t d = act ? ((uint32_t)(key[e] >> shift) & 255u) : (256u + lane);
        const unsigned peers = __match_any_sync(GSX_FULL, d);
        const uint32_t before = act ? wcnt[w][d] : 0u;
        const uint32_t r = before + __popc(peers & ((1u << lane) - 1u));
        if (e & 1) rank2[e >> 1] |= r << 16;
        else rank2[e >> 1] = r;
        __syncwarp();
        if (act && (peers & ((1u << lane) - 1u)) == 0u) wcnt[w][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // digit d = thread d: tile count -> publish -> look back -> global base of this tile's run of digit d
    uint32_t dcount;
    {
        const int d = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) {
            uint32_t c = wcnt[ww][d];
            wcnt[ww][d] = run;
            run += c;
        }
        dcount = run;
        volatile uint32_t* lb = lookback;
        lb[(size_t)tile * 256 + d] = dcount | (tile == 0 ? kOsInc : kOsAgg);
        uint32_t excl = 0;
        for (int64_t t = (int64_t)tile - 1; t >= 0; --t) {
            uint32_t v, spins = 0;
            while (((v = lb[(size_t)t * 256 + d]) & (kOsAgg | kOsInc)) == 0u)
                if (++spins > kOsSpinLimit) __trap();   // a lower tile is always resident: this cannot wait forever
            excl += v & kOsVal;
            if (v & kOsInc) break;
        }
        if (tile != 0) lb[(size_t)tile * 256 + d] = (excl + dcount) | kOsInc;
        gbase[d] = gbase_pass[d] + excl;
    }
    {
        uint32_t x = dcount;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(GSX_FULL, x, o);
            if (lane >= o) x += y;
        }
        __shared__ uint32_t wtot[8];
        if (lane == 31) wtot[w] = x;
        __syncthreads();
        uint32_t woff = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < w) woff += wtot[i];
        dstart[threadIdx.x] = woff + x - dcount;
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < kRsPerThread; ++e) {
        const int64_t i = wbase + e * 32 + lane;
        if (i < n) {
            const uint32_t d = (uint32_t)(key[e] >> shift) & 255u;
            const uint32_t lp = dstart[d] + wcnt[w][d] + ((rank2[e >> 1] >> (16 * (e & 1))) & 0xffffu);
            skeys[lp] = key[e];
            if (PAIRS) svals[lp] = vals_in[i];
        }
    }
    __syncthreads();
    const int cnt = (int)(n - tbase < kRsTile ? n - tbase : kRsTile);
    for (int j = threadIdx.x; j < cnt; j += kRsThreads) {
        const uint64_t k = skeys[j];
        const uint32_t d = (uint32_t)(k >> shift) & 255u;
        const uint32_t pos = gbase[d] + ((uint32_t)j - dstart[d]);
        keys_out[pos] = k;
        if (PAIRS) vals_out[pos] = svals[j];
    }
}

static size_t os_ws_elems(int64_t n) {   // histograms + tile counters + look-back words of up to kOsMaxPass passes
    const int64_t ntiles = (n + kRsTile - 1) / kRsTile;
    return (size_t)kOsMaxPass * 256 + 64 + (size_t)kOsMaxPass * 256 * ntiles;
}

template <bool PAIRS>
static int onesweep_sort(uint64_t* keys0, uint64_t* keys1, int32_t* vals0, int32_t* vals1, int64_t n, int begin_bit,
                         int end_bit, uint32_t* ws, uint64_t** keys_sorted, int32_t** vals_sorted, cudaStream_t st) {
    const int64_t ntiles = (n + kRsTile - 1) / kRsTile;
    const int npass = (end_bit - begin_bit + 7) / 8;
    uint32_t* ghist = ws;                                  // [kOsMaxPass][256]
    unsigned int* counters = ws + kOsMaxPass * 256;        // [kOsMaxPass] tile counters (64 reserved)
    uint32_t* lookback = ws + kOsMaxPass * 256 + 64;       // [npass][ntiles][256]
    GSX_CUDA_CHECK(cudaMemsetAsync(ws, 0, ((size_t)kOsMaxPass * 256 + 64 + (size_t)npass * 256 * ntiles) * sizeof(uint32_t), st));
    static int hist_blocks = 0;
    if (!hist_blocks) {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        hist_blocks = sms * 8;
    }
    int64_t hb = (n + 255) / 256;
    if (hb > hist_blocks) hb = hist_blocks;
    k_os_hist<<<(unsigned)hb, 256, 0, st>>>(keys0, n, begin_bit, npass, ghist);
    GSX_KERNEL_CHECK();
    k_os_scan<<<npass, 256, 0, st>>>(ghist);
    GSX_KERNEL_CHECK();
    GSX_CUDA_CHECK(cudaFuncSetAttribute(k_os_pass<PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)os_pass_smem<PAIRS>()));
    uint64_t *kin = keys0, *kout = keys1;
    int32_t *vin = vals0, *vout = vals1;
    for (int p = 0; p < npass; ++p) {
        k_os_pass<PAIRS><<<(unsigned)ntiles, kRsThreads, os_pass_smem<PAIRS>(), st>>>(
            kin, vin, kout, vout, n, begin_bit + 8 * p, ghist + p * 256, lookback + (size_t)p * 256 * ntiles, counters + p);
        GSX_KERNEL_CHECK();
        uint64_t* tk = kin;
        kin = kout;
        kout = tk;
        int32_t* tv = vin;
        vin = vout;
        vout = tv;
    }
    *keys_sorted = kin;
    if (vals_sorted) *vals_sorted = vin;
    return GSX_OK;
}

size_t radix_ws_bytes(int64_t n) {
    if (n < 1) n = 1;
    int64_t ntiles = (n + kRsTile - 1) / kRsTile;
    size_t hist = (size_t)256 * ntiles;
    size_t three_kernel = hist + scan_ws_elems((int64_t)hist) + 256;
    size_t onesweep = os_ws_elems(n);
    return (three_kernel > onesweep ? three_kernel : onesweep) * sizeof(uint32_t);
}

template <bool PAIRS>
static int three_kernel_sort(uint64_t* keys0, uint64_t* keys1, int32_t* vals0, int32_t* vals1, int64_t n, int begin_bit,
                             int end_bit, void* ws, uint64_t** keys_sorted, int32_t** vals_sorted, cudaStream_t st) {
    const int64_t ntiles = (n + kRsTile - 1) / kRsTile;
    uint32_t* hist = (uint32_t*)ws;
    uint32_t* scan_ws = hist + (size_t)256 * ntiles;
    GSX_CUDA_CHECK(cudaFuncSetAttribute(k_rs_scatter<PAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)rs_scatter_smem<PAIRS>()));
    uint64_t *kin = keys0, *kout = keys1;
    int32_t *vin = vals0, *vout = vals1;
    for (int shift = begin_bit; shift < end_bit; shift += 8) {
        k_rs_hist<<<(unsigned)ntiles, kRsThreads, 0, st>>>(kin, n, shift, ntiles, hist);
        GSX_KERNEL_CHECK();
        int rc = exclusive_scan_u32(hist, (int64_t)256 * ntiles, scan_ws, st);
        if (rc) return rc;
        k_rs_scatter<PAIRS><<<(unsigned)ntiles, kRsThreads, rs_scatter_smem<PAIRS>(), st>>>(kin, vin, kout, vout, n,
                                                                                             shift, ntiles, hist);
        GSX_KERNEL_CHECK();
        uint64_t* tk = kin;
        kin = kout;
        kout = tk;
        int32_t* tv = vin;
        vin = vout;
        vout = tv;
    }
    *keys_sorted = kin;
    if (vals_sorted) *vals_sorted = vin;
    return GSX_OK;
}

int radix_sort_pairs(uint64_t* keys0, uint64_t* keys1, int32_t* vals0, int32_t* vals1, int64_t n, int begin_bit,
                     int end_bit, void* ws, size_t ws_bytes, uint64_t** keys_sorted, int32_t** vals_sorted,
                     cudaStream_t st) {
    GSX_NVTX("gsx::radix_sort_pairs");
    GSX_REQUIRE(n >= 1 && n < kRsMaxN, GSX_ERR_ARG, "radix: n out of range");
    GSX_REQUIRE(ws_bytes >= radix_ws_bytes(n), GSX_ERR_WORKSPACE, "radix: workspace too small");
    GSX_REQUIRE(begin_bit >= 0 && end_bit <= 64 && begin_bit < end_bit, GSX_ERR_ARG, "radix: bad bit range");
    // GSX_RADIX_ONESWEEP=0 builds keep the three-kernel passes at every n for the A/B in profiles/
    if (GSX_RADIX_ONESWEEP && n < GSX_RADIX_ONESWEEP_MAX_N)
        return onesweep_sort<true>(keys0, keys1, vals0, vals1, n, begin_bit, end_bit, (uint32_t*)ws, keys_sorted,
                                   vals_sorted, st);
    return three_kernel_sort<true>(keys0, keys1, vals0, vals1, n, begin_bit, end_bit, ws, keys_sorted, vals_sorted, st);
}

int radix_sort_keys(uint64_t* keys0, uint64_t* keys1, int64_t n, int begin_bit, int end_bit, void* ws, size_t ws_bytes,
                    uint64_t** keys_sorted, cudaStream_t st) {
    GSX_NVTX("gsx::radix_sort_keys");
    GSX_REQUIRE(n >= 1 && n < kRsMaxN, GSX_ERR_ARG, "radix: n out of range");
    GSX_REQUIRE(ws_bytes >= radix_ws_bytes(n), GSX_ERR_WORKSPACE, "radix: workspace too small");
    GSX_REQUIRE(begin_bit >= 0 && end_bit <= 64 && begin_bit < end_bit, GSX_ERR_ARG, "radix: bad bit range");
    if (n < GSX_RADIX_ONESWEEP_MAX_N)
        return onesweep_sort<false>(keys0, keys1, nullptr, nullptr, n, begin_bit, end_bit, (uint32_t*)ws, keys_sorted,
                                    nullptr, st);
    return three_kernel_sort<false>(keys0, keys1, nullptr, nullptr, n, begin_bit, end_bit, ws, keys_sorted, nullptr, st);
}

}  // namespace gsx
