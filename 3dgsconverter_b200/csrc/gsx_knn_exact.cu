// gsx_knn_exact.cu -- SOR with the reference's CPU-path semantics (exact KNN, float64) on sm_100a.
//
// Replaces /root/reference/gsconverter/processing/data_processor.py:155-173: scipy cKDTree over the
// float32 coordinates promoted to float64, query k+1 nearest (the first is the point itself or a
// coincident twin), mean of neighbours 1..k in float64 (NumPy's pairwise row reduction), stored as
// float32.  SURVEY Appendix A.2.  The threshold/mask step (:176-180) is gsx_mean_std_f32 +
// gsx_threshold_mask, shared with the Taichi-semantics path.
//
// cKDTree's distance is sqrt(((dx*dx)+(dy*dy))+(dz*dz)) in float64 without fma (verified against SciPy
// in tests); only the multiset of the k+1 smallest values matters, so any exact search gives the same
// bits.  Search structure: points sorted by a 48-bit Morton code; bounding boxes over aligned runs of
// 32 / 1024 / 32768 / 1048576 sorted points; one warp per query walks the 4-level hierarchy nearest
// box first and prunes with lb >= tau, where lb is evaluated with the same monotone float64 op
// sequence as d^2 (so lb <= d^2 of every point in the box, exactly).
#include "../../include/gsx.h"
#include "gsx_common.cuh"
#include "gsx_knn_exact.cuh"
#include "gsx_sor.cuh"

#include "gsx_radix.cuh"
#include <math.h>

namespace gsx {

#define GSX_FULL 0xffffffffu
constexpr int kExLevels = 4;  // 32^1 .. 32^4 points per box

struct ExWs {
    int64_t n;
    uint64_t *keys0, *keys1;
    int32_t *vals0, *vals1;
    float4* spos;
    float4* box[kExLevels];
    int64_t cnt[kExLevels];
    float* partial;
    float* minmax;
    unsigned int* counters;
    char* sort_ws;
    size_t sort_ws_bytes;
    size_t total;
    bool ok;
};

static size_t ex_sort_ws_bytes(int64_t n) { return radix_ws_bytes(n) + 256; }

static ExWs ex_carve(void* ws, size_t bytes, int64_t n, size_t sort_ws_bytes) {
    ExWs w;
    Carver c(ws, bytes);
    w.n = n;
    w.keys0 = c.take<uint64_t>(n);
    w.keys1 = c.take<uint64_t>(n);
    w.vals0 = c.take<int32_t>(n);
    w.vals1 = c.take<int32_t>(n);
    w.spos = c.take<float4>(n);
    int64_t m = n;
    for (int l = 0; l < kExLevels; ++l) {
        m = (m + 31) / 32;
        w.cnt[l] = m;
        w.box[l] = c.take<float4>(2 * m);
    }
    w.partial = c.take<float>(6 * 1024);
    w.minmax = c.take<float>(8);
    w.counters = c.take<unsigned int>(64);
    w.sort_ws_bytes = sort_ws_bytes;
    w.sort_ws = c.take<char>(sort_ws_bytes);
    w.total = align_up(c.off, 256);
    w.ok = c.ok();
    return w;
}

int64_t knn_exact_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    ExWs w = ex_carve(nullptr, 0, n, ex_sort_ws_bytes(n));
    return (int64_t)w.total + 1024;
}

__device__ __forceinline__ uint64_t spread16(uint32_t v) {  // 16 bits -> every third bit of 48
    uint64_t x = v & 0xffffu;
    x = (x | (x << 16)) & 0x0000ff0000ffull;
    x = (x | (x << 8)) & 0x00f00f00f00full;
    x = (x | (x << 4)) & 0x0c30c30c30c3ull;
    x = (x | (x << 2)) & 0x249249249249ull;
    return x;
}

__global__ void __launch_bounds__(256) k_ex_keys(const float* __restrict__ xyz, int64_t n, float bx, float by,
                                                 float bz, float sx, float sy, float sz,
                                                 uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // ordering only: any monotone quantisation works
    uint32_t qx = (uint32_t)fminf(65535.f, fmaxf(0.f, (xyz[3 * i] - bx) * sx));
    uint32_t qy = (uint32_t)fminf(65535.f, fmaxf(0.f, (xyz[3 * i + 1] - by) * sy));
    uint32_t qz = (uint32_t)fminf(65535.f, fmaxf(0.f, (xyz[3 * i + 2] - bz) * sz));
    keys[i] = (spread16(qx) << 2) | (spread16(qy) << 1) | spread16(qz);
    vals[i] = (int32_t)i;
}

// gather into sorted float4 (w = original index) + level-0 boxes (one warp = one chunk of 32)
__global__ void __launch_bounds__(256) k_ex_gather(const float* __restrict__ xyz, const int32_t* __restrict__ order,
                                                   int64_t n, float4* __restrict__ spos, float4* __restrict__ box0) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (j < n) {
        int32_t idx = order[j];
        float x = xyz[3 * (int64_t)idx], y = xyz[3 * (int64_t)idx + 1], z = xyz[3 * (int64_t)idx + 2];
        spos[j] = make_float4(x, y, z, __int_as_float(idx));
        lo[0] = hi[0] = x, lo[1] = hi[1] = y, lo[2] = hi[2] = z;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(GSX_FULL, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(GSX_FULL, hi[a], o));
        }
    int64_t chunk = j >> 5;
    if ((threadIdx.x & 31) == 0 && chunk * 32 < n) {
        box0[2 * chunk] = make_float4(lo[0], lo[1], lo[2], hi[0]);
        box0[2 * chunk + 1] = make_float4(hi[1], hi[2], 0.f, 0.f);
    }
}

// level l+1 boxes from level l boxes (one warp reduces 32 children)
__global__ void __launch_bounds__(256) k_ex_boxes_up(const float4* __restrict__ child, int64_t nchild,
                                                     float4* __restrict__ parent, int64_t nparent) {
    int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (wid >= nparent) return;
    int64_t c = wid * 32 + lane;
    float v[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
    if (c < nchild) {
        float4 a = child[2 * c], b = child[2 * c + 1];
        v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y;
    }
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float t = __shfl_xor_sync(GSX_FULL, v[a], o);
            v[a] = a < 3 ? fminf(v[a], t) : fmaxf(v[a], t);
        }
    if (lane == 0) {
        parent[2 * wid] = make_float4(v[0], v[1], v[2], v[3]);
        parent[2 * wid + 1] = make_float4(v[4], v[5], 0.f, 0.f);
    }
}

// ------------------------------------------------------------------------------------- query
__device__ __forceinline__ double shfl_d(double v, int src) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_sync(GSX_FULL, lo, src);
    hi = __shfl_sync(GSX_FULL, hi, src);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_up_d(double v, int d) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_up_sync(GSX_FULL, lo, d);
    hi = __shfl_up_sync(GSX_FULL, hi, d);
    return __hiloint2double(hi, lo);
}

struct TopK64 {  // ascending list of the KK smallest d^2 (float64), rank r in lane r&31 of v[r>>5]
    double v0, v1, tau;
    int KK;
    __device__ __forceinline__ void init(int kk) {
        KK = kk;
        v0 = v1 = tau = __longlong_as_double(0x7ff0000000000000ll);  // +inf: "no neighbour" like cKDTree
    }
    __device__ __forceinline__ void insert(double x, int lane) {
        double up0 = shfl_up_d(v0, 1), top0 = shfl_d(v0, 31), up1 = shfl_up_d(v1, 1);
        if (lane == 0) up1 = top0, up0 = -1.0;
        if (v1 > x) v1 = fmax(up1, x);
        if (v0 > x) v0 = fmax(up0, x);
        tau = KK > 32 ? shfl_d(v1, KK - 33) : shfl_d(v0, KK - 1);
    }
};

__device__ __forceinline__ double box_lb_d(const float4* __restrict__ box, int64_t id, double qx, double qy,
                                           double qz) {
    float4 a = __ldg(box + 2 * id), b = __ldg(box + 2 * id + 1);
    double dx = fmax(fmax(__dsub_rn((double)a.x, qx), __dsub_rn(qx, (double)a.w)), 0.0);
    double dy = fmax(fmax(__dsub_rn((double)a.y, qy), __dsub_rn(qy, (double)b.x)), 0.0);
    double dz = fmax(fmax(__dsub_rn((double)a.z, qz), __dsub_rn(qz, (double)b.y)), 0.0);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

__device__ __forceinline__ void scan_chunk_d(const float4* __restrict__ spos, int64_t chunk, int64_t n, double qx,
                                             double qy, double qz, TopK64& tk, int lane) {
    int64_t j = chunk * 32 + lane;
    double d2 = __longlong_as_double(0x7ff0000000000000ll);
    bool valid = j < n;
    if (valid) {
        float4 c = __ldg(spos + j);
        double ax = __dsub_rn(qx, (double)c.x), ay = __dsub_rn(qy, (double)c.y), az = __dsub_rn(qz, (double)c.z);
        d2 = __dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az));
    }
    unsigned m = __ballot_sync(GSX_FULL, valid && d2 < tk.tau);
    while (m) {
        int src = __ffs(m) - 1;
        m &= m - 1;
        double x = shfl_d(d2, src);
        if (x < tk.tau) tk.insert(x, lane);
    }
}

struct ExTree {
    const float4* spos;
    const float4* box[kExLevels];
    int64_t cnt[kExLevels];
    int64_t n;
};

// visit the (up to 32) children of node `node` at level LEVEL (children live at LEVEL-1; level 0
// children are points), nearest child first, pruning with lb >= tau
template <int LEVEL>
__device__ __forceinline__ void visit(const ExTree& t, int64_t node, int64_t skip_chunk, double qx, double qy,
                                      double qz, TopK64& tk, int lane) {
    if constexpr (LEVEL == 0) {
        if (node != skip_chunk) scan_chunk_d(t.spos, node, t.n, qx, qy, qz, tk, lane);
    } else {
        const int64_t child = node * 32 + lane;
        unsigned key = 0xffffffffu;
        if (child < t.cnt[LEVEL - 1] && !(LEVEL == 1 && child == skip_chunk)) {
            double lb = box_lb_d(t.box[LEVEL - 1], child, qx, qy, qz);
            if (lb < tk.tau) key = __float_as_uint(__double2float_rd(lb));  // order only; pruning uses lb itself
        }
        for (;;) {
            unsigned mk = __reduce_min_sync(GSX_FULL, key);
            if (mk == 0xffffffffu) break;
            int src = __ffs(__ballot_sync(GSX_FULL, key == mk)) - 1;
            if (lane == src) key = 0xffffffffu;
            // re-test the chosen child against the (possibly smaller) tau with its exact float64 bound
            const int64_t cid = node * 32 + src;
            double lbc = box_lb_d(t.box[LEVEL - 1], cid, qx, qy, qz);
            if (!(lbc < tk.tau)) continue;
            visit<LEVEL - 1>(t, cid, skip_chunk, qx, qy, qz, tk, lane);
        }
    }
}

__global__ void __launch_bounds__(256, 4)
    k_knn_exact(ExTree t, float* __restrict__ out_means, unsigned int* __restrict__ work, int k) {
    const int lane = threadIdx.x & 31;
    const int KK = k + 1;
    for (;;) {
        unsigned int b0 = 0;
        if (lane == 0) b0 = atomicAdd(work, 8u);
        b0 = __shfl_sync(GSX_FULL, b0, 0);
        if ((int64_t)b0 >= t.n) break;
        int64_t qe = (int64_t)b0 + 8 < t.n ? (int64_t)b0 + 8 : t.n;
#pragma unroll 1
        for (int64_t i = b0; i < qe; ++i) {
            const float4 q = __ldg(t.spos + i);
            const double qx = (double)q.x, qy = (double)q.y, qz = (double)q.z;
            TopK64 tk;
            tk.init(KK);
            const int64_t own = i >> 5;
            scan_chunk_d(t.spos, own, t.n, qx, qy, qz, tk, lane);  // contains the query itself (d = 0)
            // top level: groups of 32 level-3 boxes
            for (int64_t g = 0; g < t.cnt[kExLevels - 1]; g += 32) {
                const int64_t node = g + lane;
                unsigned key = 0xffffffffu;
                if (node < t.cnt[kExLevels - 1]) {
                    double lb = box_lb_d(t.box[kExLevels - 1], node, qx, qy, qz);
                    if (lb < tk.tau) key = __float_as_uint(__double2float_rd(lb));
                }
                for (;;) {
                    unsigned mk = __reduce_min_sync(GSX_FULL, key);
                    if (mk == 0xffffffffu) break;
                    int src = __ffs(__ballot_sync(GSX_FULL, key == mk)) - 1;
                    if (lane == src) key = 0xffffffffu;
                    double lbc = box_lb_d(t.box[kExLevels - 1], g + src, qx, qy, qz);
                    if (!(lbc < tk.tau)) continue;
                    visit<kExLevels - 1>(t, g + src, own, qx, qy, qz, tk, lane);
                }
            }
            // data_processor.py:172: np.mean(dists[:, 1:], axis=1) -- NumPy pairwise float64 over k values
            const double r0 = __dsqrt_rn(tk.v0), r1 = __dsqrt_rn(tk.v1);
            auto rank = [&](int j) { return j < 32 ? shfl_d(r0, j) : shfl_d(r1, j - 32); };  // j = 1..k
            double res;
            if (k < 8) {
                res = 0.0;
                for (int j = 0; j < k; ++j) res = __dadd_rn(res, rank(1 + j));
            } else {
                double r[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) r[j] = rank(1 + j);
                int j = 8;
                for (; j < k - (k % 8); j += 8) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) r[e] = __dadd_rn(r[e], rank(1 + j + e));
                }
                res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                                __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
                for (; j < k; ++j) res = __dadd_rn(res, rank(1 + j));
            }
            if (lane == 0) out_means[__float_as_int(q.w)] = __double2float_rn(__ddiv_rn(res, (double)k));
        }
    }
}

int knn_exact_mean_dists(const float* xyz, int64_t n, int k, float* means, void* ws, int64_t ws_bytes,
                         cudaStream_t st) {
    GSX_REQUIRE(n >= 1 && n < GSX_N_LIMIT, GSX_ERR_ARG, "knn_exact: n out of range");
    GSX_REQUIRE(k >= 1 && k <= 63, GSX_ERR_UNSUPPORTED, "knn_exact: k must be in [1,63] (got %d)", k);
    ExWs w = ex_carve(ws, (size_t)ws_bytes, n, ex_sort_ws_bytes(n));
    GSX_REQUIRE(w.ok, GSX_ERR_WORKSPACE, "knn_exact: workspace too small");
    int rc = sor_minmax(xyz, n, w.minmax, w.partial, st);
    if (rc) return rc;
    float mm[6];
    GSX_CUDA_CHECK(cudaMemcpyAsync(mm, w.minmax, sizeof(mm), cudaMemcpyDeviceToHost, st));
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    float sc[3];
    for (int a = 0; a < 3; ++a) {
        float e = mm[3 + a] - mm[a];
        sc[a] = e > 0.f ? 65535.f / e : 0.f;
    }
    int blocks = (int)((n + 255) / 256);
    k_ex_keys<<<blocks, 256, 0, st>>>(xyz, n, mm[0], mm[1], mm[2], sc[0], sc[1], sc[2], w.keys0, w.vals0);
    GSX_KERNEL_CHECK();
    uint64_t* keys_sorted = nullptr;
    int32_t* order = nullptr;
    if ((rc = radix_sort_pairs(w.keys0, w.keys1, w.vals0, w.vals1, n, 0, 48, w.sort_ws, w.sort_ws_bytes, &keys_sorted,
                               &order, st)))
        return rc;
    k_ex_gather<<<blocks, 256, 0, st>>>(xyz, order, n, w.spos, w.box[0]);
    GSX_KERNEL_CHECK();
    for (int l = 1; l < kExLevels; ++l) {
        int64_t warps = w.cnt[l];
        k_ex_boxes_up<<<(int)((warps * 32 + 255) / 256), 256, 0, st>>>(w.box[l - 1], w.cnt[l - 1], w.box[l], w.cnt[l]);
        GSX_KERNEL_CHECK();
    }
    GSX_CUDA_CHECK(cudaMemsetAsync(w.counters, 0, sizeof(unsigned int), st));
    ExTree t;
    t.spos = w.spos;
    t.n = n;
    for (int l = 0; l < kExLevels; ++l) t.box[l] = w.box[l], t.cnt[l] = w.cnt[l];
    int per_sm = 0;
    GSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_knn_exact, 256, 0));
    int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 2);
    int64_t want = (n + 63) / 64;
    if (grid > want) grid = want;
    k_knn_exact<<<(int)grid, 256, 0, st>>>(t, means, w.counters, k);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

}  // namespace gsx
