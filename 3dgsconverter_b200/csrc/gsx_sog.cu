// gsx_sog.cu -- device helpers for the steps either side of K-Means in the SOG writer (SURVEY §8(f) item 1).
//
//   gsx_lexsort_zyx            np.lexsort((z, y, x))                      formats/sog.py:264
//   gsx_quantize_to_codebook   sorted-codebook nearest entry               formats/sog.py:408-419
//
// lexsort: stable LSD over the three float32 keys with our radix sort -- first by z (32 bits), then by the
// 64-bit key x:y -- after mapping floats to order-preserving unsigned ints (-0.0 is folded into +0.0 because
// NumPy compares them equal).  quantize: lower_bound in the (<= 4096-entry) codebook held in shared memory,
// clip, then the reference's left-neighbour test |v - cb[left]| < |v - cb[idx]| in float32.
#include "../../include/gsx.h"
#include "gsx_common.cuh"
#include "gsx_radix.cuh"
#include "gsx_sog.cuh"

namespace gsx {

__device__ __forceinline__ uint32_t float_key(float f) {
    f = f + 0.0f;  // -0.0 -> +0.0 (equal keys in NumPy)
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(256) k_lex_keys_z(const float* __restrict__ xyz, int64_t n,
                                                    uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = (uint64_t)float_key(xyz[3 * i + 2]);
    vals[i] = (int32_t)i;
}

__global__ void __launch_bounds__(256) k_lex_keys_xy(const float* __restrict__ xyz, const int32_t* __restrict__ order,
                                                     int64_t n, uint64_t* __restrict__ keys) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int64_t i = order[j];
    keys[j] = ((uint64_t)float_key(xyz[3 * i]) << 32) | (uint64_t)float_key(xyz[3 * i + 1]);
}

int64_t lexsort_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    return (int64_t)(2 * align_up((size_t)n * 8, 256) + 2 * align_up((size_t)n * 4, 256) + radix_ws_bytes(n) + 1024);
}

int lexsort_zyx(const float* xyz, int64_t n, int32_t* order_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
    if (n == 0) return GSX_OK;
    GSX_REQUIRE(n < GSX_N_LIMIT, GSX_ERR_ARG, "lexsort: n out of range");
    GSX_REQUIRE(ws_bytes >= lexsort_workspace_bytes(n), GSX_ERR_WORKSPACE, "lexsort: workspace too small");
    Carver c(ws, (size_t)ws_bytes);
    uint64_t* k0 = c.take<uint64_t>((size_t)n);
    uint64_t* k1 = c.take<uint64_t>((size_t)n);
    int32_t* v0 = c.take<int32_t>((size_t)n);
    int32_t* v1 = c.take<int32_t>((size_t)n);
    char* rws = c.take<char>(radix_ws_bytes(n));
    int blocks = (int)((n + 255) / 256);
    k_lex_keys_z<<<blocks, 256, 0, st>>>(xyz, n, k0, v0);
    GSX_KERNEL_CHECK();
    uint64_t* ks = nullptr;
    int32_t* vs = nullptr;
    int rc = radix_sort_pairs(k0, k1, v0, v1, n, 0, 32, rws, radix_ws_bytes(n), &ks, &vs, st);
    if (rc) return rc;
    // second (more significant) key pair, gathered in the current order; reuse the buffer vs does not occupy
    uint64_t* kin = (ks == k0) ? k0 : k1;  // keys are dead: overwrite the buffer that pairs with vs
    uint64_t* kalt = (ks == k0) ? k1 : k0;
    int32_t* valt = (vs == v0) ? v1 : v0;
    k_lex_keys_xy<<<blocks, 256, 0, st>>>(xyz, vs, n, kin);
    GSX_KERNEL_CHECK();
    uint64_t* ks2 = nullptr;
    int32_t* vs2 = nullptr;
    rc = radix_sort_pairs(kin, kalt, vs, valt, n, 0, 64, rws, radix_ws_bytes(n), &ks2, &vs2, st);
    if (rc) return rc;
    GSX_CUDA_CHECK(cudaMemcpyAsync(order_out, vs2, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    return GSX_OK;
}

constexpr int kMaxCodebook = 4096;

__global__ void __launch_bounds__(256) k_quantize_codebook(const float* __restrict__ vals, int64_t n,
                                                           const float* __restrict__ cb, int m,
                                                           uint8_t* __restrict__ labels) {
    __shared__ float scb[kMaxCodebook];
    for (int t = threadIdx.x; t < m; t += blockDim.x) scb[t] = cb[t];
    __syncthreads();
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float v = vals[i];
        int lo = 0, hi = m;  // np.searchsorted(cb, v) (side='left'): first index with cb[idx] >= v
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if (scb[mid] < v) lo = mid + 1; else hi = mid;
        }
        int idx = lo < m - 1 ? lo : m - 1;          // np.clip(idx, 0, len(cb)-1)
        int left = idx - 1 > 0 ? idx - 1 : 0;        // np.maximum(idx-1, 0)
        float d_idx = fabsf(__fsub_rn(v, scb[idx])), d_left = fabsf(__fsub_rn(v, scb[left]));
        if (d_left < d_idx) idx = left;
        labels[i] = (uint8_t)idx;                    // .astype(np.uint8)
    }
}

int quantize_to_codebook(const float* vals, int64_t n, const float* codebook_host, int m, uint8_t* labels, void* ws,
                         int64_t ws_bytes, cudaStream_t st) {
    if (n == 0) return GSX_OK;
    GSX_REQUIRE(m >= 1 && m <= kMaxCodebook, GSX_ERR_UNSUPPORTED, "quantize: codebook size must be in [1,%d]",
                kMaxCodebook);
    GSX_REQUIRE(ws_bytes >= (int64_t)m * 4, GSX_ERR_WORKSPACE, "quantize: workspace too small");
    if (m == 1) {  // sog.py:410
        GSX_CUDA_CHECK(cudaMemsetAsync(labels, 0, (size_t)n, st));
        return GSX_OK;
    }
    GSX_CUDA_CHECK(cudaMemcpyAsync(ws, codebook_host, (size_t)m * 4, cudaMemcpyHostToDevice, st));
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));  // codebook_host may be a temporary
    int blocks = sm_count() * 8;
    int64_t need = (n + 255) / 256;
    if ((int64_t)blocks > need) blocks = (int)need;
    k_quantize_codebook<<<blocks, 256, 0, st>>>(vals, n, (const float*)ws, m, labels);
    GSX_KERNEL_CHECK();
    return GSX_OK;
}

}  // namespace gsx
