// gsx_abi.cu -- the extern "C" surface of libgsx.so (declared in include/gsx.h).
//
// Thin: argument checks, workspace carving, stream plumbing and the host-buffer convenience
// entry points.  No torch types, no C++ types in any signature.
#include "../../include/gsx.h"

#include "gsx_common.cuh"
#include "gsx_compact.cuh"
#include "gsx_density.cuh"
#include "gsx_hostcopy.cuh"
#include "gsx_hostrows.cuh"
#include "gsx_kmeans.cuh"
#include "gsx_knn_exact.cuh"
#include "gsx_masks.cuh"
#include "gsx_morton.cuh"
#include "gsx_radix.cuh"
#include "gsx_records.cuh"
#include "gsx_sog.cuh"
#include "gsx_sor.cuh"

#include <atomic>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

namespace gsx {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count() {
    static int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cached = v;
        cached_dev = dev;
    }
    return cached;
}

// keep freed blocks in the default memory pool across calls: without this the pool is trimmed at every
// stream synchronisation and each *_host call pays ~20 ms of cudaMalloc for its workspace again
static void keep_pool_warm() {
    static thread_local int done_for = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    done_for = dev;
}

struct DevBuf {  // stream-ordered device allocation for the *_host entry points
    void* p = nullptr;
    cudaStream_t st;
    explicit DevBuf(cudaStream_t s) : st(s) { keep_pool_warm(); }
    int alloc(size_t bytes) {
        cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 1, st);
        if (e != cudaSuccess) {
            set_error("cudaMallocAsync(%zu) -> %s", bytes, cudaGetErrorString(e));
            p = nullptr;
            return GSX_ERR_CUDA;
        }
        return GSX_OK;
    }
    ~DevBuf() {
        if (p) cudaFreeAsync(p, st);
    }
};

}  // namespace gsx

using namespace gsx;

extern "C" {

const char* gsx_last_error(void) { return g_err; }
int gsx_version(void) { return 100; }
const char* gsx_build_info(void) { return sor_build_info(); }
long long gsx_kernel_launches(void) { return g_launches.load(); }
int gsx_device_sm_count(void) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return GSX_ERR_CUDA;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return GSX_ERR_CUDA;
    return v;
}

/* ------------------------------------------------------------------ SOR */

// The workspace sizes of the entry points bounded by GSX_N_LIMIT refuse what those entry points refuse.
#define GSX_WS_LIMIT(what, n)                                                                                    \
    GSX_REQUIRE((n) < GSX_N_LIMIT, GSX_ERR_ARG, what ": n=%lld out of range [0, 2^31-64)", (long long)(n))

int64_t gsx_sor_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("sor", n);
    return sor_workspace_bytes(n);
}
int64_t gsx_sor_grid_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("sor", n);
    return sor_grid_workspace_bytes(n);
}

// grid-only functions (build_from_sorted, mean_dists) accept the shorter gsx_sor_grid_workspace_bytes blob
static int carve_grid_checked(void* ws, int64_t ws_bytes, int64_t n, SorWs& w) {
    GSX_REQUIRE(n >= 1 && n < GSX_N_LIMIT, GSX_ERR_ARG, "sor: n=%lld out of range [1, 2^31-64)", (long long)n);
    GSX_REQUIRE(ws != nullptr, GSX_ERR_WORKSPACE, "sor: null workspace");
    w = sor_carve(ws, ws_bytes, n, sor_sort_ws_bytes(n));
    GSX_REQUIRE(w.grid_ok, GSX_ERR_WORKSPACE, "sor: grid workspace too small (%lld < %zu)", (long long)ws_bytes,
                w.grid_total);
    return GSX_OK;
}

static int carve_checked(void* ws, int64_t ws_bytes, int64_t n, SorWs& w) {
    GSX_REQUIRE(n >= 1 && n < GSX_N_LIMIT, GSX_ERR_ARG, "sor: n=%lld out of range [1, 2^31-64)", (long long)n);
    GSX_REQUIRE(ws != nullptr, GSX_ERR_WORKSPACE, "sor: null workspace");
    w = sor_carve(ws, ws_bytes, n, sor_sort_ws_bytes(n));
    GSX_REQUIRE(w.ok, GSX_ERR_WORKSPACE, "sor: workspace too small (%lld < %zu)", (long long)ws_bytes, w.total);
    return GSX_OK;
}

int gsx_sor_minmax(const float* xyz_dev, int64_t n, float* minmax_dev, void* ws, int64_t ws_bytes, void* stream) {
    GSX_REQUIRE(n >= 1, GSX_ERR_ARG, "sor: minmax of an empty cloud");
    GSX_REQUIRE(ws != nullptr && ws_bytes >= 6 * 1024 * (int64_t)sizeof(float), GSX_ERR_WORKSPACE,
                "sor: minmax needs 24 KiB of scratch");
    return sor_minmax(xyz_dev, n, minmax_dev, (float*)ws, (cudaStream_t)stream);  // scratch = the head of ws
}

/* gpu_ops.py:203-213 with NumPy-2 semantics: extent/vol in float32; vol<=0 -> python float 1.0 (then
 * float64 arithmetic); avg = max(1e-8, vol/N) keeps the float32 unless the python float wins; the
 * cube root is float32 powf for a float32 base, float64 pow otherwise; floor of 1e-4. */
float gsx_sor_cell_size(const float* mm, int64_t n) {
    float ex = mm[3] - mm[0], ey = mm[4] - mm[1], ez = mm[5] - mm[2];
    float vol = (ex * ey) * ez;
    double cell;
    if (vol <= 0.0f || vol != vol) {
        if (vol != vol) {
            cell = NAN;
        } else {
            double avg = 1.0 / (double)n;
            if (!(avg > 1e-8)) avg = 1e-8;
            cell = pow(avg * 32.0, 1.0 / 3.0);
        }
    } else {
        float avgf = vol / (float)n;
        if ((double)avgf > 1e-8) {  /* python max(1e-8, avgf) returns avgf only if avgf > 1e-8 */
            float cv = avgf * 32.0f;
            cell = (double)powf(cv, (float)(1.0 / 3.0));
        } else {
            cell = pow(1e-8 * 32.0, 1.0 / 3.0);
        }
    }
    if (!(cell > 1e-4)) cell = 1e-4; /* max(cell_size, 1e-4) */
    return (float)cell;
}

int gsx_sor_build(const float* xyz_dev, int64_t n, const float* bmin_host, float cell, void* ws, int64_t ws_bytes,
                  void* stream) {
    SorWs w;
    int rc = carve_checked(ws, ws_bytes, n, w);
    if (rc) return rc;
    GSX_REQUIRE(cell > 0.f, GSX_ERR_ARG, "sor: cell size must be > 0");
    return sor_build(xyz_dev, n, bmin_host, cell, w, (cudaStream_t)stream);
}

int gsx_sor_dist_local_run(const float* xyz_local_dev, int64_t n_local, int64_t idx_base, int64_t n_global,
                           int32_t world, const float* bmin_host, float cell, float* pos4_out_dev,
                           int64_t* cuts_dev, void* ws, int64_t ws_bytes, void* stream) {
    SorWs w;
    int rc = carve_checked(ws, ws_bytes, n_local > 0 ? n_local : 1, w);
    if (rc) return rc;
    GSX_REQUIRE(n_global >= n_local && n_global >= 1 && n_global < GSX_N_LIMIT, GSX_ERR_ARG, "sor: bad n_global");
    return sor_dist_local_run(xyz_local_dev, n_local, idx_base, n_global, world, bmin_host, cell,
                              (float4*)pos4_out_dev, (long long*)cuts_dev, w, (cudaStream_t)stream);
}

int gsx_sor_dist_merge(const float* pos4_dev, int64_t m, int64_t n_global, int64_t bucket_lo, int64_t bucket_hi,
                       const float* bmin_host, float cell, float* pos4_sorted_dev, uint8_t* flags_sorted_dev, void* ws,
                       int64_t ws_bytes, void* stream) {
    if (m == 0) return GSX_OK;
    SorWs w;
    int rc = carve_checked(ws, ws_bytes, m, w);
    if (rc) return rc;
    return sor_dist_merge((const float4*)pos4_dev, m, n_global, bucket_lo, bucket_hi, bmin_host, cell,
                          (float4*)pos4_sorted_dev, flags_sorted_dev, w, (cudaStream_t)stream);
}

int64_t gsx_sor_spos_offset(int64_t n) {
    if (n < 1) return -1;
    SorWs w = sor_carve(nullptr, 0, n, sor_sort_ws_bytes(n));
    return (int64_t)((char*)w.spos - (char*)nullptr);
}

int gsx_sor_build_from_sorted(const float* spos4_dev, const uint8_t* flags_dev, int64_t n, const float* bmin_host,
                              float cell, void* ws, int64_t ws_bytes, void* stream) {
    SorWs w;
    int rc = carve_grid_checked(ws, ws_bytes, n, w);
    if (rc) return rc;
    GSX_REQUIRE(cell > 0.f, GSX_ERR_ARG, "sor: cell size must be > 0");
    return sor_build_from_sorted((const float4*)spos4_dev, flags_dev, n, bmin_host, cell, w, (cudaStream_t)stream);
}

int gsx_sor_mean_dists_range(int64_t n, int64_t q_begin, int64_t q_end, int32_t k, int32_t hash_mode,
                             const float* bmin_host, float cell, void* ws, int64_t ws_bytes, float* final_means_dev,
                             unsigned long long* stats_dev, void* stream) {
    SorWs w;
    int rc = carve_grid_checked(ws, ws_bytes, n, w);
    if (rc) return rc;
    return sor_mean_dists(w, q_begin, q_end, 1, 0, k, hash_mode, bmin_host, cell, final_means_dev, stats_dev,
                          (cudaStream_t)stream);
}

int gsx_sor_mean_dists_strided(int64_t n, int32_t stride, int32_t phase, int32_t k, int32_t hash_mode,
                               const float* bmin_host, float cell, void* ws, int64_t ws_bytes, float* final_means_dev,
                               unsigned long long* stats_dev, void* stream) {
    SorWs w;
    int rc = carve_grid_checked(ws, ws_bytes, n, w);
    if (rc) return rc;
    return sor_mean_dists(w, 0, n, stride, phase, k, hash_mode, bmin_host, cell, final_means_dev, stats_dev,
                          (cudaStream_t)stream);
}

int gsx_sor_mean_dists(int64_t n, int32_t k, int32_t hash_mode, const float* bmin_host, float cell, void* ws,
                       int64_t ws_bytes, float* final_means_dev, unsigned long long* stats_dev, void* stream) {
    return gsx_sor_mean_dists_range(n, 0, n, k, hash_mode, bmin_host, cell, ws, ws_bytes, final_means_dev, stats_dev,
                                    stream);
}

int64_t gsx_mean_std_workspace_bytes(int64_t n) { return (int64_t)mean_std_ws_bytes(n); }

int gsx_mean_std_f32(const float* a_dev, int64_t n, float* out_dev, void* ws, int64_t ws_bytes, void* stream) {
    return mean_std_f32(a_dev, n, out_dev, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int64_t gsx_pairwise_slots(int64_t n) { return pairwise_slots(n); }

int gsx_pairwise_leaves_dist(const float* a_local_dev, int64_t base, int64_t n_local, int64_t n_global, int32_t sq,
                             const float* meanstd_dev, const float* halo_dev, const int64_t* bases_dev, int32_t world,
                             float* slot_dev, void* stream) {
    return pairwise_leaves_dist(a_local_dev, base, n_local, n_global, sq, meanstd_dev, halo_dev,
                                (const long long*)bases_dev, world, slot_dev, (cudaStream_t)stream);
}

int gsx_pairwise_finish(float* slot_dev, int64_t n_global, int32_t sq, float* meanstd_dev, void* stream) {
    GSX_REQUIRE(n_global >= 1, GSX_ERR_ARG, "pairwise_finish: n must be >= 1");
    return pairwise_finish(slot_dev, n_global, sq, meanstd_dev, (cudaStream_t)stream);
}

int gsx_threshold_mask(const float* a_dev, int64_t n, const float* meanstd_dev, float threshold_factor,
                       uint8_t* mask_dev, void* stream) {
    return threshold_mask(a_dev, n, meanstd_dev, threshold_factor, mask_dev, (cudaStream_t)stream);
}

int gsx_sor_filter_device(const float* xyz_dev, int64_t n, int32_t k, float threshold_factor, int32_t hash_mode,
                          uint8_t* mask_dev, float* means_dev, void* ws, int64_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    SorWs w;
    int rc = carve_checked(ws, ws_bytes, n, w);
    if (rc) return rc;
    GSX_REQUIRE(k >= 1, GSX_ERR_ARG, "sor: k must be >= 1 (got %d)", k);
    if ((rc = sor_minmax(xyz_dev, n, w.minmax, w.partial, st))) return rc;
    float mm[6];
    GSX_CUDA_CHECK(cudaMemcpyAsync(mm, w.minmax, sizeof(mm), cudaMemcpyDeviceToHost, st));
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    float cell = gsx_sor_cell_size(mm, n);
    GSX_REQUIRE(cell == cell, GSX_ERR_ARG, "sor: non-finite coordinates");
    if ((rc = sor_build(xyz_dev, n, mm, cell, w, st))) return rc;
    // the keys buffers are dead after the build: park the means there when the caller wants none
    float* means = means_dev ? means_dev : reinterpret_cast<float*>(w.keys0);
    if ((rc = sor_mean_dists(w, 0, n, 1, 0, k, hash_mode, mm, cell, means, nullptr, st))) return rc;
    if ((rc = mean_std_f32(means, n, w.meanstd, w.ms_ws, w.ms_bytes, st))) return rc;
    return threshold_mask(means, n, w.meanstd, threshold_factor, mask_dev, st);
}

int gsx_sor_filter_host(const float* xyz_host, int64_t n, int32_t k, float threshold_factor, int32_t hash_mode,
                        uint8_t* mask_host, float* means_host) {
    GSX_REQUIRE(n >= 1 && n < GSX_N_LIMIT, GSX_ERR_ARG, "sor: n=%lld out of range", (long long)n);
    cudaStream_t st = 0;
    int64_t wsb = sor_workspace_bytes(n);
    DevBuf xyz(st), ws(st), mask(st), means(st);
    int rc;
    if ((rc = xyz.alloc((size_t)n * 12))) return rc;
    if ((rc = ws.alloc((size_t)wsb))) return rc;
    if ((rc = mask.alloc((size_t)n))) return rc;
    if ((rc = means.alloc((size_t)n * 4))) return rc;
    if ((rc = copy_h2d(xyz.p, xyz_host, (size_t)n * 12, st))) return rc;
    if ((rc = gsx_sor_filter_device((const float*)xyz.p, n, k, threshold_factor, hash_mode, (uint8_t*)mask.p,
                                    (float*)means.p, ws.p, wsb, st)))
        return rc;
    // the kernels are queued: make the (usually never touched) destination pages resident while the GPU works
    prefault_host(mask_host, (size_t)n);
    if (means_host) prefault_host(means_host, (size_t)n * 4);
    if ((rc = copy_d2h(mask_host, mask.p, (size_t)n, st))) return rc;
    if (means_host && (rc = copy_d2h(means_host, means.p, (size_t)n * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSX_OK;
}

/* ------------------------------------------------------------------ pair sort (gpu_ops.py:227) */

int64_t gsx_sort_pairs_workspace_bytes(int64_t n) {
    GSX_REQUIRE(n < (1ll << 32), GSX_ERR_ARG, "sort: n=%lld out of range [0, 2^32)", (long long)n);
    if (n < 1) n = 1;
    return (int64_t)(align_up((size_t)n * 8, 256) + align_up((size_t)n * 4, 256) + radix_ws_bytes(n) + 1024);
}

int gsx_sort_pairs(uint64_t* keys_dev, int32_t* vals_dev, int64_t n, int32_t begin_bit, int32_t end_bit, void* ws,
                   int64_t ws_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return GSX_OK;
    GSX_REQUIRE(ws_bytes >= gsx_sort_pairs_workspace_bytes(n), GSX_ERR_WORKSPACE, "sort: workspace too small");
    Carver c(ws, (size_t)ws_bytes);
    uint64_t* k1 = c.take<uint64_t>((size_t)n);
    int32_t* v1 = c.take<int32_t>((size_t)n);
    char* rws = c.take<char>(radix_ws_bytes(n));
    uint64_t* ks = nullptr;
    int32_t* vs = nullptr;
    int rc = vals_dev ? radix_sort_pairs(keys_dev, k1, vals_dev, v1, n, begin_bit, end_bit, rws, radix_ws_bytes(n), &ks, &vs, st)
                      : radix_sort_keys(keys_dev, k1, n, begin_bit, end_bit, rws, radix_ws_bytes(n), &ks, st);
    if (rc) return rc;
    if (ks != keys_dev) {
        GSX_CUDA_CHECK(cudaMemcpyAsync(keys_dev, ks, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
        if (vals_dev) GSX_CUDA_CHECK(cudaMemcpyAsync(vals_dev, vs, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    }
    return GSX_OK;
}

/* ------------------------------------------------------------------ SOR, cKDTree semantics */

int64_t gsx_knn_exact_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("knn_exact", n);
    return knn_exact_workspace_bytes(n);
}

int gsx_knn_exact_mean_dists(const float* xyz_dev, int64_t n, int32_t k, float* means_dev, void* ws, int64_t ws_bytes,
                             void* stream) {
    return knn_exact_mean_dists(xyz_dev, n, k, means_dev, ws, ws_bytes, (cudaStream_t)stream);
}

int gsx_sor_ckdtree_filter_host(const float* xyz_host, int64_t n, int32_t k, float threshold_factor, uint8_t* mask_host,
                                float* means_host) {
    GSX_REQUIRE(n >= 1 && n < GSX_N_LIMIT, GSX_ERR_ARG, "sor: n=%lld out of range", (long long)n);
    cudaStream_t st = 0;
    int64_t wsb = knn_exact_workspace_bytes(n);
    int64_t msb = (int64_t)mean_std_ws_bytes(n);
    DevBuf xyz(st), ws(st), mask(st), means(st), ms(st), msws(st);
    int rc;
    if ((rc = xyz.alloc((size_t)n * 12))) return rc;
    if ((rc = ws.alloc((size_t)wsb))) return rc;
    if ((rc = mask.alloc((size_t)n))) return rc;
    if ((rc = means.alloc((size_t)n * 4))) return rc;
    if ((rc = ms.alloc(64))) return rc;
    if ((rc = msws.alloc((size_t)msb))) return rc;
    if ((rc = copy_h2d(xyz.p, xyz_host, (size_t)n * 12, st))) return rc;
    if ((rc = knn_exact_mean_dists((const float*)xyz.p, n, k, (float*)means.p, ws.p, wsb, st))) return rc;
    if ((rc = mean_std_f32((const float*)means.p, n, (float*)ms.p, msws.p, (size_t)msb, st))) return rc;
    if ((rc = threshold_mask((const float*)means.p, n, (const float*)ms.p, threshold_factor, (uint8_t*)mask.p, st)))
        return rc;
    // the kernels are queued: make the (usually never touched) destination pages resident while the GPU works
    prefault_host(mask_host, (size_t)n);
    if (means_host) prefault_host(means_host, (size_t)n * 4);
    if ((rc = copy_d2h(mask_host, mask.p, (size_t)n, st))) return rc;
    if (means_host && (rc = copy_d2h(means_host, means.p, (size_t)n * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSX_OK;
}

/* ------------------------------------------------------------------ bbox / alpha */

int gsx_bbox_mask(const float* xyz_dev, int64_t n, const float* lohi_host, uint8_t* mask_dev, void* stream) {
    GSX_REQUIRE(n >= 0, GSX_ERR_ARG, "bbox: n < 0");
    return bbox_mask(xyz_dev, n, lohi_host, mask_dev, (cudaStream_t)stream);
}

int gsx_alpha_mask(const float* opacity_dev, int64_t n, double logit_thresh, uint8_t* mask_dev, void* stream) {
    GSX_REQUIRE(n >= 0, GSX_ERR_ARG, "alpha: n < 0");
    return alpha_mask(opacity_dev, n, logit_thresh, mask_dev, (cudaStream_t)stream);
}

double gsx_alpha_logit_threshold(double min_opacity_u8) {
    double a = min_opacity_u8 / 255.0;
    if (a < 1e-6) a = 1e-6;
    if (a > 1.0 - 1e-6) a = 1.0 - 1e-6;
    return log(a / (1.0 - a));
}

/* ------------------------------------------------------------------ compaction between filters */

int64_t gsx_compact_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("compact", n);
    return compact_workspace_bytes(n);
}

int gsx_compact_points(const uint8_t* mask_dev, int64_t n, const float* xyz_dev, const float* opacity_dev,
                       const int32_t* idx_dev, float* xyz_out_dev, float* opacity_out_dev, int32_t* idx_out_dev,
                       int64_t* count_host, void* ws, int64_t ws_bytes, void* stream) {
    return compact_points(mask_dev, n, xyz_dev, opacity_dev, idx_dev, xyz_out_dev, opacity_out_dev, idx_out_dev,
                          count_host, ws, ws_bytes, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------ density */

int64_t gsx_density_workspace_bytes(int64_t n, int64_t cap) { return density_workspace_bytes(n, cap); }

int gsx_density_voxel_count(const float* xyz_dev, int64_t n, float voxel, int64_t min_points, int64_t* dense_vox_host,
                            int32_t* dense_cnt_host, int64_t cap, int64_t* n_dense_host, int64_t* n_voxels_host,
                            void* ws, int64_t ws_bytes, void* stream) {
    return density_voxel_count(xyz_dev, n, voxel, min_points, dense_vox_host, dense_cnt_host, cap, n_dense_host,
                               n_voxels_host, ws, ws_bytes, (cudaStream_t)stream);
}

int gsx_density_member_mask(const float* xyz_dev, int64_t n, float voxel, const int64_t* keep_vox_host, int64_t n_keep,
                            uint8_t* mask_dev, void* ws, int64_t ws_bytes, void* stream) {
    return density_member_mask(xyz_dev, n, voxel, keep_vox_host, n_keep, mask_dev, ws, ws_bytes,
                               (cudaStream_t)stream);
}

void gsx_density_voxel_range(const float* minmax_host, float voxel, int64_t* q0_out, int64_t* dim_out) {
    density_voxel_range(minmax_host, voxel, q0_out, dim_out);
}

int gsx_density_grid_count(const float* xyz_dev, int64_t n, float voxel, const int64_t* q0, const int64_t* dim,
                           int32_t* grid_dev, unsigned long long* oob_dev, void* stream) {
    return density_grid_count(xyz_dev, n, voxel, q0, dim, grid_dev, oob_dev, (cudaStream_t)stream);
}

int gsx_density_grid_dense(const int32_t* grid_dev, const int64_t* q0, const int64_t* dim, int64_t min_points,
                           int64_t* dense_vox_host, int32_t* dense_cnt_host, int64_t cap, int64_t* n_dense_host,
                           int64_t* n_voxels_host, void* ws, int64_t ws_bytes, void* stream) {
    return density_grid_dense(grid_dev, q0, dim, min_points, dense_vox_host, dense_cnt_host, cap, n_dense_host,
                              n_voxels_host, ws, ws_bytes, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------ SOG writer helpers (SURVEY 8f-1) */

int64_t gsx_lexsort_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("lexsort", n);
    return lexsort_workspace_bytes(n);
}

int gsx_lexsort_zyx(const float* xyz_dev, int64_t n, int32_t* order_dev, void* ws, int64_t ws_bytes, void* stream) {
    return lexsort_zyx(xyz_dev, n, order_dev, ws, ws_bytes, (cudaStream_t)stream);
}

int gsx_quantize_to_codebook(const float* vals_dev, int64_t n, const float* codebook_host, int32_t m,
                             uint8_t* labels_dev, void* ws, int64_t ws_bytes, void* stream) {
    return quantize_to_codebook(vals_dev, n, codebook_host, m, labels_dev, ws, ws_bytes, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------ K-Means */

int64_t gsx_kmeans_workspace_bytes(int64_t n_total, int32_t nprob, int32_t K, int32_t D) {
    return kmeans_workspace_bytes(n_total, nprob, K, D);
}

int gsx_kmeans_lloyd_device(const float* X_dev, const int64_t* row_off_host, int32_t nprob, int32_t K, int32_t D,
                            int32_t max_iter, float* C_dev, int32_t* labels_dev, int32_t* counts_dev, void* ws,
                            int64_t ws_bytes, int32_t assign_mode, unsigned long long* tc_stats_dev, void* stream) {
    return kmeans_lloyd(X_dev, row_off_host, nprob, K, D, max_iter, C_dev, labels_dev, counts_dev, ws, ws_bytes,
                        assign_mode, tc_stats_dev, (cudaStream_t)stream);
}

int32_t gsx_kmeans_tensor_core_supported(int32_t K, int32_t D) {
    return kmeans_tc_supported(K, D) ? (kmeans_tc16_built() ? 3 : 1) : 0;   // bit 0: TF32 kernel, bit 1: split-bf16 build
}

int gsx_kmeans_tc_debug_scores(const float* X_dev, int64_t rows, const float* C_dev, int32_t K, int32_t D,
                               int32_t variant, float* scores_dev, void* ws, int64_t ws_bytes, void* stream) {
    return kmeans_tc_debug_scores(X_dev, rows, C_dev, K, D, variant, scores_dev, ws, ws_bytes, (cudaStream_t)stream);
}

int gsx_kmeans_host(const float* X_host, int64_t n, int32_t K, int32_t D, int32_t max_iter, float* C_host_inout,
                    int32_t* labels_host, int32_t assign_mode) {
    GSX_REQUIRE(n >= 1 && K >= 1 && D >= 1, GSX_ERR_ARG, "kmeans: bad shape");
    cudaStream_t st = 0;
    DevBuf X(st), C(st), L(st), cnt(st), ws(st);
    int rc;
    int64_t wsb = kmeans_workspace_bytes(n, 1, K, D);
    if ((rc = X.alloc((size_t)n * D * 4))) return rc;
    if ((rc = C.alloc((size_t)K * D * 4))) return rc;
    if ((rc = L.alloc((size_t)n * 4))) return rc;
    if ((rc = cnt.alloc((size_t)K * 4))) return rc;
    if ((rc = ws.alloc((size_t)wsb))) return rc;
    if ((rc = copy_h2d(X.p, X_host, (size_t)n * D * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaMemcpyAsync(C.p, C_host_inout, (size_t)K * D * 4, cudaMemcpyHostToDevice, st));
    GSX_CUDA_CHECK(cudaMemsetAsync(L.p, 0, (size_t)n * 4, st));
    int64_t off[2] = {0, n};
    if ((rc = kmeans_lloyd((const float*)X.p, off, 1, K, D, max_iter, (float*)C.p, (int*)L.p, (int*)cnt.p, ws.p, wsb, assign_mode, nullptr, st)))
        return rc;
    prefault_host(labels_host, (size_t)n * 4);   // while the Lloyd iterations run
    GSX_CUDA_CHECK(cudaMemcpyAsync(C_host_inout, C.p, (size_t)K * D * 4, cudaMemcpyDeviceToHost, st));
    if ((rc = copy_d2h(labels_host, L.p, (size_t)n * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSX_OK;
}

/* SOG shN schedule in one call on HOST buffers: nprob problems stored back to back in X_host (rows row_off[p] ..
 * row_off[p+1]), each with K centroids; C_host_inout [nprob*K*D] holds the init on entry, the centroids on return. */
int gsx_kmeans_host_batched(const float* X_host, const int64_t* row_off_host, int32_t nprob, int32_t K, int32_t D,
                            int32_t max_iter, float* C_host_inout, int32_t* labels_host, int32_t assign_mode) {
    GSX_REQUIRE(nprob >= 1 && K >= 1 && D >= 1, GSX_ERR_ARG, "kmeans: bad shape");
    GSX_REQUIRE(row_off_host[0] == 0, GSX_ERR_ARG, "kmeans: row_off[0] must be 0");
    const int64_t n = row_off_host[nprob];
    GSX_REQUIRE(n >= 1, GSX_ERR_ARG, "kmeans: no rows");
    cudaStream_t st = 0;
    DevBuf X(st), C(st), L(st), cnt(st), ws(st);
    int rc;
    int64_t wsb = kmeans_workspace_bytes(n, nprob, K, D);
    if ((rc = X.alloc((size_t)n * D * 4))) return rc;
    if ((rc = C.alloc((size_t)nprob * K * D * 4))) return rc;
    if ((rc = L.alloc((size_t)n * 4))) return rc;
    if ((rc = cnt.alloc((size_t)nprob * K * 4))) return rc;
    if ((rc = ws.alloc((size_t)wsb))) return rc;
    if ((rc = copy_h2d(X.p, X_host, (size_t)n * D * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaMemcpyAsync(C.p, C_host_inout, (size_t)nprob * K * D * 4, cudaMemcpyHostToDevice, st));
    GSX_CUDA_CHECK(cudaMemsetAsync(L.p, 0, (size_t)n * 4, st));
    if ((rc = kmeans_lloyd((const float*)X.p, row_off_host, nprob, K, D, max_iter, (float*)C.p, (int*)L.p, (int*)cnt.p,
                           ws.p, wsb, assign_mode, nullptr, st)))
        return rc;
    prefault_host(labels_host, (size_t)n * 4);   // while the Lloyd iterations run
    GSX_CUDA_CHECK(cudaMemcpyAsync(C_host_inout, C.p, (size_t)nprob * K * D * 4, cudaMemcpyDeviceToHost, st));
    if ((rc = copy_d2h(labels_host, L.p, (size_t)n * 4, st))) return rc;
    GSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return GSX_OK;
}

/* ------------------------------------------------------------------ pageable host buffers <-> HBM */
int gsx_copy_h2d(void* dst_dev, const void* src_host, int64_t bytes, void* stream) {
    GSX_REQUIRE(bytes >= 0 && (bytes == 0 || (dst_dev && src_host)), GSX_ERR_ARG, "copy_h2d: bad arguments");
    return copy_h2d(dst_dev, src_host, (size_t)bytes, (cudaStream_t)stream);
}
int gsx_copy_d2h(void* dst_host, const void* src_dev, int64_t bytes, void* stream) {
    GSX_REQUIRE(bytes >= 0 && (bytes == 0 || (dst_host && src_dev)), GSX_ERR_ARG, "copy_d2h: bad arguments");
    return copy_d2h(dst_host, src_dev, (size_t)bytes, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------ host-resident records: threaded row movement */
int gsx_host_gather_rows(const void* src_host, int64_t n_rows, int64_t row_bytes, const int64_t* idx_host, int64_t m,
                         void* dst_host) {
    return host_gather_rows(src_host, n_rows, row_bytes, idx_host, m, dst_host);
}
int gsx_host_extract_xyz_opacity(const void* src_host, int64_t n_rows, int64_t row_bytes, int64_t off_x, int64_t off_y,
                                 int64_t off_z, int64_t off_opacity, float* xyz_out_host, float* opacity_out_host) {
    return host_extract_xyz_opacity(src_host, n_rows, row_bytes, off_x, off_y, off_z, off_opacity, xyz_out_host,
                                    opacity_out_host);
}

/* ------------------------------------------------------------------ device-resident records (SURVEY 8f 2,4) */
int gsx_records_extract_xyz_opacity(const float* rows_dev, int64_t n, int32_t F, int32_t cx, int32_t cy, int32_t cz,
                                    int32_t cop, float* xyz_dev, float* opacity_dev, void* stream) {
    return records_extract_xyz_opacity(rows_dev, n, F, cx, cy, cz, cop, xyz_dev, opacity_dev, (cudaStream_t)stream);
}
int gsx_records_gather_rows(const float* rows_dev, const int32_t* idx_dev, int64_t m, int32_t F, float* out_dev,
                            void* stream) {
    return records_gather_rows(rows_dev, idx_dev, m, F, out_dev, (cudaStream_t)stream);
}
int gsx_records_color_rgba8(const float* rows_dev, int64_t n, int32_t F, int32_t c0, int32_t c1, int32_t c2, int32_t cop,
                            float scale, uint8_t* rgba_dev, void* stream) {
    return records_color_rgba8(rows_dev, n, F, c0, c1, c2, cop, scale, rgba_dev, (cudaStream_t)stream);
}
int gsx_records_scale_exp(const float* rows_dev, int64_t n, int32_t F, int32_t s0, int32_t s1, int32_t s2, float* out_dev,
                          void* stream) {
    return records_scale_exp(rows_dev, n, F, s0, s1, s2, out_dev, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------ Morton ordering primitive (SURVEY 8f 3) */
int64_t gsx_morton_workspace_bytes(int64_t n) {
    GSX_WS_LIMIT("morton", n);
    return morton_workspace_bytes(n);
}
int gsx_morton_order(const float* xyz_dev, int64_t n, int32_t* order_dev, int32_t run_limit, int32_t* levels_out, void* ws,
                     int64_t ws_bytes, void* stream) {
    int lv = 0;
    int rc = morton_order(xyz_dev, n, order_dev, run_limit, 16, &lv, ws, ws_bytes, (cudaStream_t)stream);
    if (levels_out) *levels_out = lv;
    return rc;
}
int gsx_chunk_minmax(const float* rows_dev, int64_t n, int32_t F, const int32_t* order_dev, int32_t chunk,
                     const int32_t* cols_host, int32_t ncol, float clip_lo, float clip_hi, float* lo_dev, float* hi_dev,
                     void* ws, int64_t ws_bytes, void* stream) {
    return chunk_minmax(rows_dev, n, F, order_dev, chunk, cols_host, ncol, clip_lo, clip_hi, lo_dev, hi_dev, ws, ws_bytes,
                        (cudaStream_t)stream);
}

/* free / total device memory of the current device (sizing decisions of the host-buffer entry points) */
int gsx_device_memory(int64_t* free_bytes, int64_t* total_bytes) {
    size_t f = 0, t = 0;
    GSX_CUDA_CHECK(cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = (int64_t)f;
    if (total_bytes) *total_bytes = (int64_t)t;
    return GSX_OK;
}

}  // extern "C"
