/*
 * gsx.h -- C ABI of libgsx.so, the B200-native (sm_100a) backend for the per-point
 * filtering + codebook clustering hot path of francescofugazzi/3dgsconverter.
 *
 * The reference has no FFI of its own (it is pure Python + Taichi); the boundary it
 * exposes is the Python module surface gsconverter.processing.{gpu_ops,data_processor}.
 * Each entry point below names the reference interface it replaces (path:line relative
 * to /root/reference/gsconverter/).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - plain C types only; device pointers are ordinary pointers into CUDA device
 *     memory of the *current* device; `stream` is a cudaStream_t passed as void*
 *     (NULL = default stream).
 *   - every function returns 0 on success, <0 on error (GSX_ERR_*); the message is
 *     available from gsx_last_error() (thread-local).  The Python wrapper turns a
 *     non-zero status into an exception, which preserves the reference's
 *     "GPU exception => caller falls back" convention (data_processor.py:146-153,
 *     gpu_ops.py:40-46).
 *   - the library never owns device memory in the *_device entry points: the caller
 *     provides outputs and one scratch blob whose size comes from *_workspace_bytes.
 *     The *_host convenience entry points take host buffers and manage device memory
 *     internally (cudaMallocAsync), copies included.
 *   - all masks are uint8 (0/1), one byte per point, like numpy bool.
 *   - N < 2^31 - 64 = GSX_N_LIMIT (int32 indices, as in gpu_ops.py:224,233-234) for every entry point that takes a
 *     point count, except the generic gsx_sort_pairs (n < 2^32).  The *_workspace_bytes functions of those entry
 *     points return GSX_ERR_ARG for an n outside the range.
 *     Two primitives change algorithm at 2^30 rows, because below it they chain 30-bit running counts through
 *     decoupled look-back words (one kernel): the radix sort (gsx_sort_pairs and every sort inside SOR, lexsort,
 *     Morton order and the cKDTree-semantics KNN) runs onesweep passes for n < 2^30 and three-kernel
 *     histogram / scan / scatter passes with 32-bit offsets from 2^30 on; gsx_compact_points runs one look-back pass
 *     for n < 2^30 and count / scan / scatter from 2^30 on.  tests/test_size_limits_gpu.py runs both sides: the
 *     shipped library at n > 2^30, and the existing small-n checks against builds whose switch-over is 4096 rows.
 */
#ifndef GSX_H
#define GSX_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSX_N_LIMIT 2147483584LL /* 2^31 - 64: every point count n < GSX_N_LIMIT */

#define GSX_HASH_I32WRAP 0 /* probe hash with wrapping int32 products: Taichi default_ip (faithful, SURVEY F8) */
#define GSX_HASH_I64 1     /* probe hash with int64 products: what the host table build uses (intended) */

/* ---- library ---------------------------------------------------------------------- */
const char* gsx_last_error(void);
int gsx_version(void);          /* 100*major + minor */
const char* gsx_build_info(void); /* compile-time switches of the SOR query kernel ("knn=r02c;epi_smem=1;..."): names the
                                   * build an ncu capture / a bench line was taken with */
int gsx_device_sm_count(void);  /* SMs of the current device (grid sizing), <0 on error */
long long gsx_kernel_launches(void); /* cumulative number of gsx kernels launched by this process */

/* ---- SOR, Taichi semantics: gpu_ops.py:193-263 (filter_sor_gpu) + :98-176 (kernel) - */

/* Scratch needed by gsx_sor_filter_device / the gsx_sor_* stages for n points.  The grid the query kernel reads
 * (sorted positions, bucket table, boxes) is a PREFIX of that blob: gsx_sor_build_from_sorted and
 * gsx_sor_mean_dists[_range] also accept a blob of only gsx_sor_grid_workspace_bytes(n) (no sort buffers) -- what
 * every rank of the distributed build holds for the union cloud. */
int64_t gsx_sor_workspace_bytes(int64_t n);
int64_t gsx_sor_grid_workspace_bytes(int64_t n);

/* gpu_ops.py:203-204: per-axis min/max of xyz[n,3] -> minmax_dev[6] = {minx,miny,minz,maxx,maxy,maxz}.
 * Scratch: the first 24 KiB of ws (any workspace of gsx_sor_workspace_bytes, or a small blob of its own). */
int gsx_sor_minmax(const float* xyz_dev, int64_t n, float* minmax_dev, void* ws, int64_t ws_bytes, void* stream);

/* gpu_ops.py:205-213 on the host (NumPy-2 float32 semantics, powf).  minmax is a HOST array of 6. */
float gsx_sor_cell_size(const float* minmax_host, int64_t n);

/* gpu_ops.py:216-237: grid index, int64 hash mod n, sort by bucket, bucket table.  Fills the
 * workspace with the hash-sorted float4 positions (w = original index), the bucket table and the
 * 32-/1024-point bounding boxes used for exact pruning.  bmin = the 3 minima, cell = cell size. */
int gsx_sor_build(const float* xyz_dev, int64_t n, const float* bmin_host, float cell, void* ws, int64_t ws_bytes,
                  void* stream);

/* Distributed form of gsx_sor_build for a cloud sharded over G processes (one per GPU); the collectives
 * between the stages are the caller's (gsx/dist.py uses NCCL).  Bucket-range ownership: rank o owns the
 * buckets [ceil(o*n_global/G), ceil((o+1)*n_global/G)).
 *  A. local_run:  stable partition of the slab by bucket owner (one radix pass); outputs float4
 *     {x,y,z, bits(idx_base + local index)} grouped by owner and cuts_dev[G+1] = first position of every owner
 *     -> the caller exchanges the groups (all-to-all).
 *  B. merge:      sorts the m received points of this rank's bucket range [bucket_lo, bucket_hi) by (bucket, in-cell Morton)
 *     -> the caller all-gathers the segments in owner order = the globally hash-sorted array.  With flags_sorted_dev
 *     the owner also emits one byte per sorted point (bit 0: starts a bucket, bit 1: other grid cell than the point
 *     before) -- exchanged along with the segment (1 B/pt next to 16 B/pt), it spares every receiving rank the
 *     re-hash of every point in its replicated stage C.
 *  C. build_from_sorted: bucket table ({start,end} per bucket, 8 B, the only part that is pre-zeroed), bucket boxes
 *     and chunk/super boxes from that array in one fused pass + one pass over the bucket starts (what
 *     gsx_sor_build leaves in the workspace), after which gsx_sor_mean_dists[_range] can run.  If spos4_dev already points at
 *     ws + gsx_sor_spos_offset(n) (all-gather straight into the workspace) no copy is made.
 * ws of A and B: gsx_sor_workspace_bytes(n_local) resp. (m); of C: gsx_sor_workspace_bytes(n_global). */
int gsx_sor_dist_local_run(const float* xyz_local_dev, int64_t n_local, int64_t idx_base, int64_t n_global,
                           int32_t world, const float* bmin_host, float cell, float* pos4_out_dev,
                           int64_t* cuts_dev, void* ws, int64_t ws_bytes, void* stream);
int gsx_sor_dist_merge(const float* pos4_dev, int64_t m, int64_t n_global, int64_t bucket_lo, int64_t bucket_hi,
                       const float* bmin_host, float cell, float* pos4_sorted_dev,
                       uint8_t* flags_sorted_dev /* uint8[m] or NULL */, void* ws, int64_t ws_bytes, void* stream);
int64_t gsx_sor_spos_offset(int64_t n);
int gsx_sor_build_from_sorted(const float* spos4_dev, const uint8_t* flags_dev /* uint8[n] or NULL */, int64_t n,
                              const float* bmin_host, float cell, void* ws, int64_t ws_bytes, void* stream);

/* gpu_ops.py:98-176 + :255-256: K = min(k,50) nearest candidates over the 27 probed buckets, mean of
 * their distances, written in the caller's point order (the "unsort" is fused).  Must follow
 * gsx_sor_build on the same workspace.  hash_mode = GSX_HASH_*.  stats_dev (may be NULL, else 16 zeroed uint64)
 * accumulates {reference-model visits V, candidates actually scanned, box tests, queries, queries answered by the
 * group path, 0, 0, 0, then 4 cycle counts and 4 query counts per class of centre-bucket size (<= 64, <= 1024,
 * <= 16384, larger) -- these 8 only in a -DGSX_KNN_PROFILE=1 build}. */
int gsx_sor_mean_dists(int64_t n, int32_t k, int32_t hash_mode, const float* bmin_host, float cell, void* ws,
                       int64_t ws_bytes, float* final_means_dev, unsigned long long* stats_dev, void* stream);

/* Multi-GPU variant: only the hash-sorted positions [q_begin, q_end) are queried; the rows of
 * final_means_dev belonging to other queries are left untouched (caller zero-fills and all-reduces). */
int gsx_sor_mean_dists_range(int64_t n, int64_t q_begin, int64_t q_end, int32_t k, int32_t hash_mode,
                             const float* bmin_host, float cell, void* ws, int64_t ws_bytes, float* final_means_dev,
                             unsigned long long* stats_dev, void* stream);

/* Multi-GPU variant with COST-balanced sharding: the hash-sorted positions are cut into batches of 16; this call
 * queries the batches b with b % stride == phase (stride = number of ranks, phase = rank), so every rank samples the
 * whole hash range -- the expensive (clustered) buckets are spread over all ranks instead of falling to the owner of
 * their hash range.  Rows of final_means_dev belonging to other batches are left untouched. */
int gsx_sor_mean_dists_strided(int64_t n, int32_t stride, int32_t phase, int32_t k, int32_t hash_mode,
                               const float* bmin_host, float cell, void* ws, int64_t ws_bytes, float* final_means_dev,
                               unsigned long long* stats_dev, void* stream);

/* gpu_ops.py:227 (np.argsort of the bucket hashes): stable LSD radix sort, in place, of (uint64 key, int32
 * value) pairs on the key bits [begin_bit, end_bit): 8-bit digits, one "onesweep" kernel per digit (decoupled
 * look-back over per-tile digit counts) after a single histogram pass; from n = 2^30 on, histogram / scan / scatter
 * kernels per digit.  vals_dev == NULL sorts bare 64-bit words: the form the hash-grid build uses, with
 * word = bucket | in-cell Morton code | original index and only the bits above the index sorted -- 8 instead of 12
 * bytes moved per point and pass.  1 <= n < 2^32 (n = 0 is a no-op); the workspace size is GSX_ERR_ARG above. */
int64_t gsx_sort_pairs_workspace_bytes(int64_t n);
int gsx_sort_pairs(uint64_t* keys_dev, int32_t* vals_dev, int64_t n, int32_t begin_bit, int32_t end_bit, void* ws,
                   int64_t ws_bytes, void* stream);

/* gpu_ops.py:259-260 / data_processor.py:176-177: np.mean and np.std of a float32 vector with
 * float32 accumulators and NumPy's pairwise summation order, bit-for-bit.  out_dev[0]=mean, [1]=std. */
int64_t gsx_mean_std_workspace_bytes(int64_t n);
int gsx_mean_std_f32(const float* a_dev, int64_t n, float* out_dev, void* ws, int64_t ws_bytes, void* stream);

/* The same statistics for a vector sharded over G processes (rank r holds a[bases[r] .. bases[r+1]) ): NumPy's
 * pairwise tree depends only on n, so every leaf (<= 128 consecutive elements) is summed by the rank that holds
 * its first element -- spill-over elements come from halo_dev = float32[G*128], the first 128 elements of every
 * slab (all-gathered by the caller) -- into slot_dev[gsx_pairwise_slots(n)] (0 elsewhere); the caller all-reduces
 * (sum, exact: one writer per slot) and gsx_pairwise_finish combines the inner nodes: sq=0 writes meanstd_dev[0] =
 * mean, sq=1 (after the mean is known) writes meanstd_dev[1] = std.  Bit-identical to gsx_mean_std_f32 on the
 * concatenated vector.  bases_dev: int64[G+1] on the device. */
int64_t gsx_pairwise_slots(int64_t n);
int gsx_pairwise_leaves_dist(const float* a_local_dev, int64_t base, int64_t n_local, int64_t n_global, int32_t sq,
                             const float* meanstd_dev, const float* halo_dev, const int64_t* bases_dev, int32_t world,
                             float* slot_dev, void* stream);
int gsx_pairwise_finish(float* slot_dev, int64_t n_global, int32_t sq, float* meanstd_dev, void* stream);

/* gpu_ops.py:261-263 / data_processor.py:178-180: mask[i] = a[i] < mean + f32(threshold_factor)*std. */
int gsx_threshold_mask(const float* a_dev, int64_t n, const float* meanstd_dev, float threshold_factor,
                       uint8_t* mask_dev, void* stream);

/* Whole filter on device buffers (one 24-byte D2H sync inside for the cell size).
 * means_dev may be NULL.  Equivalent of filter_sor_gpu(data, k, threshold_factor). */
int gsx_sor_filter_device(const float* xyz_dev, int64_t n, int32_t k, float threshold_factor, int32_t hash_mode,
                          uint8_t* mask_dev, float* means_dev, void* ws, int64_t ws_bytes, void* stream);

/* Whole filter on HOST buffers: the binding target for gpu_ops.filter_sor_gpu (gpu_ops.py:193).
 * xyz_host float32[n,3]; mask_host uint8[n]; means_host float32[n] or NULL. */
int gsx_sor_filter_host(const float* xyz_host, int64_t n, int32_t k, float threshold_factor, int32_t hash_mode,
                        uint8_t* mask_host, float* means_host);

/* ---- SOR, cKDTree semantics: data_processor.py:155-180 (the reference's CPU path) ------------ */
/* data_processor.py:160-173: exact (k+1)-NN in float64 over the float32 coordinates (the nearest is the
 * point itself or a coincident twin and is dropped), mean of neighbours 1..k in float64 (NumPy pairwise
 * row reduction), stored as float32 in the caller's point order.  1 <= k <= 63. */
int64_t gsx_knn_exact_workspace_bytes(int64_t n);
int gsx_knn_exact_mean_dists(const float* xyz_dev, int64_t n, int32_t k, float* means_dev, void* ws, int64_t ws_bytes,
                             void* stream);
/* the same plus data_processor.py:176-180 (threshold and mask -- the mask the reference computes and then
 * discards, SURVEY F5) on HOST buffers. */
int gsx_sor_ckdtree_filter_host(const float* xyz_host, int64_t n, int32_t k, float threshold_factor, uint8_t* mask_host,
                                float* means_host);

/* ---- bbox / alpha masks: data_processor.py:215-231, :184-213 ------------------------ */
/* keep <=> lo <= v <= hi on all axes, float32 compares (bounds already rounded to float32 by caller). */
int gsx_bbox_mask(const float* xyz_dev, int64_t n, const float* lohi_host /*[6]*/, uint8_t* mask_dev, void* stream);
/* keep <=> (double)opacity >= logit_thresh (float64 compare, data_processor.py:208). */
int gsx_alpha_mask(const float* opacity_dev, int64_t n, double logit_thresh, uint8_t* mask_dev, void* stream);
/* host helper: data_processor.py:203-205 -> logit threshold for min_opacity_u8 in (0,255), libm log
 * (NumPy's SIMD log may differ by one float64 ulp; the Python plugin passes NumPy's own value). */
double gsx_alpha_logit_threshold(double min_opacity_u8);

/* ---- compaction of the filters' working set: the `vertices[mask]` steps of data_processor.py:114,149,209,
 * 217-224 for the columns the filters read (xyz, opacity) plus the surviving ORIGINAL row indices; stable like
 * NumPy boolean indexing.  opacity_dev/opacity_out_dev may both be NULL; idx_dev NULL = identity.
 * *count_host = number of survivors (one 4-byte D2H sync). */
int64_t gsx_compact_workspace_bytes(int64_t n);
int gsx_compact_points(const uint8_t* mask_dev, int64_t n, const float* xyz_dev, const float* opacity_dev,
                       const int32_t* idx_dev, float* xyz_out_dev, float* opacity_out_dev, int32_t* idx_out_dev,
                       int64_t* count_host, void* ws, int64_t ws_bytes, void* stream);

/* ---- density filter: data_processor.py:38-52 (voxel histogram) and :111-112 (member mask) ---- */
int64_t gsx_density_workspace_bytes(int64_t n, int64_t cap);
/* q = floor(xyz / f32(voxel)) -> int64 triple (data_processor.py:39); counts per voxel (:43); every voxel
 * with count >= max(min_points,1) (:48-51) is returned to the HOST arrays dense_vox_host (int64[cap,3]) and
 * dense_cnt_host (int32[cap]), in no particular order; *n_dense_host = how many (> cap => GSX_ERR_WORKSPACE);
 * *n_voxels_host (may be NULL) = number of distinct voxels (len(unique_voxels), :45). */
int gsx_density_voxel_count(const float* xyz_dev, int64_t n, float voxel, int64_t min_points, int64_t* dense_vox_host,
                            int32_t* dense_cnt_host, int64_t cap, int64_t* n_dense_host, int64_t* n_voxels_host,
                            void* ws, int64_t ws_bytes, void* stream);
/* data_processor.py:111-112: mask[i] = voxel(point i) is one of the n_keep voxels of keep_vox_host
 * (HOST int64[n_keep,3], the output of the host-side cluster selection :59-106). */
int gsx_density_member_mask(const float* xyz_dev, int64_t n, float voxel, const int64_t* keep_vox_host, int64_t n_keep,
                            uint8_t* mask_dev, void* ws, int64_t ws_bytes, void* stream);

/* Staged form for sharded clouds (one process per GPU): every rank counts its slab into an int32 grid over
 * the GLOBAL voxel box (q0[3], dim[3] voxels; from the all-reduced min/max via gsx_density_voxel_range), the
 * caller all-reduces the grid (sum) and extracts the dense voxels from it.  Same results as
 * gsx_density_voxel_count on the union cloud.  *oob_dev counts points outside the box (must stay 0). */
void gsx_density_voxel_range(const float* minmax_host /*[6]*/, float voxel, int64_t* q0_out, int64_t* dim_out);
int gsx_density_grid_count(const float* xyz_dev, int64_t n, float voxel, const int64_t* q0, const int64_t* dim,
                           int32_t* grid_dev, unsigned long long* oob_dev, void* stream);
int gsx_density_grid_dense(const int32_t* grid_dev, const int64_t* q0, const int64_t* dim, int64_t min_points,
                           int64_t* dense_vox_host, int32_t* dense_cnt_host, int64_t cap, int64_t* n_dense_host,
                           int64_t* n_voxels_host, void* ws, int64_t ws_bytes, void* stream);

/* ---- SOG writer helpers, the steps either side of K-Means (SURVEY 8(f) item 1) ------------------- */
/* formats/sog.py:264  np.lexsort((z, y, x)): order_dev[j] = index of the j-th splat in (x, then y, then z) order,
 * stable; -0.0 == +0.0 as in NumPy.  (NaN coordinates are not supported.) */
int64_t gsx_lexsort_workspace_bytes(int64_t n);
int gsx_lexsort_zyx(const float* xyz_dev, int64_t n, int32_t* order_dev, void* ws, int64_t ws_bytes, void* stream);
/* formats/sog.py:408-419 quantize_to_codebook: index of the nearest entry of an ascending float32 codebook
 * (searchsorted-left, clip, prefer the left neighbour if strictly closer), as uint8.  1 <= m <= 4096; ws >= 4*m B. */
int gsx_quantize_to_codebook(const float* vals_dev, int64_t n, const float* codebook_host, int32_t m,
                             uint8_t* labels_dev, void* ws, int64_t ws_bytes, void* stream);

/* ---- K-Means: gpu_ops.py:57-96 (kernels) + :186-188 (Lloyd loop) ---------------------- */
/* Batched over `nprob` independent problems stored back to back (SOG shN chunks, sog.py:527-549):
 * problem p has rows [row_off[p], row_off[p+1]) of X[*,D] and K centroids at C[p*K*D].
 * One call = max_iter x (assign ; update) with the serial index-order float32 sums of SURVEY A.5.
 * labels are those of the last assign (one update behind C, SURVEY F9); counts int32[nprob*K]. */
int64_t gsx_kmeans_workspace_bytes(int64_t n_total, int32_t nprob, int32_t K, int32_t D);
/* assign_mode (per call; the labels are bit-identical in every mode):
 *   AUTO           tensor cores when the shape allows it (gsx_kmeans_tensor_core_supported), else STRICT
 *   STRICT         the contract's distance for every (point, centroid) on the FP32 pipes
 *   FMA_PREFILTER  D >= 9: one fma per (point, centroid, dim) scores every centroid, the strict distance is
 *                  evaluated only for the centroids within a proven rounding-error margin of the best score
 *   TENSOR         the same scheme with the score matrix X.C^T - ||c||^2/2 computed by tcgen05.mma (kind::tf32, float32
 *                  accumulators in TMEM, two-pass epilogue: row maximum, candidate mask); error if the shape is
 *                  unsupported (D in {9,24,45}, K <= 256)
 *   TENSOR_BF16    variant with split-bf16 operands (x = x1 + x2, three kind::f16 MMAs per K step, score error 2^-16
 *                  instead of 2^-9, so ~0.2 % instead of ~9 % of the points need a strict evaluation) and a single-pass
 *                  packed-key top-2 epilogue; measured slower than TENSOR on B200 (the top-2 costs more ALU work than
 *                  it saves in TMEM reads, profiles/r02_km_tc16_ncu.json).  A BUILD-TIME experiment: the shipped library
 *                  returns GSX_ERR_UNSUPPORTED for it unless gsx_kmeans_tc.cu was compiled with -DGSX_KM_TC16=1
 *                  (gsx_kmeans_tensor_core_supported reports bit 1 then)
 * tc_stats_dev (may be NULL): 3 uint64 counters accumulated by the TENSOR path {strict distance evaluations,
 * points with more than one candidate, points that needed the full strict scan}. */
#define GSX_KM_ASSIGN_AUTO 0
#define GSX_KM_ASSIGN_STRICT 1
#define GSX_KM_ASSIGN_FMA_PREFILTER 2
#define GSX_KM_ASSIGN_TENSOR 3
#define GSX_KM_ASSIGN_TENSOR_BF16 4
int gsx_kmeans_lloyd_device(const float* X_dev, const int64_t* row_off_host, int32_t nprob, int32_t K, int32_t D,
                            int32_t max_iter, float* C_dev, int32_t* labels_dev, int32_t* counts_dev, void* ws,
                            int64_t ws_bytes, int32_t assign_mode, unsigned long long* tc_stats_dev, void* stream);
/* 0: shape unsupported; bit 0: the TF32 kernel takes it; bit 1: the split-bf16 variant is compiled in */
int32_t gsx_kmeans_tensor_core_supported(int32_t K, int32_t D);
/* Test hook of the tensor-core assign: raw scores s[r][c] = x_r.c - ||c||^2/2 of the first min(rows,128) rows
 * against the K centroids, scores_dev float32[128 * roundup32(K)].  ws >= 1024 bytes. */
int gsx_kmeans_tc_debug_scores(const float* X_dev, int64_t rows, const float* C_dev, int32_t K, int32_t D,
                               int32_t variant, float* scores_dev, void* ws, int64_t ws_bytes, void* stream);
/* Single problem on HOST buffers: binding target for gpu_ops.kmeans on the GPU path (gpu_ops.py:178-191)
 * with the init centroids chosen by the caller (the reference's np.random.choice draw). */
int gsx_kmeans_host(const float* X_host, int64_t n, int32_t K, int32_t D, int32_t max_iter, float* C_host_inout,
                    int32_t* labels_host, int32_t assign_mode);

/* ---- device-resident splat records (SURVEY 8(f) items 2 and 4) ------------------------------------------------
 * rows_dev: the reference's interchange records (structures.py:23-59) as a row-major float32 matrix [n, F]
 * (F = 62 for SH degree 3), uploaded once.  Column arguments are field positions inside a row.
 *  extract : np.column_stack((x,y,z)) / v['opacity'] of data_processor.py:38,139,184 -> xyz [n,3], opacity [n] (or NULL)
 *  gather  : vertices[mask] of data_processor.py:114,149,209,224 for the surviving (ascending) row indices
 *  color   : RGBA8 of formats/splat.py:131-144, ksplat.py:464-468: clip((0.5 + scale*f_dc)*255).astype(u8) x3 (bit-exact
 *            float32 ops; scale = SH_C0 for .splat/.ksplat, 0.15 for spz.py:131) and clip(sigmoid(opacity)*255).astype(u8)
 *            (expf: may differ from NumPy's SIMD exp by one count on a ~1e-5 fraction of the splats)
 *  scale   : np.exp(scale_0..2) of formats/splat.py:108, ksplat.py:447 -> float32 [n,3] */
int gsx_records_extract_xyz_opacity(const float* rows_dev, int64_t n, int32_t F, int32_t cx, int32_t cy, int32_t cz,
                                    int32_t cop, float* xyz_dev, float* opacity_dev, void* stream);
int gsx_records_gather_rows(const float* rows_dev, const int32_t* idx_dev, int64_t m, int32_t F, float* out_dev,
                            void* stream);
int gsx_records_color_rgba8(const float* rows_dev, int64_t n, int32_t F, int32_t c0, int32_t c1, int32_t c2, int32_t cop,
                            float scale, uint8_t* rgba_dev, void* stream);
int gsx_records_scale_exp(const float* rows_dev, int64_t n, int32_t F, int32_t s0, int32_t s1, int32_t s2, float* out_dev,
                          void* stream);

/* ---- Morton ordering as a shared primitive (SURVEY 8(f) item 3) ----------------------------------------------
 * formats/compressed_ply.py:252-297 (_sort_morton_order): order_dev[j] = index of the j-th splat in the recursive
 * 3 x 10-bit Morton order (codes relative to the bounding box of the group; every run of equal codes longer than
 * run_limit (the reference: 256) is re-normalised to its own box and sorted again, until it is short or has no
 * extent).  Equal codes inside a finished run come out in ascending original index (the reference's unstable
 * np.argsort leaves that order unspecified).  *levels_out = number of levels that ran. */
int64_t gsx_morton_workspace_bytes(int64_t n);
int gsx_morton_order(const float* xyz_dev, int64_t n, int32_t* order_dev, int32_t run_limit, int32_t* levels_out, void* ws,
                     int64_t ws_bytes, void* stream);
/* compressed_ply.py:206-246 (per-256-splat chunk bounds) / ksplat.py:426-441 (np.minimum/maximum.reduceat per
 * bucket): min and max of ncol (<= 8) columns cols_host[] of the row-major float32 matrix rows_dev [n,F] over
 * consecutive chunks of `chunk` rows taken in the order order_dev (NULL = identity); values are clipped to
 * [clip_lo, clip_hi] first (np.clip(scale, -20, 20) of compressed_ply.py:213-215; pass -inf/+inf for none).
 * lo_dev / hi_dev: float32 [ceil(n/chunk), ncol].  ws >= 64 bytes. */
int gsx_chunk_minmax(const float* rows_dev, int64_t n, int32_t F, const int32_t* order_dev, int32_t chunk,
                     const int32_t* cols_host, int32_t ncol, float clip_lo, float clip_hi, float* lo_dev, float* hi_dev,
                     void* ws, int64_t ws_bytes, void* stream);

/* The SOG shN schedule (formats/sog.py:536-549: up to 64 chunks of one SH block, each clustered by its own
 * gpu_ops.kmeans call) in ONE call on HOST buffers: one upload of the block, one batched launch per phase.
 * nprob problems back to back in X_host (rows row_off[p] .. row_off[p+1]), K centroids each;
 * C_host_inout float32[nprob*K*D]: the init rows on entry, the centroids on return; labels_host int32[n]. */
int gsx_kmeans_host_batched(const float* X_host, const int64_t* row_off_host, int32_t nprob, int32_t K, int32_t D,
                            int32_t max_iter, float* C_host_inout, int32_t* labels_host, int32_t assign_mode);
/* Copies between a caller's HOST buffer and HBM, used by every *_host entry point above.  The reference's call sites
 * pass ordinary (pageable) NumPy arrays -- np.column_stack at data_processor.py:139, the shN block of
 * sog.py:536-549 -- which cudaMemcpy stages on one CPU thread at ~11 GB/s; these stage through a pool of pinned
 * chunks filled / drained by several host threads (GSX_COPY_THREADS, default 8), each enqueueing its own DMAs, so
 * the PCIe link stays busy.  Pinned / registered / managed buffers and copies below 8 MiB take plain
 * cudaMemcpyAsync (GSX_STAGED_COPY=0 forces that path).
 * gsx_copy_h2d: on return src_host has been read completely and `stream` is ordered after the last chunk.
 * gsx_copy_d2h: waits for what `stream` has produced and BLOCKS until dst_host is complete. */
int gsx_copy_h2d(void* dst_dev, const void* src_host, int64_t bytes, void* stream);
int gsx_copy_d2h(void* dst_host, const void* src_dev, int64_t bytes, void* stream);
/* HOST-side row movement around the device filter chain when the 248-byte records stay on the host (no GPU work, several
 * CPU threads -- GSX_HOST_THREADS, default 16 on a big host): what the reference does with single-threaded NumPy.
 * gsx_host_gather_rows: dst[j] = src[idx[j]] for rows of row_bytes bytes -- the `vertices[mask]` compaction of
 *   data_processor.py:114,149,209,224 with the surviving row indices; every idx must lie in [0, n_rows).
 * gsx_host_extract_xyz_opacity: np.column_stack((v['x'], v['y'], v['z'])) and v['opacity'] of data_processor.py:38,139
 *   from packed records; the fields are float32 at the given byte offsets of a row (off_opacity < 0 and a null
 *   opacity_out_host: no opacity field). */
int gsx_host_gather_rows(const void* src_host, int64_t n_rows, int64_t row_bytes, const int64_t* idx_host, int64_t m,
                         void* dst_host);
int gsx_host_extract_xyz_opacity(const void* src_host, int64_t n_rows, int64_t row_bytes, int64_t off_x, int64_t off_y,
                                 int64_t off_z, int64_t off_opacity, float* xyz_out_host, float* opacity_out_host);
/* Free / total memory of the current device, for the sizing decisions of the host-buffer callers. */
int gsx_device_memory(int64_t* free_bytes, int64_t* total_bytes);

#ifdef __cplusplus
}
#endif
#endif /* GSX_H */
