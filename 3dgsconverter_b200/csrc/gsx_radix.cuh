#pragma once
#include "gsx_common.cuh"
namespace gsx {
size_t radix_ws_bytes(int64_t n);
// in-place exclusive scan of n uint32 (multi-level block scan); scratch from scan_workspace_bytes(n)
size_t scan_workspace_bytes(int64_t n);
int exclusive_scan_u32_ws(uint32_t* data, int64_t n, uint32_t* ws, cudaStream_t st);
// Stable LSD sort of the bits [begin_bit, end_bit) of keys0 (payload vals0); keys1/vals1 are the ping-pong
// buffers.  *keys_sorted / *vals_sorted receive the buffers that hold the result.  1 <= n < 2^32: onesweep passes
// below GSX_RADIX_ONESWEEP_MAX_N (2^30), three-kernel passes from there on.
int radix_sort_pairs(uint64_t* keys0, uint64_t* keys1, int32_t* vals0, int32_t* vals1, int64_t n, int begin_bit,
                     int end_bit, void* ws, size_t ws_bytes, uint64_t** keys_sorted, int32_t** vals_sorted,
                     cudaStream_t st);
// Bare 64-bit words (payload packed into the bits below begin_bit by the caller); same range and passes as the pairs.
int radix_sort_keys(uint64_t* keys0, uint64_t* keys1, int64_t n, int begin_bit, int end_bit, void* ws, size_t ws_bytes,
                    uint64_t** keys_sorted, cudaStream_t st);
}
