// One warp sorts 128-bit keys in place: the bitonic network shared by the --write-details rows (wfl_details.cu) and
// the device-built scoring batch (wfl_resident_batch.cu).
#pragma once

#include "wfl_warp_common.cuh"

namespace wfl {
namespace {

// 128-bit keys (hi, lo), ascending; a warp sorts n (a power of two) of them in place (bitonic network)
__device__ __forceinline__ bool key_less(const ulonglong2 &a, const ulonglong2 &b) {
    return a.x < b.x || (a.x == b.x && a.y < b.y);
}
__device__ __noinline__ void warp_sort(ulonglong2 *v, int n) {
#pragma unroll 1
    for (int k = 2; k <= n; k <<= 1)
#pragma unroll 1
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll 1
            for (int i = lane_id(); i < n; i += 32) {
                const int ij = i ^ j;
                if (ij > i) {
                    const ulonglong2 a = v[i], b = v[ij];
                    if (((i & k) == 0) == key_less(b, a)) { v[i] = b; v[ij] = a; }
                }
            }
            __syncwarp();
        }
}

__device__ __forceinline__ int pow2_at_least(int n) {
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}

}  // namespace
}  // namespace wfl
