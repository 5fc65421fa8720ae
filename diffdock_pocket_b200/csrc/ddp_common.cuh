// Shared helpers for the ddp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ddp_b200.h"

#define DDP_LAUNCH_CHECK()                                  \
    do {                                                    \
        cudaError_t e__ = cudaGetLastError();               \
        if (e__ != cudaSuccess) return (int)e__;            \
    } while (0)

// Per-device caches: cudaFuncSetAttribute and the SM count belong to a DEVICE, not to the process -- a process that
// drives several GPUs through this library must opt in / count on each of them.
constexpr int DDP_MAX_DEVICES = 64;
static inline int ddp_current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < DDP_MAX_DEVICES ? dev : 0;
}
static inline int ddp_num_sms() {
    static int n[DDP_MAX_DEVICES] = {0};
    const int dev = ddp_current_device();
    if (n[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        n[dev] = v > 0 ? v : 148;
    }
    return n[dev];
}
// Opt a kernel in to `bytes` of dynamic shared memory once per device.  `done` is a caller-owned static
// bool[DDP_MAX_DEVICES] (one per kernel instantiation).
template <typename K>
static inline cudaError_t ddp_smem_opt_in(K kernel, size_t bytes, bool *done) {
    const int dev = ddp_current_device();
    if (done[dev]) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) done[dev] = true;
    return e;
}

// Fixed-point accumulation of the deterministic mode (DDP_ACC_FIXED_SHIFT, include/ddp_b200.h).  The range test also
// rejects NaN; a rejected partial adds 0 and raises the status bit instead of wrapping into a wrong integer.
__device__ __forceinline__ unsigned long long ddp_to_fixed(float v, uint32_t *status) {
    constexpr float kScale = (float)(1ull << DDP_ACC_FIXED_SHIFT);
    constexpr float kRange = (float)(1ull << (63 - DDP_ACC_FIXED_SHIFT));     // 2^31: |v * 2^S| < 2^63
    if (!(fabsf(v) < kRange)) {
        atomicOr(status, DDP_STATUS_FIXED_RANGE);
        return 0ull;
    }
    return (unsigned long long)__float2ll_rn(v * kScale);
}
__device__ __forceinline__ float ddp_from_fixed(long long q) {
    return __ll2float_rn(q) * (1.f / (float)(1ull << DDP_ACC_FIXED_SHIFT));
}

__device__ __forceinline__ int ddp_find_segment(const int32_t *__restrict__ ptr, int n_seg, int i) {
    // largest b with ptr[b] <= i  (ptr ascending, ptr[n_seg] = total)
    int lo = 0, hi = n_seg;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (ptr[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ float ddp_sqdist(float ax, float ay, float az, float bx, float by, float bz) {
    // torch_cluster kernels: dist += (x_d - y_d) * (x_d - y_d) for d = 0,1,2 with nvcc's default FMA contraction
    float t = ax - bx;
    float d = __fmaf_rn(t, t, 0.f);
    t = ay - by;
    d = __fmaf_rn(t, t, d);
    t = az - bz;
    d = __fmaf_rn(t, t, d);
    return d;
}
