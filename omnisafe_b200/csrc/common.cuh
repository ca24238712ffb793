// Shared device/host helpers for the omnisafe_b200 sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "omnisafe_b200.h"   // the C ABI: every entry point is defined against its prototype here

#define OSB_OK 0
#define OSB_ERR_ARG 1
#define OSB_ERR_CUDA 2
#define OSB_ERR_UNSUPPORTED 3

extern "C" void osb_set_error(const char* msg);
extern "C" void osb_count_launch(void);   // kernel-launch counter behind osb_launch_count() (bench.py: gpu_launches)

#define OSB_CHECK_ARG(cond, msg)                                   \
    do {                                                           \
        if (!(cond)) {                                             \
            osb_set_error("argument check failed: " msg);         \
            return OSB_ERR_ARG;                                    \
        }                                                          \
    } while (0)

#define OSB_CUDA(call)                                                               \
    do {                                                                             \
        cudaError_t e__ = (call);                                                    \
        if (e__ != cudaSuccess) {                                                    \
            char buf__[512];                                                         \
            snprintf(buf__, sizeof(buf__), "%s:%d: %s -> %s", __FILE__, __LINE__,    \
                     #call, cudaGetErrorString(e__));                                \
            osb_set_error(buf__);                                                    \
            return OSB_ERR_CUDA;                                                     \
        }                                                                            \
    } while (0)

#define OSB_LAUNCH_CHECK()              \
    do {                                \
        osb_count_launch();             \
        OSB_CUDA(cudaGetLastError());   \
    } while (0)

// Segment flag bits of the `flags[T][N]` slab (one byte per sample).
#define OSB_FLAG_TERMINATED 1u
#define OSB_FLAG_TRUNCATED 2u

namespace osb {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// lowbias32 integer finaliser; shared bit-for-bit with oracle/synthetic_env.py.
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16;
    x *= 0x7feb352dU;
    x ^= x >> 15;
    x *= 0x846ca68bU;
    x ^= x >> 16;
    return x;
}
__host__ __device__ __forceinline__ uint32_t hash4(uint32_t seed, uint32_t a, uint32_t b,
                                                   uint32_t c) {
    uint32_t h = mix32(seed ^ (a * 0x9E3779B1U));
    h = mix32(h ^ (b * 0x85EBCA77U));
    h = mix32(h ^ (c * 0xC2B2AE3DU));
    return h;
}
// uniform in [-1, 1), exactly representable in fp32.
__host__ __device__ __forceinline__ float u32_to_unit(uint32_t h) {
    return (float)(h >> 8) * (1.0f / 8388608.0f) - 1.0f;
}

}  // namespace osb
