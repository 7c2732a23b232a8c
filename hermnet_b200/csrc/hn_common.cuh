// Shared helpers for the hermnet_b200 CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <type_traits>

#include "../../include/hermnet_b200.h"

namespace hn {

extern thread_local std::string g_last_error;

inline int fail(const char *where, const char *msg) {
    g_last_error = std::string(where) + ": " + msg;
    return 1;
}

inline int check_launch(const char *where) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(where, cudaGetErrorString(e));
    return 0;
}

#define HN_CUDA(call, where)                                      \
    do {                                                          \
        cudaError_t _e = (call);                                  \
        if (_e != cudaSuccess) return hn::fail(where, cudaGetErrorString(_e)); \
    } while (0)

#define HN_REQUIRE(cond, where, msg) \
    do {                             \
        if (!(cond)) return hn::fail(where, msg); \
    } while (0)

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// Runtime flag -> template argument: calls f(std::true_type{}) or f(std::false_type{}).
template <class Fn>
inline void dispatch_bool(bool b, Fn &&f) {
    if (b) f(std::true_type{});
    else f(std::false_type{});
}

inline int num_sms() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return -1;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
        cached = n;
    }
    return cached;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// vector load/store of VEC consecutive floats (VEC in {1,2,4}), read-only path for loads
template <int VEC>
struct Vec {
    float v[VEC];
};

template <int VEC>
__device__ __forceinline__ Vec<VEC> ldv(const float *p) {
    Vec<VEC> r;
    if constexpr (VEC == 4) {
        float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
    } else if constexpr (VEC == 2) {
        float2 t = __ldg(reinterpret_cast<const float2 *>(p));
        r.v[0] = t.x; r.v[1] = t.y;
    } else {
        r.v[0] = __ldg(p);
    }
    return r;
}

template <int VEC>
__device__ __forceinline__ void stv(float *p, const Vec<VEC> &r) {
    if constexpr (VEC == 4) {
        *reinterpret_cast<float4 *>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
    } else if constexpr (VEC == 2) {
        *reinterpret_cast<float2 *>(p) = make_float2(r.v[0], r.v[1]);
    } else {
        *p = r.v[0];
    }
}

}  // namespace hn
