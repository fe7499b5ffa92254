// Shared helpers for libgen6d_b200.so (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/gen6d_b200.h"

namespace g6d {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

inline cudaStream_t as_stream(g6d_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// call after every kernel launch
#define G6D_CHECK_LAUNCH(name)                                                        \
    do {                                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) {                                                     \
            g6d::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));   \
            return G6D_ECUDA;                                                         \
        }                                                                             \
        g6d::count_launch();                                                          \
    } while (0)

#define G6D_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            g6d::set_error(__VA_ARGS__);  \
            return G6D_EINVAL;            \
        }                                 \
    } while (0)

constexpr int kNumSMs = 148;  // B200

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
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// streaming (read-once) 128-bit load that does not pollute L1
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// g6d_conv_desc.in_items: 0 (one input item per output item) or a divisor of B (the input is broadcast)
inline bool in_items_ok(const g6d_conv_desc* d) { return d->in_items == 0 || (d->in_items > 0 && d->B % d->in_items == 0); }
// the conv kernels index the prologue operands (scale [groups, (D*H*W,) Cin]) with 32-bit offsets
inline bool pro_operands_fit(const g6d_conv_desc* d) {
    if (d->prologue == G6D_PRO_NONE) return true;
    const long long gr = d->group_rows > 0 ? d->group_rows : 1;
    const long long groups = (d->B + gr - 1) / gr;
    const long long per = d->prologue == G6D_PRO_CORR ? (long long)d->D * d->H * d->W : 1;
    return groups * per * d->Cin < (1ll << 31);
}

}  // namespace g6d
