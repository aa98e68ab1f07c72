// Shared helpers for librdfc_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rdfc_b200.h"

namespace rdfc {

// thread-local error string behind rdfc_last_error()
char *err_buf();
int fail(int code, const char *fmt, ...);
void count_launch(unsigned n = 1);

#define RDFC_REQUIRE(cond, ...)                                   \
    do {                                                          \
        if (!(cond)) return ::rdfc::fail(RDFC_ERR_INVALID, __VA_ARGS__); \
    } while (0)

#define RDFC_CHECK_LAUNCH(name)                                                                   \
    do {                                                                                          \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess)                                                                   \
            return ::rdfc::fail(RDFC_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e__));          \
        ::rdfc::count_launch();                                                                   \
    } while (0)

#define RDFC_CUDA(call)                                                                           \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return ::rdfc::fail(RDFC_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e__));         \
    } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// number of SMs of the current device (cached)
int sm_count();

// development knob `name` (an RDFC_* environment variable, read once and cached; rdfc_dev_set_knob overrides it), or dflt
constexpr long long KNOB_UNSET = (long long)0x8000000000000000ull;
long long knob(const char *name, long long dflt);

// ---- storage helpers: fp32 compute, fp32 / bf16 storage -------------------------------------------------------
__device__ __forceinline__ float ldf(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ldf(const __nv_bfloat16 *p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float *p, float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }

// Split-precision operands are fp16 halves x = hi + lo, and fp16 has a narrow exponent range: a tensor is scaled by the power of two s
// with amax * s in [1024, 2048) before it is split, so that lo keeps 11 significant bits down to ~3e-5 of the largest element.
// 1 for an all-zero (or non-finite) tensor.
__device__ __forceinline__ float pow2_scale(float amax) {
    if (!(amax > 0.f) || !(amax < 3.0e38f)) return 1.f;
    int ex;
    frexpf(amax, &ex);                       // amax = f * 2^ex, f in [0.5, 1)
    ex = 11 - ex;
    ex = ex > 100 ? 100 : (ex < -100 ? -100 : ex);
    return exp2f((float)ex);
}

__device__ __forceinline__ float apply_act(float v, int act) {
    switch (act) {
        case RDFC_ACT_RELU: return fmaxf(v, 0.f);
        case RDFC_ACT_LEAKY02: return v > 0.f ? v : 0.2f * v;
        case RDFC_ACT_TANH: return tanhf(v);
        case RDFC_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        default: return v;
    }
}

}  // namespace rdfc
