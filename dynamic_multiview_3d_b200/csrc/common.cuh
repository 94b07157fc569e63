// Shared helpers for libdmv3d (sm_100a).  Error handling follows include/dmv3d.h: every
// entry point returns an int code and records a thread-local message; nothing throws.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dmv3d.h"

namespace dmv {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void count_launch_named(const char* what);      // what: a string literal (kept by address)
void count_tc_launch();
long long tc_launches();

inline int fail(int code, const char* msg) {
    set_error("%s", msg);
    return code;
}

// checks the launch that was just issued (async errors surface at the caller's next sync) and counts it under its
// label (dmv_launch_count_named), so tests can tell which kernel form ran
inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    count_launch();
    count_launch_named(what);
    return DMV_OK;
}

#define DMV_REQUIRE(cond, code, msg) \
    do {                             \
        if (!(cond)) return ::dmv::fail((code), (msg)); \
    } while (0)

__host__ __device__ inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// TF 'SAME' padding: out = ceil(in/s), total = max((out-1)s + k - in, 0), before = total/2.
struct SamePad {
    int out, before, after;
};
__host__ __device__ inline SamePad same_pad(int in, int k, int s) {
    SamePad p;
    p.out = (in + s - 1) / s;
    int total = (p.out - 1) * s + k - in;
    if (total < 0) total = 0;
    p.before = total / 2;
    p.after = total - p.before;
    return p;
}

__device__ __forceinline__ float bf2f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ __nv_bfloat16 f2bf(float v) { return __float2bfloat16_rn(v); }

template <typename T>
__device__ __forceinline__ float load_as_float(const T* p);
template <>
__device__ __forceinline__ float load_as_float<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __bfloat162float(*p);
}
template <typename T>
__device__ __forceinline__ void store_from_float(T* p, float v);
template <>
__device__ __forceinline__ void store_from_float<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void store_from_float<__nv_bfloat16>(__nv_bfloat16* p, float v) {
    *p = __float2bfloat16_rn(v);
}

// activations in the reference's algebraic forms (tf_utils.py:25-33)
__device__ __forceinline__ float apply_act(float x, int act) {
    switch (act) {
        case DMV_ACT_LRELU: return 0.6f * x + 0.4f * fabsf(x);
        case DMV_ACT_RELU: return 0.5f * x + 0.5f * fabsf(x);
        case DMV_ACT_TANH: return tanhf(x);
        default: return x;
    }
}
// derivative evaluated from the post-activation output y (TF: slope f1 + f2*sign(x), sign(0)=0)
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
    switch (act) {
        case DMV_ACT_LRELU: return y > 0.f ? 1.0f : (y < 0.f ? 0.2f : 0.6f);
        case DMV_ACT_RELU: return y > 0.f ? 1.0f : 0.0f;  // y == 0 <=> x <= 0 (x == 0 has measure zero)
        case DMV_ACT_TANH: return 1.0f - y * y;
        default: return 1.0f;
    }
}

// TF ApplyAdam on one element (SURVEY 8(a) O1); shared by adam.cu and exchange.cu so both compile to the same arithmetic
__device__ __forceinline__ void adam_one(float& th, float g, float& m, float& v, float lr_t, float omb1, float omb2, float eps) {
    m = m + (g - m) * omb1;
    v = v + (g * g - v) * omb2;
    th = th - (m * lr_t) / (sqrtf(v) + eps);
}

}  // namespace dmv
