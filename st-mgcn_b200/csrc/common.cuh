// Shared host/device helpers for libstmgcn_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/stmgcn_b200.h"

namespace stmgcn {

// ---- error reporting across the C boundary (no exceptions; thread-local message) -------------------
void set_error(const char* fmt, ...);
int32_t fail(int32_t code, const char* fmt, ...);
int32_t check_launch(const char* what);        // cudaGetLastError() only -- never synchronises
void count_launch(int n = 1);
int sm_count();
int32_t ensure_dyn_smem(const void* kernel, size_t bytes);   // per-(kernel, device) cudaFuncAttributeMaxDynamicSharedMemorySize

#define STMGCN_REQUIRE(cond, code, ...)                                   \
    do {                                                                  \
        if (!(cond)) return ::stmgcn::fail((code), __VA_ARGS__);          \
    } while (0)

#define STMGCN_CUDA(expr)                                                                     \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return ::stmgcn::fail((int32_t)_e, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- device helpers ---------------------------------------------------------------------------------
// sigmoid / tanh on the MUFU pipe: ex2.approx + rcp.approx (~2 ulp each); absolute error < 1e-6, far inside
// the 1e-4 parity budget, and 2 MUFU + 3 FP32 ops per value instead of an IEEE division sequence.
// Written with the .ftz MUFU forms directly: __expf / __fdividef wrap the same instructions in denormal-range fix-ups
// (FSETP + two predicated FMUL per ex2, a range test per division) that the saturating activations do not need --
// e^-v below 1e-38 contributes nothing to 1 + e^-v, and rcp(inf) = 0 is the correct limit.  4 / 5 instructions per value.
__device__ __forceinline__ float ex2_ftz_(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_ftz_(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sigmoidf_(float v) { return rcp_ftz_(1.0f + ex2_ftz_(-1.4426950408889634f * v)); }
__device__ __forceinline__ float tanhf_(float v) {
    return fmaf(2.0f, rcp_ftz_(1.0f + ex2_ftz_(-2.8853900817779268f * v)), -1.0f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace stmgcn
