// common.cuh -- shared device/host helpers for the sm_100a selective-scan library.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gfe_mamba_b200.h"

namespace gfe {

// ---- host side ------------------------------------------------------------
void set_error(const char *fmt, ...);
int check_launch(const char *what);   // cudaPeekAtLastError -> GFE_OK / GFE_ERR_CUDA
int sm_count();                       // SMs of the current device (148 on B200; 148 assumed if no device)

// kernel ids of the optional timing registry (api.cu)
enum KernelId {
    K_SELSCAN_FWD_SUMMARY = 0, K_SELSCAN_FWD, K_SELSCAN_BWD_SUMMARY, K_SELSCAN_BWD, K_SELSCAN_BWD_FIN_BC,
    K_SELSCAN_BWD_FIN_PAR, K_PSCAN_FWD_SUMMARY, K_PSCAN_FWD, K_PSCAN_BWD_SUMMARY, K_PSCAN_BWD,
    K_CONV_FWD, K_CONV_BWD, K_CONV_BWD_FIN, K_CONV_STEP, K_SSM_STEP, K_ADDNORM_FWD, K_ADDNORM_BWD, K_ADDNORM_BWD_FIN, K_OPT_SUMSQ, K_OPT_COEF, K_OPT_ADAM, K_POOL_FWD, K_POOL_BWD, K_COUNT
};
void timing_mark(int id, cudaStream_t st, bool begin);
struct ScopedKernelTimer {   // brackets one launch with events when timing is enabled
    int id; cudaStream_t st;
    ScopedKernelTimer(int id_, cudaStream_t st_) : id(id_), st(st_) { timing_mark(id, st, true); }
    ~ScopedKernelTimer() { timing_mark(id, st, false); }
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr int kNState = 16;     // d_state of the chained kernels (the generic kernels and the decode kernel also take 32 and 64)
// d_state values the fused scan and decode kernels are compiled for; every other value is GFE_ERR_UNSUPPORTED
static inline bool fused_d_state(int N) { return N == 16 || N == 32 || N == 64; }
constexpr int kChunk = 16;      // time steps per register chunk == checkpoint interval
constexpr int kMaxSeg = 256;    // max L-split factor (one long sequence sharded over 8 GPUs: 128 channels, 256 segments of 256 steps)
constexpr int kCkptV2 = 8;      // checkpoint interval of the chained kernels: halves the register-resident history of backward

// How one (b, channel) sequence is split along L when B*ED alone cannot fill the GPU.
struct SegPlan {
    int nseg;     // S: number of segments (1 = no split, single pass)
    int seg_len;  // steps per segment, multiple of kChunk
    int nchunks;  // ceil(L / kChunk)
};
SegPlan plan_segments(int B, int L, int ED);

// ---- device side ----------------------------------------------------------
#ifdef __CUDACC__

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

// streaming (read-once) global load / store: do not pollute L1
template <typename T> __device__ __forceinline__ T ld_stream(const T *p) { return __ldcs(p); }
template <typename T> __device__ __forceinline__ void st_stream(T *p, T v) { __stcs(p, v); }

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// packed fp32x2 math (FFMA2 / FMUL2 / FADD2 on sm_100)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 ex2_2(float2 x) { return make_float2(ex2_approx(x.x), ex2_approx(x.y)); }

// softplus(x) = log(1 + e^x), threshold 20 as torch.nn.functional.softplus (mamba.py:256).
// Also returns sigmoid(x) = d softplus / dx.  Relative accuracy ~1e-7 for all x:
// small e uses log1p(e) = 2 atanh(e / (2 + e)) because lg2.approx has only ABSOLUTE accuracy near 1.
__device__ __forceinline__ float softplus_sig(float x, float &sig) {
    if (x > 20.0f) {
        sig = 1.0f;
        return x;
    }
    const float e = ex2_approx(x * kLog2e);
    const float w = 1.0f + e;
    sig = e * rcp_approx(w);
    if (e < 0.5f) {
        const float s = e * rcp_approx(2.0f + e);
        const float s2 = s * s;
        float p = fmaf(s2, 1.0f / 9.0f, 1.0f / 7.0f);
        p = fmaf(s2, p, 1.0f / 5.0f);
        p = fmaf(s2, p, 1.0f / 3.0f);
        p = fmaf(s2, p, 1.0f);
        return 2.0f * s * p;
    }
    return kLn2 * lg2_approx(w);
}
__device__ __forceinline__ float softplus_only(float x) {
    if (x > 20.0f) return x;
    const float e = ex2_approx(x * kLog2e);
    if (e < 0.5f) {
        const float s = e * rcp_approx(2.0f + e);
        const float s2 = s * s;
        float p = fmaf(s2, 1.0f / 9.0f, 1.0f / 7.0f);
        p = fmaf(s2, p, 1.0f / 5.0f);
        p = fmaf(s2, p, 1.0f / 3.0f);
        p = fmaf(s2, p, 1.0f);
        return 2.0f * s * p;
    }
    return kLn2 * lg2_approx(1.0f + e);
}
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_approx(1.0f + ex2_approx(-x * kLog2e)); }

#endif  // __CUDACC__
}  // namespace gfe
