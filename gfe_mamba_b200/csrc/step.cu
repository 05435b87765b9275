// step.cu -- single-token decode kernels (MambaBlock.step / ssm_step, cross_atten/mamba.py:342-405).
//
// The reference issues ~15 tiny ATen kernels per token per layer around the two small GEMMs
// (x_proj, dt_proj); these two kernels cover everything that is not a GEMM:
//   gfe_conv1d_step : conv over the cached K-1 inputs + the new one, bias, SiLU, cache roll  (mamba.py:357-358,370)
//   gfe_ssm_step    : softplus(delta + bias), h = exp(delta A) h + delta B u, y = h.C + D u, gate  (mamba.py:387-403,364-367)
#include "common.cuh"

namespace gfe {

template <typename T, int K>
__global__ void __launch_bounds__(128) conv1d_step_kernel(const T *xin, int64_t x_bs, T *inputs, const float *w,
                                                          const float *bias, T *u, int64_t u_bs, int B, int ED) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (c >= ED) return;
    T *cache = inputs + ((size_t)b * ED + c) * (K - 1);   // (B, ED, K-1)
    float win[K];
#pragma unroll
    for (int k = 0; k < K - 1; ++k) win[k] = to_f(cache[k]);
    const T xnew = xin[(int64_t)b * x_bs + c];
    win[K - 1] = to_f(xnew);
    float v = bias ? __ldg(bias + c) : 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) v = fmaf(__ldg(w + (size_t)c * K + k), win[k], v);
    u[(int64_t)b * u_bs + c] = from_f<T>(v * sigmoid_fast(v));
#pragma unroll
    for (int k = 0; k < K - 2; ++k) cache[k] = cache[k + 1];   // inputs[:, :, 1:] then append (mamba.py:370)
    if (K >= 2) cache[K - 2] = xnew;
}

template <typename T, int N>
__global__ void __launch_bounds__(128) ssm_step_kernel(const T *u, int64_t u_bs, const T *delta, int64_t d_bs,
                                                       const T *z, int64_t z_bs, const T *Bm, int64_t B_bs,
                                                       const T *Cm, int64_t C_bs, const float *A_log, const float *D,
                                                       const float *dt_bias, float *h, T *out, int64_t o_bs,
                                                       int B, int ED, uint32_t flags) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (c >= ED) return;
    float dl = to_f(delta[(int64_t)b * d_bs + c]) + (dt_bias ? __ldg(dt_bias + c) : 0.f);
    if (flags & GFE_FLAG_DELTA_SOFTPLUS) dl = softplus_only(dl);
    const float uj = to_f(u[(int64_t)b * u_bs + c]);
    const float du = dl * uj;
    float4 *hrow = reinterpret_cast<float4 *>(h + ((size_t)b * ED + c) * N);
    const float4 *arow = reinterpret_cast<const float4 *>(A_log + (size_t)c * N);
    const T *Bb = Bm + (int64_t)b * B_bs, *Cb = Cm + (int64_t)b * C_bs;
    float y = 0.f;
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
        float4 hv = hrow[q];
        const float4 al = __ldg(arow + q);
        const float a0 = -expf(al.x) * kLog2e, a1 = -expf(al.y) * kLog2e, a2 = -expf(al.z) * kLog2e, a3 = -expf(al.w) * kLog2e;
        hv.x = fmaf(ex2_approx(dl * a0), hv.x, du * to_f(Bb[4 * q + 0]));
        hv.y = fmaf(ex2_approx(dl * a1), hv.y, du * to_f(Bb[4 * q + 1]));
        hv.z = fmaf(ex2_approx(dl * a2), hv.z, du * to_f(Bb[4 * q + 2]));
        hv.w = fmaf(ex2_approx(dl * a3), hv.w, du * to_f(Bb[4 * q + 3]));
        y = fmaf(hv.x, to_f(Cb[4 * q + 0]), y);
        y = fmaf(hv.y, to_f(Cb[4 * q + 1]), y);
        y = fmaf(hv.z, to_f(Cb[4 * q + 2]), y);
        y = fmaf(hv.w, to_f(Cb[4 * q + 3]), y);
        hrow[q] = hv;
    }
    y = fmaf(__ldg(D + c), uj, y);
    if (z != nullptr) {
        const float zj = to_f(z[(int64_t)b * z_bs + c]);
        y *= zj * sigmoid_fast(zj);
    }
    out[(int64_t)b * o_bs + c] = from_f<T>(y);
}

template <typename T>
static int conv_step_launch(const void *xin, int64_t x_bs, void *inputs, const float *w, const float *bias, void *u,
                            int64_t u_bs, int B, int ED, int K, cudaStream_t st) {
    const dim3 block(128), grid((ED + 127) / 128, B);
    const T *x = reinterpret_cast<const T *>(xin);
    T *in = reinterpret_cast<T *>(inputs), *uo = reinterpret_cast<T *>(u);
    ScopedKernelTimer tm(K_CONV_STEP, st);
    switch (K) {
        case 2: conv1d_step_kernel<T, 2><<<grid, block, 0, st>>>(x, x_bs, in, w, bias, uo, u_bs, B, ED); break;
        case 3: conv1d_step_kernel<T, 3><<<grid, block, 0, st>>>(x, x_bs, in, w, bias, uo, u_bs, B, ED); break;
        case 4: conv1d_step_kernel<T, 4><<<grid, block, 0, st>>>(x, x_bs, in, w, bias, uo, u_bs, B, ED); break;
        default: set_error("conv1d_step: d_conv=%d unsupported (2..4 compiled)", K); return GFE_ERR_UNSUPPORTED;
    }
    return check_launch("conv1d_step");
}

template <typename T, int N>
static int ssm_step_launch(const void *u, int64_t u_bs, const void *delta, int64_t d_bs, const void *z, int64_t z_bs,
                           const void *Bm, int64_t B_bs, const void *Cm, int64_t C_bs, const float *A_log,
                           const float *D, const float *dt_bias, float *h, void *out, int64_t o_bs, int B, int ED,
                           uint32_t flags, cudaStream_t st) {
    const dim3 block(128), grid((ED + 127) / 128, B);
    ScopedKernelTimer tm(K_SSM_STEP, st);
    ssm_step_kernel<T, N><<<grid, block, 0, st>>>(reinterpret_cast<const T *>(u), u_bs, reinterpret_cast<const T *>(delta), d_bs,
                                                  reinterpret_cast<const T *>(z), z_bs, reinterpret_cast<const T *>(Bm), B_bs,
                                                  reinterpret_cast<const T *>(Cm), C_bs, A_log, D, dt_bias, h,
                                                  reinterpret_cast<T *>(out), o_bs, B, ED, flags);
    return check_launch("ssm_step");
}

// by state size (gfe_ssm_step has checked fused_d_state)
template <typename T>
static int ssm_step_launch_n(int N, const void *u, int64_t u_bs, const void *delta, int64_t d_bs, const void *z, int64_t z_bs,
                             const void *Bm, int64_t B_bs, const void *Cm, int64_t C_bs, const float *A_log,
                             const float *D, const float *dt_bias, float *h, void *out, int64_t o_bs, int B, int ED,
                             uint32_t flags, cudaStream_t st) {
    switch (N) {
        case 16: return ssm_step_launch<T, 16>(u, u_bs, delta, d_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, o_bs, B, ED, flags, st);
        case 32: return ssm_step_launch<T, 32>(u, u_bs, delta, d_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, o_bs, B, ED, flags, st);
        default: return ssm_step_launch<T, 64>(u, u_bs, delta, d_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, o_bs, B, ED, flags, st);
    }
}

}  // namespace gfe

extern "C" {

GFE_API int gfe_conv1d_step(const void *xin, int64_t x_bs, void *inputs, const float *w, const float *bias,
                            void *u, int64_t u_bs, int B, int ED, int K, int dtype, void *stream) {
    using namespace gfe;
    if (!xin || !inputs || !w || !u) { set_error("conv1d_step: NULL pointer"); return GFE_ERR_ARG; }
    if (B <= 0 || ED <= 0 || B > 65535) { set_error("conv1d_step: bad shape"); return GFE_ERR_ARG; }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    switch (dtype) {
        case GFE_F32: return conv_step_launch<float>(xin, x_bs, inputs, w, bias, u, u_bs, B, ED, K, st);
        case GFE_BF16: return conv_step_launch<__nv_bfloat16>(xin, x_bs, inputs, w, bias, u, u_bs, B, ED, K, st);
        case GFE_F16: return conv_step_launch<__half>(xin, x_bs, inputs, w, bias, u, u_bs, B, ED, K, st);
        default: set_error("conv1d_step: bad dtype %d", dtype); return GFE_ERR_DTYPE;
    }
}

GFE_API int gfe_ssm_step(const void *u, int64_t u_bs, const void *delta, int64_t delta_bs,
                         const void *z, int64_t z_bs, const void *Bm, int64_t B_bs, const void *Cm, int64_t C_bs,
                         const float *A_log, const float *D, const float *dt_bias, float *h,
                         void *out, int64_t out_bs, int B, int ED, int N, uint32_t flags, int dtype, void *stream) {
    using namespace gfe;
    if (!u || !delta || !Bm || !Cm || !A_log || !D || !h || !out) { set_error("ssm_step: NULL pointer"); return GFE_ERR_ARG; }
    if (B <= 0 || ED <= 0 || B > 65535) { set_error("ssm_step: bad shape"); return GFE_ERR_ARG; }
    if (!fused_d_state(N)) { set_error("ssm_step: d_state=%d unsupported (compiled for 16, 32 and 64)", N); return GFE_ERR_UNSUPPORTED; }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    switch (dtype) {
        case GFE_F32: return ssm_step_launch_n<float>(N, u, u_bs, delta, delta_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, out_bs, B, ED, flags, st);
        case GFE_BF16: return ssm_step_launch_n<__nv_bfloat16>(N, u, u_bs, delta, delta_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, out_bs, B, ED, flags, st);
        case GFE_F16: return ssm_step_launch_n<__half>(N, u, u_bs, delta, delta_bs, z, z_bs, Bm, B_bs, Cm, C_bs, A_log, D, dt_bias, h, out, out_bs, B, ED, flags, st);
        default: set_error("ssm_step: bad dtype %d", dtype); return GFE_ERR_DTYPE;
    }
}

}  // extern "C"
