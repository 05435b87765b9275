/*
 * gfe_mamba_b200.h -- C ABI of the B200 (sm_100a) selective-scan library.
 *
 * This is the drop-in boundary for GFE-Mamba's Mamba hot path.  The reference
 * (Tinysqua/GFE-Mamba) is pure Python and has no FFI of its own; the entry points
 * below are what a binding for that path binds, one per reference function:
 *
 *   gfe_pscan_fwd / gfe_pscan_bwd        cross_atten/pscan.py:152-186 / :189-224  (PScan.forward / .backward)
 *   gfe_selscan_fwd / gfe_selscan_bwd    cross_atten/mamba.py:227-286 (ssm + selective_scan, with the
 *                                        softplus+bias of :255-256 and the silu(z) gate of :220-222 fused,
 *                                        i.e. the contract of the selective_scan_fn call at :251)
 *   gfe_conv1d_silu_fwd / _bwd           cross_atten/mamba.py:128-131,208-212 (causal depthwise conv + SiLU)
 *   gfe_conv1d_step / gfe_ssm_step       cross_atten/mamba.py:357-358,370 and :375-405 (decode step)
 *   gfe_conv1d_silu_fwd_state /          the same forwards continuing a decode cache (prefill: many tokens
 *   gfe_selscan_fwd_state                at once from a (h, conv window) cache, the multi-token decode step)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller; the library never
 *     allocates, frees or retains memory, and never synchronises the stream;
 *   - `stream` is a cudaStream_t passed as void*;
 *   - activations are channel-last (B, L, ED); strides are in ELEMENTS, the channel
 *     (innermost) stride is always 1, so the halves of in_proj's output and the
 *     slices of x_proj's output are consumed in place;
 *   - parameters A_log, D, dt_bias, conv weight/bias and all parameter gradients
 *     are fp32; `dtype` names the activation type;
 *   - return value: GFE_OK (0) or a negative gfe_status; gfe_last_error_string()
 *     returns a thread-local description of the last failure;
 *   - stateless and re-entrant: safe from any host thread (e.g. autograd's);
 *   - the selective scan (gfe_selscan_*) and the decode step (gfe_ssm_step) are compiled
 *     for d_state N in {16, 32, 64}; the size queries return 0 and the entry points
 *     GFE_ERR_UNSUPPORTED for any other N.
 */
#ifndef GFE_MAMBA_B200_H
#define GFE_MAMBA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GFE_API __attribute__((visibility("default")))
#else
#define GFE_API
#endif

#define GFE_VERSION 100 /* 0.1.0 */

enum gfe_dtype { GFE_F32 = 0, GFE_BF16 = 1, GFE_F16 = 2 };

enum gfe_status {
    GFE_OK = 0,
    GFE_ERR_ARG = -1,         /* null pointer / non-positive size / bad flag            */
    GFE_ERR_DTYPE = -2,       /* dtype not one of gfe_dtype                              */
    GFE_ERR_UNSUPPORTED = -3, /* shape outside the compiled envelope (e.g. d_state outside {16, 32, 64}) */
    GFE_ERR_WORKSPACE = -4,   /* workspace / checkpoint buffer missing or too small      */
    GFE_ERR_CUDA = -5         /* launch failed (cudaPeekAtLastError)                      */
};

/* flags of gfe_selscan_args.flags */
#define GFE_FLAG_DELTA_SOFTPLUS 1u /* delta = softplus(delta + dt_bias) (mamba.py:255-256); else delta + dt_bias */

GFE_API int gfe_version(void);
GFE_API const char *gfe_last_error_string(void);

/* ------------------------------------------------------------------ pscan --
 * H[t] = A[t] * H[t-1] + X[t], H[-1] = 0, independently per (b, d, n).
 * A, X, H, dH, dA, dX: contiguous (B, L, D, N) fp32.  Any L >= 1 (the reference
 * pads to the next power of two; results on [0, L) are identical).
 * bwd: dX[t] = g[t] = dH[t] + A[t+1] g[t+1];  dA[t] = H[t-1] g[t], dA[0] = 0.
 */
GFE_API size_t gfe_pscan_workspace_bytes(int B, int L, int D, int N);
GFE_API int gfe_pscan_fwd(const float *A, const float *X, float *H, int B, int L, int D, int N,
                          void *ws, size_t ws_bytes, void *stream);
GFE_API int gfe_pscan_bwd(const float *A, const float *H, const float *dH, float *dA, float *dX,
                          int B, int L, int D, int N, void *ws, size_t ws_bytes, void *stream);

/* --------------------------------------------------------- selective scan --
 * out[b,t,c] = (sum_n C[b,t,n] h[b,t,c,n] + D[c] u[b,t,c]) * silu(z[b,t,c])
 * h[t] = exp(delta A) h[t-1] + delta B[t] u[t],  A = -exp(A_log),
 * delta = softplus(delta_in + dt_bias).
 */
typedef struct gfe_selscan_args {
    int32_t batch, seqlen, d_inner, d_state;
    int32_t dtype;  /* gfe_dtype of u, delta, z, Bm, Cm, out and of their gradients */
    uint32_t flags; /* GFE_FLAG_* */

    const void *u;     int64_t u_bs, u_rs;         /* (B, L, ED): batch stride, row stride */
    const void *delta; int64_t delta_bs, delta_rs; /* (B, L, ED) pre-softplus, pre-bias    */
    const void *z;     int64_t z_bs, z_rs;         /* (B, L, ED) or NULL (no gate)         */
    const void *Bm;    int64_t B_bs, B_rs;         /* (B, L, N)                            */
    const void *Cm;    int64_t C_bs, C_rs;         /* (B, L, N)                            */
    const float *A_log;                            /* (ED, N) contiguous                   */
    const float *D;                                /* (ED)                                 */
    const float *dt_bias;                          /* (ED) or NULL                         */

    void *out;         int64_t out_bs, out_rs;     /* (B, L, ED)   [fwd only]              */
    float *last_state;                             /* (B, ED, N) or NULL [fwd only]        */

    /* chunk checkpoints: written by fwd when non-NULL, required by bwd.
     * gfe_selscan_ckpt_bytes() bytes, opaque layout. */
    void *ckpt;        size_t ckpt_bytes;
    void *ws;          size_t ws_bytes;            /* scratch, gfe_selscan_{fwd,bwd}_workspace_bytes() */

    /* ---- backward only ---- */
    const void *dout;  int64_t dout_bs, dout_rs;   /* (B, L, ED) */
    void *du;          int64_t du_bs, du_rs;
    void *ddelta;      int64_t ddelta_bs, ddelta_rs; /* gradient w.r.t. delta_in (pre-softplus) */
    void *dz;          int64_t dz_bs, dz_rs;       /* NULL iff z is NULL */
    void *dBm;         int64_t dB_bs, dB_rs;       /* (B, L, N) */
    void *dCm;         int64_t dC_bs, dC_rs;
    float *dA_log;                                 /* (ED, N)  overwritten */
    float *dD;                                     /* (ED)     overwritten */
    float *ddt_bias;                               /* (ED) or NULL, overwritten */
} gfe_selscan_args;

GFE_API size_t gfe_selscan_ckpt_bytes(int B, int L, int ED, int N);            /* upper bound over the dtypes (fp32) */
GFE_API size_t gfe_selscan_ckpt_bytes_dt(int B, int L, int ED, int N, int dtype); /* exact, for one gfe_dtype          */
GFE_API size_t gfe_selscan_fwd_workspace_bytes(int B, int L, int ED, int N);
GFE_API size_t gfe_selscan_bwd_workspace_bytes(int B, int L, int ED, int N);
GFE_API int gfe_selscan_fwd(const gfe_selscan_args *args, void *stream);
GFE_API int gfe_selscan_bwd(const gfe_selscan_args *args, void *stream);
/* Forward from a carried state (inference, prefill from a decode cache): gfe_selscan_fwd with h[-1] = h0 instead of 0.
 * h0: (B, ED, N) fp32, contiguous, 16-byte aligned, or NULL (= zeros) -- the layout of last_state and of gfe_ssm_step's h.
 * args->ckpt must be NULL (no backward from here).  args->last_state may be NULL; it must not overlap h0.
 * Same workspace query (gfe_selscan_fwd_workspace_bytes). */
GFE_API int gfe_selscan_fwd_state(const gfe_selscan_args *args, const float *h0, void *stream);

/* ------------------------------------------------ causal depthwise conv1d --
 * u[b,t,c] = silu(bias[c] + sum_k w[c,k] xin[b, t-(K-1)+k, c]),  xin = 0 for t < 0.
 * w: (ED, K) fp32 (= conv1d.weight viewed (ED,1,K)), bias: (ED) fp32 or NULL.  K in 2..4 (GFE_ERR_UNSUPPORTED otherwise).
 */
GFE_API int gfe_conv1d_silu_fwd(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                void *u, int64_t u_bs, int64_t u_rs, int B, int L, int ED, int K, int dtype,
                                void *stream);
/* Causal conv + SiLU continuing a decode cache: xin[t < 0] is read from inputs (B, ED, K-1) in the activation dtype
 * (NULL = zeros); new_inputs (B, ED, K-1), may be NULL, receives the last K-1 rows of cat(inputs, xin) along time -- the
 * cache gfe_conv1d_step would hold after the same tokens.  inputs and new_inputs must not overlap.  K in 2..4. */
GFE_API int gfe_conv1d_silu_fwd_state(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                      const void *inputs, void *new_inputs, void *u, int64_t u_bs, int64_t u_rs,
                                      int B, int L, int ED, int K, int dtype, void *stream);
GFE_API size_t gfe_conv1d_bwd_workspace_bytes(int B, int L, int ED, int K);
GFE_API int gfe_conv1d_silu_bwd(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                const void *du, int64_t du_bs, int64_t du_rs,
                                void *dxin, int64_t dx_bs, int64_t dx_rs, float *dw, float *dbias,
                                int B, int L, int ED, int K, int dtype, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------ decode step --
 * gfe_conv1d_step: window = cat(inputs, xin[:, None]) (mamba.py:357); u = silu(conv(window)[K-1]);
 *                  inputs <- window[:, :, 1:] in place (mamba.py:370).  inputs: (B, ED, K-1) activation dtype.
 * gfe_ssm_step:    h <- exp(delta A) h + delta B u;  out = (h.C + D u) * silu(z)   (mamba.py:391-403, :364-367)
 *                  h: (B, ED, N) fp32, updated in place; delta = softplus(delta_in + dt_bias).
 */
GFE_API int gfe_conv1d_step(const void *xin, int64_t x_bs, void *inputs, const float *w, const float *bias,
                            void *u, int64_t u_bs, int B, int ED, int K, int dtype, void *stream);
GFE_API int gfe_ssm_step(const void *u, int64_t u_bs, const void *delta, int64_t delta_bs,
                         const void *z, int64_t z_bs, const void *Bm, int64_t B_bs, const void *Cm, int64_t C_bs,
                         const float *A_log, const float *D, const float *dt_bias, float *h,
                         void *out, int64_t out_bs, int B, int ED, int N, uint32_t flags, int dtype, void *stream);

/* ------------------------------------------------- residual add + RMSNorm --
 * SURVEY 8f rank 1: the residual add of ResidualBlock.forward (mamba.py:103) fused with the next layer's RMSNorm
 * (mamba.py:408-418).  Row-contiguous (rows, D) tensors in the activation dtype, 16-byte aligned; w: (D) fp32.
 *   fwd: resid = x + a (a, resid may be NULL: plain RMSNorm of x);  y = (resid * rstd) * w,
 *        rstd[r] = rsqrt(mean(resid[r]^2) + eps)  (fp32, saved for backward; may be NULL for inference)
 *   bwd: dx = dres + d/dresid of the norm (dres may be NULL);  dw[j] = sum_r dy[r,j] * resid[r,j] * rstd[r]
 * D must be a multiple of 16 / sizeof(element); rows of up to 256 such vectors are held in registers, wider rows take two
 * passes (the second from cache).
 */
GFE_API int gfe_add_rmsnorm_fwd(const void *x, const void *a, const float *w, void *resid, void *y, float *rstd,
                                int64_t rows, int D, float eps, int dtype, void *stream);
GFE_API size_t gfe_add_rmsnorm_bwd_workspace_bytes(int64_t rows, int D);
GFE_API int gfe_add_rmsnorm_bwd(const void *resid, const float *w, const float *rstd, const void *dy, const void *dres,
                                void *dx, float *dw, int64_t rows, int D, int dtype, void *ws, size_t ws_bytes,
                                void *stream);
/* The same with two element types: the residual stream (x, resid, dres, dx: res_dtype) and the branch side (a, y, dy, da:
 * io_dtype).  res_dtype == io_dtype is the call above; res_dtype = GFE_F32 with a 16-bit io_dtype is the Mamba stack under
 * autocast (fp32 residual stream, mixers in bf16 / fp16, mamba.py:103 + :408-418 as autocast runs them): the cast kernels
 * around the norm disappear.  D: multiple of 16 / sizeof(res element).  da (optional): the gradient of `a` in io_dtype
 * (the values of dx, rounded). */
GFE_API int gfe_add_rmsnorm_fwd_mixed(const void *x, const void *a, const float *w, void *resid, void *y, float *rstd,
                                      int64_t rows, int D, float eps, int res_dtype, int io_dtype, void *stream);
GFE_API int gfe_add_rmsnorm_bwd_mixed(const void *resid, const float *w, const float *rstd, const void *dy, const void *dres,
                                      void *dx, void *da, float *dw, int64_t rows, int D, int res_dtype, int io_dtype,
                                      void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------ final residual add + mean over L (head) --
 * out[b, d] = mean_t (a[b, t, d] + r[b, t, d]): the last residual add of the Mamba stack (mamba.py:103) fused with the
 * classifier head's pooling (mamba_transformer.py:123, torch.mean(x, dim=1)).  a, r: contiguous (B, L, D), r may be NULL;
 * out: (B, D), same dtype.  bwd: da[b, t, d] = dout[b, d] / L (the gradient of both operands).
 */
GFE_API size_t gfe_add_mean_pool_workspace_bytes(int B, int L, int D);
GFE_API int gfe_add_mean_pool_fwd(const void *a, const void *r, void *out, int B, int L, int D, int dtype, void *ws, size_t ws_bytes,
                                  void *stream);
GFE_API int gfe_mean_pool_bwd(const void *dout, void *da, int B, int L, int D, int dtype, void *stream);
/* The same with an element type per operand: a in a_dtype, r in r_dtype (ignored when r is NULL).  The pairs are equal types,
 * or GFE_F32 with GFE_BF16 / GFE_F16 in either order -- the stack under autocast, whose last branch is 16-bit next to the
 * fp32 residual stream; any other pair returns GFE_ERR_DTYPE.  out and dout are in the promoted type (torch's a + r):
 * GFE_F32 when the two differ.  bwd writes da in a_dtype and, when dr is not NULL, dr in r_dtype from the same pass. */
GFE_API int gfe_add_mean_pool_fwd_mixed(const void *a, const void *r, void *out, int B, int L, int D, int a_dtype, int r_dtype,
                                        void *ws, size_t ws_bytes, void *stream);
GFE_API int gfe_mean_pool_bwd_mixed(const void *dout, void *da, void *dr, int B, int L, int D, int a_dtype, int r_dtype,
                                    void *stream);

/* ------------------------------------------- multi-tensor clip + Adam step --
 * One optimiser step for a whole parameter list in three launches; replaces the per-parameter loop
 *     for p in params: torch.nn.utils.clip_grad_norm_(p, max_norm)      (classify_mamba.py:106-107)
 *     optimizer.step(); optimizer.zero_grad()                            (classify_mamba.py:108-109, torch.optim.Adam)
 * All tables live in DEVICE memory and are built once by the caller:
 *   p_ptr, g_ptr, m_ptr, v_ptr [ntensors]  device addresses (as int64) of the fp32 parameter, gradient, exp_avg, exp_avg_sq
 *   numel [ntensors];  the tensors are cut into chunks of gfe_clip_adam_chunk_elems() elements:
 *   chunk_tensor [nchunks], chunk_start [nchunks] (element offset in the tensor), tensor_chunk0 [ntensors + 1]
 *   partial [nchunks], coef [ntensors]  scratch;  step [1]  int32 step counter, incremented by the call
 * clip: coef = min(1, max_norm / (norm + 1e-6)) per tensor (global_norm = 0, the reference loop) or over the whole
 * list (global_norm = 1); max_norm <= 0 disables clipping.  zero_grad != 0 leaves the gradients zeroed, else clipped.
 */
GFE_API int gfe_clip_adam_chunk_elems(void);
GFE_API int gfe_clip_adam_step(const int64_t *p_ptr, const int64_t *g_ptr, const int64_t *m_ptr, const int64_t *v_ptr,
                               const int64_t *numel, const int32_t *chunk_tensor, const int64_t *chunk_start,
                               const int32_t *tensor_chunk0, float *partial, float *coef, int32_t *step, int ntensors,
                               int nchunks, float lr, float beta1, float beta2, float eps, float max_norm, int global_norm,
                               int zero_grad, void *stream);

/* -------------------------------------------------------- instrumentation --
 * Optional per-kernel device timing: when enabled, every kernel the library launches is bracketed by a
 * cudaEvent pair on the launching stream.  gfe_timing_collect() synchronises those events, adds the elapsed
 * milliseconds and launch counts per kernel id into the caller's arrays (length n >= gfe_timing_kernel_count())
 * and clears the records.  Off by default (zero overhead); used by bench.py for the roofline line.
 */
GFE_API int gfe_timing_enable(int on);
GFE_API int gfe_timing_kernel_count(void);
GFE_API const char *gfe_timing_kernel_name(int id);
GFE_API int gfe_timing_collect(double *total_ms, int64_t *launches, int n);

#ifdef __cplusplus
}
#endif
#endif /* GFE_MAMBA_B200_H */
