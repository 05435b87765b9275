// pool.cu -- final residual add fused with the mean over L (SURVEY 8f rank 4).
//
// The classifier head pools the Mamba stack's output over the sequence (mamba_transformer.py:122-123:
//     x = self.transformer(x); x = torch.mean(x, dim=1, keepdims=True)),
// and the stack's last operation is the residual add of its last layer (mamba.py:103).  Unfused that is one pass writing the
// (B, L, D) sum and one pass reading it back; here the two (B, L, D) operands are read once and only (B, D) is written:
//   fwd   out[b, d] = (1 / L) * sum_t (a[b, t, d] + r[b, t, d])          reads 2 B L D, writes B D
//   bwd   da[b, t, d] = dr[b, t, d] = dout[b, d] / L                      writes B L D per operand that needs it
// Deterministic: per-(row tile) partial sums in fp32, added in tile order by a second tiny kernel.
// The operands may differ in element type the way addnorm.cu's do: under autocast the last branch (out_proj's output) is
// 16-bit and the residual stream fp32.  Then out and dout are fp32, as torch promotes a + r, every element is read in its own
// type (no cast pass over (B, L, D)), and backward writes each operand's gradient in its own type in the same pass.
#include "common.cuh"

namespace gfe {

constexpr int kPoolTile = 64;   // rows per partial sum
constexpr int kPoolNT = 128;

// element type of out / dout: the operands' when they agree, else fp32 (the other one is 16-bit)
template <typename TA, typename TR> struct PoolOut { using type = float; };
template <typename T> struct PoolOut<T, T> { using type = T; };

template <typename TA, typename TR>
__global__ void __launch_bounds__(kPoolNT) add_mean_pool_partial_kernel(const TA *__restrict__ a, const TR *__restrict__ r,
                                                                         float *__restrict__ part, int L, int D, int ntile) {
    const int d = blockIdx.x * kPoolNT + threadIdx.x;
    const int tile = blockIdx.y, b = blockIdx.z;
    if (d >= D) return;
    const int t0 = tile * kPoolTile, t1 = min(L, t0 + kPoolTile);
    const TA *pa = a + ((size_t)b * L + t0) * D + d;
    const TR *pr = r ? r + ((size_t)b * L + t0) * D + d : nullptr;
    float acc0 = 0.f, acc1 = 0.f;
    int t = t0;
    for (; t + 1 < t1; t += 2) {   // two independent chains: the loads of both rows are in flight together
        acc0 += to_f(ld_stream(pa)) + (pr ? to_f(ld_stream(pr)) : 0.f);
        acc1 += to_f(ld_stream(pa + D)) + (pr ? to_f(ld_stream(pr + D)) : 0.f);
        pa += 2 * (size_t)D;
        if (pr) pr += 2 * (size_t)D;
    }
    if (t < t1) acc0 += to_f(ld_stream(pa)) + (pr ? to_f(ld_stream(pr)) : 0.f);
    part[((size_t)b * ntile + tile) * D + d] = acc0 + acc1;
}

template <typename T>
__global__ void __launch_bounds__(kPoolNT) add_mean_pool_final_kernel(const float *__restrict__ part, T *__restrict__ out, int L, int D, int ntile) {
    const int d = blockIdx.x * kPoolNT + threadIdx.x, b = blockIdx.y;
    if (d >= D) return;
    float acc = 0.f;
    for (int i = 0; i < ntile; ++i) acc += part[((size_t)b * ntile + i) * D + d];
    out[(size_t)b * D + d] = from_f<T>(acc / (float)L);
}

// dout / L rounded once per operand type; dr == nullptr: only a's gradient (no r, or r needs none, or the caller shares da)
template <typename TA, typename TR>
__global__ void __launch_bounds__(kPoolNT) mean_pool_bwd_kernel(const typename PoolOut<TA, TR>::type *__restrict__ dout,
                                                                TA *__restrict__ da, TR *__restrict__ dr, int L, int D) {
    const int d = blockIdx.x * kPoolNT + threadIdx.x;
    const int tile = blockIdx.y, b = blockIdx.z;
    if (d >= D) return;
    const float g = to_f(dout[(size_t)b * D + d]) / (float)L;
    const TA va = from_f<TA>(g);
    const TR vr = from_f<TR>(g);
    const int t0 = tile * kPoolTile, t1 = min(L, t0 + kPoolTile);
    const size_t o = ((size_t)b * L + t0) * D + d;
    TA *p = da + o;
    for (int t = t0; t < t1; ++t, p += D) st_stream(p, va);
    if (dr != nullptr) {
        TR *q = dr + o;
        for (int t = t0; t < t1; ++t, q += D) st_stream(q, vr);
    }
}

template <typename T> struct PoolTag { using type = T; };

// (a, r) element types the kernels are compiled for: equal, or fp32 next to a 16-bit type in either order
template <typename F>
static int pool_dispatch(int a_dtype, int r_dtype, const char *what, F &&f) {
    if (a_dtype == r_dtype) {
        switch (a_dtype) {
            case GFE_F32: return f(PoolTag<float>{}, PoolTag<float>{});
            case GFE_BF16: return f(PoolTag<__nv_bfloat16>{}, PoolTag<__nv_bfloat16>{});
            case GFE_F16: return f(PoolTag<__half>{}, PoolTag<__half>{});
            default: break;
        }
    } else if (a_dtype == GFE_F32) {
        if (r_dtype == GFE_BF16) return f(PoolTag<float>{}, PoolTag<__nv_bfloat16>{});
        if (r_dtype == GFE_F16) return f(PoolTag<float>{}, PoolTag<__half>{});
    } else if (r_dtype == GFE_F32) {
        if (a_dtype == GFE_BF16) return f(PoolTag<__nv_bfloat16>{}, PoolTag<float>{});
        if (a_dtype == GFE_F16) return f(PoolTag<__half>{}, PoolTag<float>{});
    }
    set_error("%s: unsupported dtype pair (a %d, r %d)", what, a_dtype, r_dtype);
    return GFE_ERR_DTYPE;
}

}  // namespace gfe

extern "C" {

GFE_API size_t gfe_add_mean_pool_workspace_bytes(int B, int L, int D) {
    if (B <= 0 || L <= 0 || D <= 0) return 0;
    return (size_t)B * ((L + gfe::kPoolTile - 1) / gfe::kPoolTile) * D * sizeof(float);
}

GFE_API int gfe_add_mean_pool_fwd_mixed(const void *a, const void *r, void *out, int B, int L, int D, int a_dtype, int r_dtype,
                                        void *ws, size_t ws_bytes, void *stream) {
    using namespace gfe;
    if (!a || !out || B <= 0 || L <= 0 || D <= 0 || B > 65535) { set_error("add_mean_pool_fwd: bad argument"); return GFE_ERR_ARG; }
    if (!ws || ws_bytes < gfe_add_mean_pool_workspace_bytes(B, L, D)) { set_error("add_mean_pool_fwd: workspace too small"); return GFE_ERR_WORKSPACE; }
    if (!r) r_dtype = a_dtype;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    float *part = reinterpret_cast<float *>(ws);
    const int ntile = (L + kPoolTile - 1) / kPoolTile;
    return pool_dispatch(a_dtype, r_dtype, "add_mean_pool_fwd", [&](auto ta, auto tr) {
        using TA = typename decltype(ta)::type;
        using TR = typename decltype(tr)::type;
        using TO = typename PoolOut<TA, TR>::type;
        { ScopedKernelTimer tm(K_POOL_FWD, st);
          add_mean_pool_partial_kernel<TA, TR><<<dim3((D + kPoolNT - 1) / kPoolNT, ntile, B), kPoolNT, 0, st>>>(
              reinterpret_cast<const TA *>(a), reinterpret_cast<const TR *>(r), part, L, D, ntile);
          add_mean_pool_final_kernel<TO><<<dim3((D + kPoolNT - 1) / kPoolNT, B), kPoolNT, 0, st>>>(part, reinterpret_cast<TO *>(out), L, D, ntile); }
        return check_launch("add_mean_pool_fwd");
    });
}

GFE_API int gfe_add_mean_pool_fwd(const void *a, const void *r, void *out, int B, int L, int D, int dtype, void *ws, size_t ws_bytes,
                                  void *stream) {
    return gfe_add_mean_pool_fwd_mixed(a, r, out, B, L, D, dtype, dtype, ws, ws_bytes, stream);
}

GFE_API int gfe_mean_pool_bwd_mixed(const void *dout, void *da, void *dr, int B, int L, int D, int a_dtype, int r_dtype, void *stream) {
    using namespace gfe;
    if (!dout || !da || B <= 0 || L <= 0 || D <= 0 || B > 65535) { set_error("mean_pool_bwd: bad argument"); return GFE_ERR_ARG; }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int ntile = (L + kPoolTile - 1) / kPoolTile;
    return pool_dispatch(a_dtype, r_dtype, "mean_pool_bwd", [&](auto ta, auto tr) {
        using TA = typename decltype(ta)::type;
        using TR = typename decltype(tr)::type;
        using TO = typename PoolOut<TA, TR>::type;
        { ScopedKernelTimer tm(K_POOL_BWD, st);
          mean_pool_bwd_kernel<TA, TR><<<dim3((D + kPoolNT - 1) / kPoolNT, ntile, B), kPoolNT, 0, st>>>(
              reinterpret_cast<const TO *>(dout), reinterpret_cast<TA *>(da), reinterpret_cast<TR *>(dr), L, D); }
        return check_launch("mean_pool_bwd");
    });
}

GFE_API int gfe_mean_pool_bwd(const void *dout, void *da, int B, int L, int D, int dtype, void *stream) {
    return gfe_mean_pool_bwd_mixed(dout, da, nullptr, B, L, D, dtype, dtype, stream);
}

}  // extern "C"
