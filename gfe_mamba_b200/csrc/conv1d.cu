// conv1d.cu -- causal depthwise conv1d + bias + SiLU, channel-last, forward and backward.
//
// Replaces nn.Conv1d(groups=ED, kernel_size=K, padding=K-1)(x.transpose(1,2))[:, :, :L].transpose(1,2)
// followed by F.silu (cross_atten/mamba.py:128-131, 208-212): no transposes, the strided x half of
// in_proj's output is read in place, the K-wide window slides through registers so every input element
// is loaded once per time tile (+ K-1 halo).  A lane owns 4 (16-bit) / 2 (fp32) adjacent channels and moves them with
// one 8-byte access, so a warp request covers 256 contiguous bytes of a row.
//   forward : read xin, write u                      (2 * ED * s bytes / token)
//   backward: read xin, du, write dxin               (3 * ED * s bytes / token), dw/dbias via
//             per-(b, tile) partial sums + a deterministic finalize kernel.
#include <type_traits>

#include "common.cuh"

namespace gfe {

// time steps per thread (one partial dw|dbias row per tile); 64 and 256 measured, no gain (profiles/r02_chain_variants.txt)
constexpr int kConvTile = 128;

struct ConvParams {
    const void *xin, *du;
    void *u, *dxin;
    const float *w, *bias;
    float *dw, *dbias, *part;   // part: [B*ntiles][K+1][ED]
    int64_t x_bs, x_rs, u_bs, u_rs, du_bs, du_rs, dx_bs, dx_rs;
    int B, L, ED, ntiles;
    // forward continuing a decode cache (gfe_conv1d_silu_fwd_state): rows t < 0 are read from cin (B, ED, K-1) instead of
    // being zeros, and the last tile writes the last K-1 rows of cat(cin, xin) to cout (B, ED, K-1); either may be NULL
    const void *cin;
    void *cout;
};

// V adjacent channels per lane, moved as ONE load / store of V * sizeof(T) bytes (8 bytes when the layout allows it: 4
// channels for 16-bit activations, 2 for fp32), so a warp request covers 256 contiguous bytes instead of 64 / 128.
template <int BYTES> struct RawBytes;
template <> struct RawBytes<2> { using type = unsigned short; };
template <> struct RawBytes<4> { using type = unsigned int; };
template <> struct RawBytes<8> { using type = uint2; };
template <typename T, int V> struct ChanVec {
    using Raw = typename RawBytes<V * (int)sizeof(T)>::type;
    Raw raw;
    __device__ __forceinline__ float get(int i) const { return to_f(reinterpret_cast<const T *>(&raw)[i]); }
    __device__ __forceinline__ void set(int i, float v) { reinterpret_cast<T *>(&raw)[i] = from_f<T>(v); }
    __device__ __forceinline__ static ChanVec load(const T *p) { ChanVec r; r.raw = __ldcs(reinterpret_cast<const Raw *>(p)); return r; }
    __device__ __forceinline__ void store(T *p) const { __stcs(reinterpret_cast<Raw *>(p), raw); }
};

template <typename T, int K, int V>
__global__ void __launch_bounds__(128) conv1d_silu_fwd_kernel(ConvParams p) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * V;
    if (c >= p.ED) return;
    const int tile = blockIdx.y, b = blockIdx.z;
    const int t0 = tile * kConvTile, t1 = min(p.L, t0 + kConvTile);
    const T *x = reinterpret_cast<const T *>(p.xin) + (int64_t)b * p.x_bs + c;
    T *u = reinterpret_cast<T *>(p.u) + (int64_t)b * p.u_bs + c;
    float w[V][K], bias[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) w[i][k] = __ldg(p.w + (size_t)(c + i) * K + k);
        bias[i] = p.bias ? __ldg(p.bias + c + i) : 0.f;
    }
    float win[V][K];   // win[.][k] = xin[t - (K-1) + k]
    const T *cin = reinterpret_cast<const T *>(p.cin) + ((size_t)b * p.ED + c) * (K - 1);   // row t < 0: cin[t + K - 1]
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
        const int t = t0 - (K - 1) + k;
        ChanVec<T, V> xv{};
        if (t >= 0) xv = ChanVec<T, V>::load(x + (int64_t)t * p.x_rs);
#pragma unroll
        for (int i = 0; i < V; ++i) win[i][k + 1] = t >= 0 ? xv.get(i) : (p.cin != nullptr ? to_f(cin[i * (K - 1) + k]) : 0.f);
    }
    constexpr int U = 8;
    // rows of the next group, in flight while the current group is computed (measured on both directions: fp32 backward 14 %
    // faster, 16-bit 3-4 % slower; profiles/r02_chain_variants.txt)
    ChanVec<T, V> xn[U];
#pragma unroll
    for (int j = 0; j < U; ++j) xn[j] = ChanVec<T, V>::load(x + (int64_t)min(t0 + j, t1 - 1) * p.x_rs);
    for (int tb = t0; tb < t1; tb += U) {
        ChanVec<T, V> xr[U];
#pragma unroll
        for (int j = 0; j < U; ++j) xr[j] = xn[j];
        if (tb + U < t1) {
#pragma unroll
            for (int j = 0; j < U; ++j) xn[j] = ChanVec<T, V>::load(x + (int64_t)min(tb + U + j, t1 - 1) * p.x_rs);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (tb + j < t1) {
                ChanVec<T, V> o;
#pragma unroll
                for (int i = 0; i < V; ++i) {
#pragma unroll
                    for (int k = 0; k < K - 1; ++k) win[i][k] = win[i][k + 1];
                    win[i][K - 1] = xr[j].get(i);
                    float v = bias[i];
#pragma unroll
                    for (int k = 0; k < K; ++k) v = fmaf(w[i][k], win[i][k], v);
                    o.set(i, v * sigmoid_fast(v));
                }
                o.store(u + (int64_t)(tb + j) * p.u_rs);
            }
        }
    }
    if (p.cout != nullptr && blockIdx.y == gridDim.y - 1) {   // last tile: the window holds the last K-1 rows of cat(cin, xin)
        T *cout = reinterpret_cast<T *>(p.cout) + ((size_t)blockIdx.z * p.ED + (blockIdx.x * blockDim.x + threadIdx.x) * V) * (K - 1);
#pragma unroll
        for (int i = 0; i < V; ++i) {
#pragma unroll
            for (int k = 0; k < K - 1; ++k) cout[i * (K - 1) + k] = from_f<T>(win[i][k + 1]);
        }
    }
}

template <typename T, int K, int V>
__global__ void __launch_bounds__(128) conv1d_silu_bwd_kernel(ConvParams p) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * V;
    if (c >= p.ED) return;
    const int tile = blockIdx.y, b = blockIdx.z;
    const int t0 = tile * kConvTile, t1 = min(p.L, t0 + kConvTile);
    const T *x = reinterpret_cast<const T *>(p.xin) + (int64_t)b * p.x_bs + c;
    const T *du = reinterpret_cast<const T *>(p.du) + (int64_t)b * p.du_bs + c;
    T *dx = reinterpret_cast<T *>(p.dxin) + (int64_t)b * p.dx_bs + c;
    float w[V][K], bias[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) w[i][k] = __ldg(p.w + (size_t)(c + i) * K + k);
        bias[i] = p.bias ? __ldg(p.bias + c + i) : 0.f;
    }
    float win[V][K], dvw[V][K], dw[V][K], db[V];   // dvw[.][k] = dv[t - (K-1) + k]
#pragma unroll
    for (int i = 0; i < V; ++i) {
        db[i] = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) { dvw[i][k] = 0.f; dw[i][k] = 0.f; }
    }
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
        const int t = t0 - (K - 1) + k;
        ChanVec<T, V> xv{};
        if (t >= 0) xv = ChanVec<T, V>::load(x + (int64_t)t * p.x_rs);
#pragma unroll
        for (int i = 0; i < V; ++i) win[i][k + 1] = t >= 0 ? xv.get(i) : 0.f;
    }
    // dv is needed K-1 steps past the tile to finish dxin of the tile's last steps
    const int tend = t1 + (K - 1);
    constexpr int U = 8;
    ChanVec<T, V> xn[U], gn[U];   // rows of the next group, in flight while the current group is computed
#pragma unroll
    for (int j = 0; j < U; ++j) {
        const int t = min(t0 + j, p.L - 1);
        xn[j] = ChanVec<T, V>::load(x + (int64_t)t * p.x_rs);
        gn[j] = ChanVec<T, V>::load(du + (int64_t)t * p.du_rs);
    }
    for (int tb = t0; tb < tend; tb += U) {
        ChanVec<T, V> xr[U], gr[U];
#pragma unroll
        for (int j = 0; j < U; ++j) { xr[j] = xn[j]; gr[j] = gn[j]; }
        if (tb + U < tend) {
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const int t = min(tb + U + j, p.L - 1);
                xn[j] = ChanVec<T, V>::load(x + (int64_t)t * p.x_rs);
                gn[j] = ChanVec<T, V>::load(du + (int64_t)t * p.du_rs);
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int t = tb + j;
            if (t < tend) {
                const int s_out = t - (K - 1);   // dxin[s] = sum_k w[k] dv[s + K-1 - k]
                ChanVec<T, V> o;
#pragma unroll
                for (int i = 0; i < V; ++i) {
#pragma unroll
                    for (int k = 0; k < K - 1; ++k) { win[i][k] = win[i][k + 1]; dvw[i][k] = dvw[i][k + 1]; }
                    float dv = 0.f;
                    if (t < p.L) {
                        win[i][K - 1] = xr[j].get(i);
                        float v = bias[i];
#pragma unroll
                        for (int k = 0; k < K; ++k) v = fmaf(w[i][k], win[i][k], v);
                        const float sg = sigmoid_fast(v);
                        dv = gr[j].get(i) * sg * fmaf(v, 1.0f - sg, 1.0f);
                        if (t < t1) {   // parameter gradients: own tile only
                            db[i] += dv;
#pragma unroll
                            for (int k = 0; k < K; ++k) dw[i][k] = fmaf(dv, win[i][k], dw[i][k]);
                        }
                    }
                    dvw[i][K - 1] = dv;
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < K; ++k) acc = fmaf(w[i][k], dvw[i][K - 1 - k], acc);
                    o.set(i, acc);
                }
                if (s_out >= t0 && s_out < t1) o.store(dx + (int64_t)s_out * p.dx_rs);
            }
        }
    }
    float *part = p.part + ((size_t)(b * p.ntiles + tile) * (K + 1)) * p.ED + c;
#pragma unroll
    for (int i = 0; i < V; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) part[(size_t)k * p.ED + i] = dw[i][k];
        part[(size_t)K * p.ED + i] = db[i];
    }
}

// ---- packed variants: NP channel PAIRS per lane (2 for 16-bit activations, 1 for fp32), every FP32 op on a float2 ----------
// The scalar kernels above spend ~25 instructions per element in 16-bit (unpack, per-channel FFMA chains, 64-bit address
// arithmetic per row): issue-bound at a third of the HBM peak.  Here the window, the weights and every product are float2 over
// a channel pair, rows are addressed through running pointers, and full groups of 8 rows run without row checks.
template <typename T, int NP> struct PairVec;
template <> struct PairVec<float, 1> {
    using Raw = float2;
    static __device__ __forceinline__ void unpack(Raw r, float2 (&v)[1]) { v[0] = r; }
    static __device__ __forceinline__ Raw pack(const float2 (&v)[1]) { return v[0]; }
};
template <> struct PairVec<__nv_bfloat16, 2> {
    using Raw = uint2;
    static __device__ __forceinline__ void unpack(Raw r, float2 (&v)[2]) {
        v[0] = make_float2(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u));
        v[1] = make_float2(__uint_as_float(r.y << 16), __uint_as_float(r.y & 0xffff0000u));
    }
    static __device__ __forceinline__ Raw pack(const float2 (&v)[2]) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0].x, v[0].y), b = __floats2bfloat162_rn(v[1].x, v[1].y);
        return make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
    }
};
template <> struct PairVec<__nv_bfloat16, 1> {   // one channel pair per lane: 4-byte accesses, half the registers
    using Raw = unsigned int;
    static __device__ __forceinline__ void unpack(Raw r, float2 (&v)[1]) { v[0] = make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); }
    static __device__ __forceinline__ Raw pack(const float2 (&v)[1]) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0].x, v[0].y);
        return *reinterpret_cast<const uint32_t *>(&a);
    }
};
template <> struct PairVec<__half, 1> {
    using Raw = unsigned int;
    static __device__ __forceinline__ void unpack(Raw r, float2 (&v)[1]) { v[0] = __half22float2(*reinterpret_cast<const __half2 *>(&r)); }
    static __device__ __forceinline__ Raw pack(const float2 (&v)[1]) {
        const __half2 a = __floats2half2_rn(v[0].x, v[0].y);
        return *reinterpret_cast<const uint32_t *>(&a);
    }
};
template <> struct PairVec<__half, 2> {
    using Raw = uint2;
    static __device__ __forceinline__ void unpack(Raw r, float2 (&v)[2]) {
        v[0] = __half22float2(*reinterpret_cast<const __half2 *>(&r.x));
        v[1] = __half22float2(*reinterpret_cast<const __half2 *>(&r.y));
    }
    static __device__ __forceinline__ Raw pack(const float2 (&v)[2]) {
        const __half2 a = __floats2half2_rn(v[0].x, v[0].y), b = __floats2half2_rn(v[1].x, v[1].y);
        return make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
    }
};
__device__ __forceinline__ float2 sigmoid2(float2 v) {
    const float2 den = fadd2(ex2_2(fmul2(v, splat2(-kLog2e))), splat2(1.0f));
    return make_float2(rcp_approx(den.x), rcp_approx(den.y));
}

template <typename T, int K, int NP>
__global__ void __launch_bounds__(128) conv1d_silu_fwd_pk_kernel(ConvParams p) {
    using PV = PairVec<T, NP>;
    using Raw = typename PV::Raw;
    constexpr int V = 2 * NP;
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * V;
    if (c >= p.ED) return;
    const int tile = blockIdx.y, b = blockIdx.z;
    const int t0 = tile * kConvTile, t1 = min(p.L, t0 + kConvTile);
    const int64_t xs = p.x_rs * (int64_t)sizeof(T), us = p.u_rs * (int64_t)sizeof(T);
    const char *xp = reinterpret_cast<const char *>(reinterpret_cast<const T *>(p.xin) + (int64_t)b * p.x_bs + c) + (int64_t)t0 * xs;
    char *up = reinterpret_cast<char *>(reinterpret_cast<T *>(p.u) + (int64_t)b * p.u_bs + c) + (int64_t)t0 * us;
    float2 w[NP][K], bias[NP], win[NP][K];   // win[.][k] = xin[t - (K-1) + k]
#pragma unroll
    for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) w[i][k] = make_float2(__ldg(p.w + (size_t)(c + 2 * i) * K + k), __ldg(p.w + (size_t)(c + 2 * i + 1) * K + k));
        bias[i] = p.bias ? make_float2(__ldg(p.bias + c + 2 * i), __ldg(p.bias + c + 2 * i + 1)) : make_float2(0.f, 0.f);
    }
    const T *cin = reinterpret_cast<const T *>(p.cin) + ((size_t)b * p.ED + c) * (K - 1);   // row t < 0: cin[t + K - 1]
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
        const int t = t0 - (K - 1) + k;
        float2 v[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) v[i] = make_float2(0.f, 0.f);
        if (t >= 0) {
            PV::unpack(__ldcs(reinterpret_cast<const Raw *>(xp + (int64_t)(k - (K - 1)) * xs)), v);
        } else if (p.cin != nullptr) {
#pragma unroll
            for (int i = 0; i < NP; ++i) v[i] = make_float2(to_f(cin[2 * i * (K - 1) + k]), to_f(cin[(2 * i + 1) * (K - 1) + k]));
        }
#pragma unroll
        for (int i = 0; i < NP; ++i) win[i][k + 1] = v[i];
    }
    constexpr int U = 8;
    auto group = [&](auto full_c, int nrows) {
        constexpr bool FULL = decltype(full_c)::value;
        Raw xr[U];
#pragma unroll
        for (int j = 0; j < U; ++j)
            if (FULL || j < nrows) xr[j] = __ldcs(reinterpret_cast<const Raw *>(xp + j * xs));
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (FULL || j < nrows) {
                float2 v[NP], o[NP];
                PV::unpack(xr[j], v);
#pragma unroll
                for (int i = 0; i < NP; ++i) {
#pragma unroll
                    for (int k = 0; k < K - 1; ++k) win[i][k] = win[i][k + 1];
                    win[i][K - 1] = v[i];
                    float2 acc = bias[i];
#pragma unroll
                    for (int k = 0; k < K; ++k) acc = ffma2(w[i][k], win[i][k], acc);
                    o[i] = fmul2(acc, sigmoid2(acc));
                }
                __stcs(reinterpret_cast<Raw *>(up + j * us), PV::pack(o));
            }
        }
        xp += U * xs;
        up += U * us;
    };
    int tb = t0;
    for (; tb + U <= t1; tb += U) group(std::true_type{}, U);
    if (tb < t1) group(std::false_type{}, t1 - tb);
    if (p.cout != nullptr && blockIdx.y == gridDim.y - 1) {   // last tile: the window holds the last K-1 rows of cat(cin, xin)
        T *cout = reinterpret_cast<T *>(p.cout) + ((size_t)blockIdx.z * p.ED + (blockIdx.x * blockDim.x + threadIdx.x) * V) * (K - 1);
#pragma unroll
        for (int i = 0; i < NP; ++i) {
#pragma unroll
            for (int k = 0; k < K - 1; ++k) {
                cout[2 * i * (K - 1) + k] = from_f<T>(win[i][k + 1].x);
                cout[(2 * i + 1) * (K - 1) + k] = from_f<T>(win[i][k + 1].y);
            }
        }
    }
}

template <typename T, int K, int NP>
__global__ void __launch_bounds__(128) conv1d_silu_bwd_pk_kernel(ConvParams p) {
    using PV = PairVec<T, NP>;
    using Raw = typename PV::Raw;
    constexpr int V = 2 * NP;
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * V;
    if (c >= p.ED) return;
    const int tile = blockIdx.y, b = blockIdx.z;
    const int t0 = tile * kConvTile, t1 = min(p.L, t0 + kConvTile);
    const int64_t xs = p.x_rs * (int64_t)sizeof(T), gs = p.du_rs * (int64_t)sizeof(T), ds = p.dx_rs * (int64_t)sizeof(T);
    const char *xp = reinterpret_cast<const char *>(reinterpret_cast<const T *>(p.xin) + (int64_t)b * p.x_bs + c) + (int64_t)t0 * xs;
    const char *gp = reinterpret_cast<const char *>(reinterpret_cast<const T *>(p.du) + (int64_t)b * p.du_bs + c) + (int64_t)t0 * gs;
    // dxin[s] is complete when dv[s + K - 1] is known: the row stored while step t is processed is t - (K - 1)
    char *dp = reinterpret_cast<char *>(reinterpret_cast<T *>(p.dxin) + (int64_t)b * p.dx_bs + c) + (int64_t)(t0 - (K - 1)) * ds;
    float2 w[NP][K], bias[NP], win[NP][K], dvw[NP][K], dw[NP][K], db[NP];   // dvw[.][k] = dv[t - (K-1) + k]
#pragma unroll
    for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            w[i][k] = make_float2(__ldg(p.w + (size_t)(c + 2 * i) * K + k), __ldg(p.w + (size_t)(c + 2 * i + 1) * K + k));
            dvw[i][k] = dw[i][k] = make_float2(0.f, 0.f);
        }
        bias[i] = p.bias ? make_float2(__ldg(p.bias + c + 2 * i), __ldg(p.bias + c + 2 * i + 1)) : make_float2(0.f, 0.f);
        db[i] = make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
        const int t = t0 - (K - 1) + k;
        float2 v[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) v[i] = make_float2(0.f, 0.f);
        if (t >= 0) PV::unpack(__ldcs(reinterpret_cast<const Raw *>(xp + (int64_t)(k - (K - 1)) * xs)), v);
#pragma unroll
        for (int i = 0; i < NP; ++i) win[i][k + 1] = v[i];
    }
    // dv is needed K-1 steps past the tile to finish dxin of the tile's last steps
    const int tend = t1 + (K - 1);
    constexpr int U = 8;
    // MAIN: every row of the group lies in [t0, t1) and its output row t - (K-1) >= t0 is checked per row only in the first group
    auto group = [&](auto main_c, int tb) {
        constexpr bool MAIN = decltype(main_c)::value;   // all U rows < t1 (hence < L): own-tile rows, no bounds checks on loads
        Raw xr[U], gr[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (MAIN || tb + j < p.L) {
                xr[j] = __ldcs(reinterpret_cast<const Raw *>(xp + j * xs));
                gr[j] = __ldcs(reinterpret_cast<const Raw *>(gp + j * gs));
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int t = tb + j;
            if (MAIN || t < tend) {
                float2 xv[NP], gv[NP], o[NP];
                const bool live = MAIN || t < p.L;
                if (live) { PV::unpack(xr[j], xv); PV::unpack(gr[j], gv); }
#pragma unroll
                for (int i = 0; i < NP; ++i) {
#pragma unroll
                    for (int k = 0; k < K - 1; ++k) { win[i][k] = win[i][k + 1]; dvw[i][k] = dvw[i][k + 1]; }
                    float2 dv = make_float2(0.f, 0.f);
                    if (live) {
                        win[i][K - 1] = xv[i];
                        float2 v = bias[i];
#pragma unroll
                        for (int k = 0; k < K; ++k) v = ffma2(w[i][k], win[i][k], v);
                        const float2 sg = sigmoid2(v);
                        // d silu = sg (1 + v (1 - sg)) = sg (1 + v - v sg)
                        const float2 vs = fmul2(v, sg);
                        dv = fmul2(fmul2(gv[i], sg), fadd2(fadd2(v, splat2(1.0f)), make_float2(-vs.x, -vs.y)));
                        if (MAIN || t < t1) {   // parameter gradients: own tile only
                            db[i] = fadd2(db[i], dv);
#pragma unroll
                            for (int k = 0; k < K; ++k) dw[i][k] = ffma2(dv, win[i][k], dw[i][k]);
                        }
                    }
                    dvw[i][K - 1] = dv;
                    float2 acc = fmul2(w[i][0], dvw[i][K - 1]);
#pragma unroll
                    for (int k = 1; k < K; ++k) acc = ffma2(w[i][k], dvw[i][K - 1 - k], acc);
                    o[i] = acc;
                }
                const int s_out = t - (K - 1);
                if (s_out >= t0 && s_out < t1) __stcs(reinterpret_cast<Raw *>(dp + j * ds), PV::pack(o));
            }
        }
        xp += U * xs;
        gp += U * gs;
        dp += U * ds;
    };
    int tb = t0;
    for (; tb + U <= t1; tb += U) group(std::true_type{}, tb);
    for (; tb < tend; tb += U) group(std::false_type{}, tb);
    float *part = p.part + ((size_t)(b * p.ntiles + tile) * (K + 1)) * p.ED + c;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int k = 0; k < K; ++k) *reinterpret_cast<float2 *>(part + (size_t)k * p.ED + 2 * i) = dw[i][k];
        *reinterpret_cast<float2 *>(part + (size_t)K * p.ED + 2 * i) = db[i];
    }
}

// block (32 channels, 8 slices of the B * ntiles partial rows): coalesced reads, 8-way split of the serial sum
template <int K>
__global__ void __launch_bounds__(256) conv1d_bwd_finalize_kernel(ConvParams p) {
    __shared__ float s_acc[8][33];
    const int c = blockIdx.x * 32 + threadIdx.x;
    const int k = blockIdx.y;   // 0..K
    float acc = 0.f;
    const int n = p.B * p.ntiles;
    if (c < p.ED)
        for (int i = threadIdx.y; i < n; i += 8) acc += p.part[((size_t)i * (K + 1) + k) * p.ED + c];
    s_acc[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && c < p.ED) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += s_acc[q][threadIdx.x];
        if (k < K) p.dw[(size_t)c * K + k] = t;
        else if (p.dbias) p.dbias[c] = t;
    }
}

// channels per lane: 8-byte accesses when every base pointer and stride keeps them aligned, else one channel per lane
template <typename T>
static int conv_vec(const ConvParams &p, bool bwd) {
    constexpr int V = 8 / (int)sizeof(T);
    if (p.ED % V != 0) return 1;
    auto ok = [&](const void *q, int64_t bs, int64_t rs) {
        return q == nullptr || ((reinterpret_cast<uintptr_t>(q) & 7) == 0 && (bs * (int64_t)sizeof(T)) % 8 == 0 && (rs * (int64_t)sizeof(T)) % 8 == 0);
    };
    bool a = ok(p.xin, p.x_bs, p.x_rs);
    a = a && (bwd ? ok(p.du, p.du_bs, p.du_rs) && ok(p.dxin, p.dx_bs, p.dx_rs) : ok(p.u, p.u_bs, p.u_rs));
    return a ? V : 1;
}

template <typename T, int K>
static int conv_fwd_launch(ConvParams &p, cudaStream_t st) {
    constexpr int V = 8 / (int)sizeof(T);
    const int v = conv_vec<T>(p, false);
    const dim3 block(128), grid((p.ED / v + 127) / 128, p.ntiles, p.B);
    { ScopedKernelTimer tm(K_CONV_FWD, st);
      if (v == V) conv1d_silu_fwd_pk_kernel<T, K, V / 2><<<grid, block, 0, st>>>(p);
      else conv1d_silu_fwd_kernel<T, K, 1><<<grid, block, 0, st>>>(p); }
    return check_launch("conv1d_silu_fwd");
}

template <typename T, int K>
static int conv_bwd_launch(ConvParams &p, cudaStream_t st) {
    constexpr int V = 8 / (int)sizeof(T);
    const int v = conv_vec<T>(p, true);
    const dim3 block(128), grid((p.ED / v + 127) / 128, p.ntiles, p.B);
    { ScopedKernelTimer tm(K_CONV_BWD, st);
      // packed backward: one channel pair per lane for every dtype (16-bit: 4-byte accesses, 94 registers, 5 % faster than
      // two pairs with 8-byte accesses and 166 registers)
      if (v == V) conv1d_silu_bwd_pk_kernel<T, K, 1><<<dim3((p.ED / 2 + 127) / 128, p.ntiles, p.B), block, 0, st>>>(p);
      else conv1d_silu_bwd_kernel<T, K, 1><<<grid, block, 0, st>>>(p); }
    int rc = check_launch("conv1d_silu_bwd");
    if (rc != GFE_OK) return rc;
    { ScopedKernelTimer tm(K_CONV_BWD_FIN, st);
      conv1d_bwd_finalize_kernel<K><<<dim3((p.ED + 31) / 32, K + 1), dim3(32, 8), 0, st>>>(p); }
    return check_launch("conv1d_bwd_finalize");
}

template <typename T>
static int conv_dispatch_k(bool bwd, int K, ConvParams &p, cudaStream_t st) {
    switch (K) {
        case 2: return bwd ? conv_bwd_launch<T, 2>(p, st) : conv_fwd_launch<T, 2>(p, st);
        case 3: return bwd ? conv_bwd_launch<T, 3>(p, st) : conv_fwd_launch<T, 3>(p, st);
        case 4: return bwd ? conv_bwd_launch<T, 4>(p, st) : conv_fwd_launch<T, 4>(p, st);
        default: set_error("conv1d: d_conv=%d unsupported (2..4 compiled)", K); return GFE_ERR_UNSUPPORTED;
    }
}

static int conv_dispatch(bool bwd, int K, int dtype, ConvParams &p, cudaStream_t st) {
    switch (dtype) {
        case GFE_F32: return conv_dispatch_k<float>(bwd, K, p, st);
        case GFE_BF16: return conv_dispatch_k<__nv_bfloat16>(bwd, K, p, st);
        case GFE_F16: return conv_dispatch_k<__half>(bwd, K, p, st);
        default: set_error("conv1d: bad dtype %d", dtype); return GFE_ERR_DTYPE;
    }
}

}  // namespace gfe

extern "C" {

GFE_API int gfe_conv1d_silu_fwd(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                void *u, int64_t u_bs, int64_t u_rs, int B, int L, int ED, int K, int dtype,
                                void *stream) {
    return gfe_conv1d_silu_fwd_state(xin, x_bs, x_rs, w, bias, nullptr, nullptr, u, u_bs, u_rs, B, L, ED, K, dtype, stream);
}

GFE_API int gfe_conv1d_silu_fwd_state(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                      const void *inputs, void *new_inputs, void *u, int64_t u_bs, int64_t u_rs,
                                      int B, int L, int ED, int K, int dtype, void *stream) {
    using namespace gfe;
    if (!xin || !w || !u) { set_error("conv1d_fwd: NULL pointer"); return GFE_ERR_ARG; }
    if (B <= 0 || L <= 0 || ED <= 0 || B > 65535) { set_error("conv1d_fwd: bad shape"); return GFE_ERR_ARG; }
    if (inputs != nullptr && new_inputs != nullptr && K >= 2) {
        const size_t bytes = (size_t)B * ED * (K - 1) * (dtype == GFE_F32 ? 4 : 2);
        const char *a = reinterpret_cast<const char *>(inputs), *c = reinterpret_cast<const char *>(new_inputs);
        if (a < c + bytes && c < a + bytes) { set_error("conv1d_fwd: inputs and new_inputs overlap"); return GFE_ERR_ARG; }
    }
    ConvParams p{};
    p.xin = xin; p.u = u; p.w = w; p.bias = bias; p.cin = inputs; p.cout = new_inputs;
    p.x_bs = x_bs; p.x_rs = x_rs; p.u_bs = u_bs; p.u_rs = u_rs;
    p.B = B; p.L = L; p.ED = ED; p.ntiles = (L + kConvTile - 1) / kConvTile;
    return conv_dispatch(false, K, dtype, p, reinterpret_cast<cudaStream_t>(stream));
}

GFE_API size_t gfe_conv1d_bwd_workspace_bytes(int B, int L, int ED, int K) {
    if (B <= 0 || L <= 0 || ED <= 0 || K <= 0) return 0;
    const size_t ntiles = (L + gfe::kConvTile - 1) / gfe::kConvTile;
    return (size_t)B * ntiles * (K + 1) * ED * sizeof(float);
}

GFE_API int gfe_conv1d_silu_bwd(const void *xin, int64_t x_bs, int64_t x_rs, const float *w, const float *bias,
                                const void *du, int64_t du_bs, int64_t du_rs,
                                void *dxin, int64_t dx_bs, int64_t dx_rs, float *dw, float *dbias,
                                int B, int L, int ED, int K, int dtype, void *ws, size_t ws_bytes, void *stream) {
    using namespace gfe;
    if (!xin || !w || !du || !dxin || !dw) { set_error("conv1d_bwd: NULL pointer"); return GFE_ERR_ARG; }
    if (B <= 0 || L <= 0 || ED <= 0 || B > 65535) { set_error("conv1d_bwd: bad shape"); return GFE_ERR_ARG; }
    const size_t need = gfe_conv1d_bwd_workspace_bytes(B, L, ED, K);
    if (!ws || ws_bytes < need) { set_error("conv1d_bwd: workspace too small (%zu < %zu)", ws ? ws_bytes : (size_t)0, need); return GFE_ERR_WORKSPACE; }
    ConvParams p{};
    p.xin = xin; p.du = du; p.dxin = dxin; p.w = w; p.bias = bias; p.dw = dw; p.dbias = dbias;
    p.part = reinterpret_cast<float *>(ws);
    p.x_bs = x_bs; p.x_rs = x_rs; p.du_bs = du_bs; p.du_rs = du_rs; p.dx_bs = dx_bs; p.dx_rs = dx_rs;
    p.B = B; p.L = L; p.ED = ED; p.ntiles = (L + kConvTile - 1) / kConvTile;
    return conv_dispatch(true, K, dtype, p, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
