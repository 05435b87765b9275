// selscan_shared.cuh -- parameter block and device helpers shared by every selective-scan kernel
// (chained kernels in selscan_v4_fwd.cu / selscan_chain_bwd.cu, their segment summaries in selscan_seg.cu, generic kernels in selscan.cu).
#pragma once

#include "common.cuh"

namespace gfe {

struct ScanParams {
    int B, L, ED;
    int nseg, seg_len, nchunks;
    uint32_t flags;
    const void *u, *delta, *z, *Bm, *Cm;
    int64_t u_bs, u_rs, d_bs, d_rs, z_bs, z_rs, B_bs, B_rs, C_bs, C_rs;
    const float *A_log, *D, *dt_bias;
    void *out;
    int64_t o_bs, o_rs;
    float *last_state;
    float2 *ckpt;   // [B][nchunks][N / 2][ED]
    void *ysave;    // [B][L][ED] activation dtype: y before the gate, lives behind ckpt (written by the chained kernels only)
    float2 *seg_h;  // [B][nseg][N / 2][ED]  segment-local end state (fwd) / start carry (bwd)
    float *seg_sd;  // [B][nseg][ED]     sum of delta over the segment
    // backward
    const void *dout;
    int64_t do_bs, do_rs;
    void *du, *ddelta, *dz, *dBm, *dCm;
    int64_t du_bs, du_rs, dd_bs, dd_rs, dz_bs, dz_rs, dB_bs, dB_rs, dC_bs, dC_rs;
    float *dA_log, *dD, *ddt_bias;
    float *part_bc;   // [G][B][L][2 N]   per-warp dB|dC rows
    float *part_par;  // [B][nseg][N + 2][ED]
    int G;            // ceil(ED / 32)
    int bc_interleaved;   // part_bc rows: 1 = {dB[n], dC[n]} pairs (chained backward), 0 = dB[N] | dC[N] (generic backward)
    const float *h0;      // forward: (B, ED, N) state before token 0 (gfe_selscan_fwd_state), or NULL: zeros
    // backward through a carried state (gfe_selscan_bwd_carry), (B, ED, N) like last_state, or NULL: dlast seeds the reverse
    // carry of the last token (NULL: zeros), dh0 receives the reverse carry left after token 0 (NULL: not written)
    const float *dlast;
    float *dh0;
};

constexpr int kPairs = kNState / 2;

// Dynamic chaining of L-segments (chained kernels): persistent CTAs draw (segment, batch row, channel block) units from an
// atomic counter in segment-major order; a unit waits for the flag of its predecessor segment, reads the carried
// state, and publishes its own.  Units are drawn in dependency order, so a waiting CTA only ever waits on a unit that
// is already running or finished: no deadlock, no tail quantisation, no recomputation.
struct ChainSched {
    int *counter;   // [1]
    int *flags;     // [nseg][B * nblk], zeroed before the launch
    float *carry;   // [B][ED][16] state handed from one segment to the next
    int nseg, seg_len, nblk, total;
    // Independent segments (small B * ED: too few chains to fill the GPU by waiting): every segment's carry-in is known
    // before the launch -- a summary pass (selscan_seg.cu) leaves each segment's local aggregate and sum(delta), a combine
    // pass turns them into carries -- so units neither wait nor publish.
    int independent;
    float *segc;    // [nseg - 1][B][ED][16]  slot s: forward carry-in of segment s + 1 / reverse carry-in of segment s
    float *segsd;   // [nseg - 1][B][ED]      sum of delta over the segment the slot's aggregate was taken from
};

#ifdef __CUDACC__
// ---- cp.async helpers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one 16-byte piece, global -> shared, bypassing L1
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// exp2 of two non-positive arguments on the FMA pipe: Cody-Waite split + degree-5 minimax with p(0) = 1 exactly (max rel err 2.4e-7
// in fp32, same class as ex2.approx), exponent inserted with integer adds.
__device__ __forceinline__ float2 ex2_poly2(float2 x) {
    x.x = fmaxf(x.x, -125.0f);
    x.y = fmaxf(x.y, -125.0f);
    const float2 magic = make_float2(12582912.0f, 12582912.0f);
    const float2 t = fadd2(x, magic);
    const float2 n = fadd2(t, make_float2(-12582912.0f, -12582912.0f));
    const float2 f = fadd2(x, make_float2(-n.x, -n.y));
    float2 p = make_float2(0.001327647129073739f, 0.001327647129073739f);
    p = ffma2(p, f, make_float2(0.009675540961325169f, 0.009675540961325169f));
    p = ffma2(p, f, make_float2(0.05550713092088699f, 0.05550713092088699f));
    p = ffma2(p, f, make_float2(0.24022120237350464f, 0.24022120237350464f));
    p = ffma2(p, f, make_float2(0.6931469440460205f, 0.6931469440460205f));
    p = ffma2(p, f, make_float2(1.0f, 1.0f));
    return make_float2(__int_as_float(__float_as_int(p.x) + (__float_as_int(t.x) << 23)),
                       __int_as_float(__float_as_int(p.y) + (__float_as_int(t.y) << 23)));
}

// Branch-free softplus of two values (one formulation for every x, so it can be interleaved with other work):
// softplus(x) = max(x, 0) + log1p(w), w = exp(-|x|) in (0, 1], log1p(w) = 2 atanh(w / (2 + w)) with six odd terms
// (s^2 <= 1/9: relative error < 1e-6 for every x; x > 20 returns x to fp32 rounding, the torch threshold).
// Not ln2 * lg2(1 + w): for x < 0 that rounds 1 + w to fp32 before the logarithm and lg2.approx is accurate to 2^-22.6 only
// in ABSOLUTE terms, so delta = softplus(x) loses all relative accuracy below x ~ -10 (100 % below -16.6) -- the step sizes
// of long-memory channels, where the generic and decode kernels (softplus_only, the same series) stay exact.
// Optionally sig = sigmoid(x) = d softplus / dx.
template <bool WANT_SIG>
__device__ __forceinline__ float2 softplus_pair(float2 x, float2 &sig) {
    const float2 w = ex2_2(make_float2(fabsf(x.x) * -kLog2e, fabsf(x.y) * -kLog2e));
    const float2 d = fadd2(w, splat2(2.0f));
    const float2 s = fmul2(w, make_float2(rcp_approx(d.x), rcp_approx(d.y)));
    const float2 s2 = fmul2(s, s);
    float2 p = ffma2(s2, splat2(2.0f / 11.0f), splat2(2.0f / 9.0f));
    p = ffma2(p, s2, splat2(2.0f / 7.0f));
    p = ffma2(p, s2, splat2(2.0f / 5.0f));
    p = ffma2(p, s2, splat2(2.0f / 3.0f));
    p = ffma2(p, s2, splat2(2.0f));
    const float2 r = fmul2(s, p);
    if (WANT_SIG) {
        const float2 q = make_float2(rcp_approx(1.0f + w.x), rcp_approx(1.0f + w.y));   // sigmoid(|x|)
        sig = make_float2(x.x >= 0.f ? q.x : w.x * q.x, x.y >= 0.f ? q.y : w.y * q.y);
    }
    return make_float2(fmaxf(x.x, 0.f) + r.x, fmaxf(x.y, 0.f) + r.y);
}

// Element type of the chained kernels' state checkpoints: fp32, except bf16 for bf16 activations (half the checkpoint
// stream; the recomputed states then carry a 2^-9 relative error, well inside the 2e-2 tolerance of that dtype; fp16 keeps
// fp32 checkpoints: states can exceed its range).
template <typename T> struct CkptOf { using type = float; };
template <> struct CkptOf<__nv_bfloat16> { using type = __nv_bfloat16; };
__device__ __forceinline__ void ckpt_store(float *dst, float4 v) { __stcs(reinterpret_cast<float4 *>(dst), v); }
__device__ __forceinline__ void ckpt_store(__nv_bfloat16 *dst, float4 v) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    __stcs(reinterpret_cast<uint2 *>(dst), make_uint2(*reinterpret_cast<const uint32_t *>(&lo), *reinterpret_cast<const uint32_t *>(&hi)));
}
__device__ __forceinline__ float4 ckpt_load_smem(const float *src) { return *reinterpret_cast<const float4 *>(src); }
__device__ __forceinline__ float4 ckpt_load_smem(const __nv_bfloat16 *src) {
    const uint2 r = *reinterpret_cast<const uint2 *>(src);
    const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&r.x)), hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&r.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// ---- chained-unit plumbing -----------------------------------------------------------------------------
__device__ __forceinline__ int ld_acquire(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- two adjacent channels at a time (item phases of the chained kernels) ------------------------------------
template <typename T> struct Pair;
template <> struct Pair<float> { using type = float2; };
template <> struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };
template <> struct Pair<__half> { using type = __half2; };
__device__ __forceinline__ float2 pair_to_f(float2 v) { return v; }
__device__ __forceinline__ float2 pair_to_f(__nv_bfloat162 v) { return __bfloat1622float2(v); }
__device__ __forceinline__ float2 pair_to_f(__half2 v) { return __half22float2(v); }
template <typename T> __device__ __forceinline__ typename Pair<T>::type pair_from_f(float a, float b);
template <> __device__ __forceinline__ float2 pair_from_f<float>(float a, float b) { return make_float2(a, b); }
template <> __device__ __forceinline__ __nv_bfloat162 pair_from_f<__nv_bfloat16>(float a, float b) { return __floats2bfloat162_rn(a, b); }
template <> __device__ __forceinline__ __half2 pair_from_f<__half>(float a, float b) { return __floats2half2_rn(a, b); }

// elements 2i, 2i+1 of a shared tile row (the tile base is 16-byte aligned)
template <typename T> __device__ __forceinline__ float2 lds_pair(const T *row, int i) {
    return pair_to_f(reinterpret_cast<const typename Pair<T>::type *>(row)[i]);
}
// four consecutive elements of a shared tile (8- / 16-byte aligned) as fp32: one load
__device__ __forceinline__ float4 lds_quad(const float *src) { return *reinterpret_cast<const float4 *>(src); }
__device__ __forceinline__ float4 lds_quad(const __nv_bfloat16 *src) { return ckpt_load_smem(src); }
__device__ __forceinline__ float4 lds_quad(const __half *src) {
    const uint2 r = *reinterpret_cast<const uint2 *>(src);
    const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&r.x)), hi = __half22float2(*reinterpret_cast<const __half2 *>(&r.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}
// streaming store of two adjacent channels; `vec` says whether the destination allows one paired store
template <typename T> __device__ __forceinline__ void stg_pair(T *dst, float a, float b, bool vec) {
    if (vec) {
        __stcs(reinterpret_cast<typename Pair<T>::type *>(dst), pair_from_f<T>(a, b));
    } else {
        st_stream(dst, from_f<T>(a));
        st_stream(dst + 1, from_f<T>(b));
    }
}

// Copy nrows rows of ROW_ELEMS contiguous elements (row stride rs elements) into a dense shared tile with plain loads, all
// NT threads of the CTA taking part: the staging path of tensors whose bases or strides rule out 16-byte cp.async pieces.
template <typename T, int ROW_ELEMS, int NT>
__device__ __forceinline__ void stage_tile(unsigned char *dst, const T *src, int64_t rs, int nrows, int tid) {
    const int total = nrows * ROW_ELEMS;
    T *d = reinterpret_cast<T *>(dst);
    for (int i = tid; i < total; i += NT) {
        const int row = i / ROW_ELEMS, col = i % ROW_ELEMS;
        d[i] = src[(int64_t)row * rs + col];
    }
}
#endif  // __CUDACC__

// Grid of a persistent kernel: min(total units, resident CTAs of the CURRENT device).  The dynamic-shared-memory opt-in
// is a per-device attribute and the occupancy depends on the device, so both are cached per (kernel, device).
#ifdef __CUDACC__
template <auto Kernel>
static int persistent_grid(int nt, size_t smem, int total) {
    constexpr int kMaxDev = 64;
    static int slots_of[kMaxDev];   // 0 = not asked yet (benign race: every thread computes the same value)
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = 0; }
    int slots = (dev >= 0 && dev < kMaxDev) ? slots_of[dev] : 0;
    if (slots == 0) {
        int per_sm = 0;
        cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, nt, smem) != cudaSuccess || per_sm < 1) {
            (void)cudaGetLastError();
            per_sm = 1;
        }
        slots = sm_count() * per_sm;
        if (dev >= 0 && dev < kMaxDev) slots_of[dev] = slots;
    }
    return total < slots ? total : slots;
}
#endif

// host side of the chained kernels (selscan_chain_host.cu, selscan_chain_bwd.cu)
// CTAs of 128 threads per SM that the chained kernels' register budgets (__launch_bounds__) and the launch plans are set for.
// Forward 3: 4 (126 registers) measured 2-8 % slower on cfg3 and cfg5.  Backward 2: 255 registers without spills; 3 caps
// it at 168 registers with spills and measured slower on both (profiles/r02_chain_variants.txt).
constexpr int kFwdMinBlocks = 3;
constexpr int kBwdMinBlocks = 2;
struct ChainPlan {
    int cpc, nblk;          // channel-block width and count
    int nseg, seg_len;      // L-segments (seg_len a multiple of kChunk)
    int independent;        // 0: segments wait for their predecessor; 1: carries come from the summary + combine passes
};
ChainPlan chain_fwd_plan(int B, int L, int ED);
ChainPlan chain_bwd_plan(int B, int L, int ED);
bool chain_applicable(int B, int L, int ED, int N);       // shape-only: both directions take the same decision
size_t chain_ckpt_state_bytes(int B, int L, int ED, int dtype);
size_t chain_fwd_workspace_bytes(int B, int L, int ED);
size_t chain_bwd_workspace_bytes(int B, int L, int ED);
int chain_launch_fwd(const gfe_selscan_args *a, const float *h0, cudaStream_t st);   // h0: state before token 0, or NULL
int chain_launch_bwd(const gfe_selscan_args *a, const float *dlast, float *dh0, cudaStream_t st);   // NULL, NULL: zero end carry
// the summary of a whole range (gfe_selscan_summary_fwd / _bwd): chained family, and the fold both families end with
size_t chain_summary_workspace_bytes(int B, int L, int ED);
int chain_launch_summary(const gfe_selscan_args *a, bool rev, float *out, float *sum_delta, cudaStream_t st);
int launch_summary_total(const float *loc, const float *segsd, const float *A_log, float *out, float *sum_delta, int nseg, int B,
                         int ED, int N, bool generic, bool rev, cudaStream_t st);   // selscan_seg.cu

}  // namespace gfe
