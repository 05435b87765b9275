// pscan.cu -- the reference's pscan(A, X) API (cross_atten/pscan.py:152-224) as HBM-streaming kernels.
//
// H[t] = A[t] * H[t-1] + X[t] per (b, d, n).  The reference runs a Blelloch tree with 2*log2(L) strided
// passes over two cloned, power-of-two padded tensors; here every thread owns 4 adjacent (d, n)
// elements (one 128-bit lane of the contiguous D*N axis), walks L sequentially with the running state
// in registers and touches every input/output element exactly once:
//   forward : read A, X            write H          (12 B / element)
//   backward: read A, dH, H        write dA, dX     (20 B / element)
// Padding to a power of two is unnecessary (it is appended after L-1 and never changes [0, L)).
// HBM needs ~12 MB of loads in flight; a launch has B*D*N*4*nloads*U bytes in flight (U = steps whose loads are issued before
// the first is used), so small problems run the SAME single pass with narrower vectors and a deeper unroll -- forward (V, U)
// = (4, 16) or (1, 32), backward (4, 8), (2, 16) or (1, 32), chosen from measurements (profiles/r02_pscan.txt) -- instead of
// paying a second pass.  Only when even
// that cannot fill the GPU (B*D*N below ~25 k elements, e.g. one long sequence with few channels) is L split into segments:
// pass 1 reduces each segment to its (product of A, local end state) pair, pass 2 starts each segment from the combined carry.
// The split only ever follows the fall to (1, 32), so the summary passes exist as (1, 32) alone; misaligned operands also run
// (1, 32).  Compiled: forward (4, 16), (1, 32), (1, 32) summary; backward (4, 8), (2, 16), (1, 32), (1, 32) summary.
#include "common.cuh"

namespace gfe {

constexpr int kPsUnrollMax = 32;

struct PscanPlan {
    int nseg, seg_len;
    int V, U;   // elements per thread, steps per load batch
};

// nloads = tensors read per step: 2 forward (A, X), 3 backward (A, dH, H): backward reaches the same bytes in flight with
// fewer steps, so it keeps the wider vectors longer (measured at B=8, L=1024, D=1024: (4, 8) 98 % of the HBM peak, (2, 16) 88 %).
static PscanPlan pscan_plan(int B, int L, int64_t DN, int nloads) {
    PscanPlan p;
    const double target = 12e6 * sm_count() / 148.0;            // bytes in flight that saturate HBM (Little: ~6.5 TB/s x ~1.5 us)
    const double per_u = (double)B * (double)DN * 4.0 * nloads;  // bytes requested per unrolled step
    if (nloads == 2) {   // forward: (4, 16) when that alone fills the pipe, else the narrowest vectors and the deepest unroll
        p.V = 4; p.U = 16;
        if (DN % 4 != 0 || per_u * 16 < target) { p.V = 1; p.U = 32; }
    } else {             // backward
        p.V = 4; p.U = 8;
        if (DN % 4 != 0 || per_u * 8 < target) { p.V = 2; p.U = 16; }
        if (DN % 2 != 0 || per_u * 16 < target) { p.V = 1; p.U = 32; }
    }
    int S = 1;
    if (per_u * p.U * 2 < target) {   // still less than half of it: split L (re-reads A and X once more)
        S = (int)(target / (per_u * p.U));
        const int max_by_len = L / 64;
        if (S > max_by_len) S = max_by_len;
        if (S > kMaxSeg) S = kMaxSeg;
        if (S < 1) S = 1;
    }
    p.seg_len = (int)ceil_div64(ceil_div64(L, S), kPsUnrollMax) * kPsUnrollMax;
    p.nseg = (int)ceil_div64(L, p.seg_len);
    return p;
}

template <int V> struct Vec;
template <> struct Vec<4> {
    using type = float4;
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ float4 one() { return make_float4(1.f, 1.f, 1.f, 1.f); }
    static __device__ __forceinline__ float4 fma(float4 a, float4 b, float4 c) {
        return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
    }
    static __device__ __forceinline__ float4 mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
    static __device__ __forceinline__ float4 add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
};
template <> struct Vec<2> {
    using type = float2;
    static __device__ __forceinline__ float2 zero() { return make_float2(0.f, 0.f); }
    static __device__ __forceinline__ float2 one() { return make_float2(1.f, 1.f); }
    static __device__ __forceinline__ float2 fma(float2 a, float2 b, float2 c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
    static __device__ __forceinline__ float2 mul(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
    static __device__ __forceinline__ float2 add(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
};
template <> struct Vec<1> {
    using type = float;
    static __device__ __forceinline__ float zero() { return 0.f; }
    static __device__ __forceinline__ float one() { return 1.f; }
    static __device__ __forceinline__ float fma(float a, float b, float c) { return fmaf(a, b, c); }
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
};

struct PscanParams {
    const float *A, *X, *H, *dH;
    float *Hout, *dA, *dX;
    float *segP, *segS;   // [B][nseg][DN]
    int B, L, nseg, seg_len;
    int64_t DN;           // D*N
};

// ---- forward -----------------------------------------------------------------------------------------
template <int V, int U, bool SUMMARY>
__global__ void __launch_bounds__(128) pscan_fwd_kernel(PscanParams p) {
    constexpr int kPsUnroll = U;
    using VT = typename Vec<V>::type;
    const int64_t nvec = p.DN / V;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nvec) return;
    const int seg = blockIdx.y, b = blockIdx.z;
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);
    const VT *A = reinterpret_cast<const VT *>(p.A + (size_t)b * p.L * p.DN) + i;
    const VT *X = reinterpret_cast<const VT *>(p.X + (size_t)b * p.L * p.DN) + i;
    VT *H = SUMMARY ? nullptr : reinterpret_cast<VT *>(p.Hout + (size_t)b * p.L * p.DN) + i;

    VT h = Vec<V>::zero(), P = Vec<V>::one();
    if (!SUMMARY) {
        for (int s = 0; s < seg; ++s) {
            const size_t o = ((size_t)b * p.nseg + s) * p.DN;
            h = Vec<V>::fma(reinterpret_cast<const VT *>(p.segP + o)[i], h, reinterpret_cast<const VT *>(p.segS + o)[i]);
        }
    }
    for (int tb = t0; tb < t1; tb += kPsUnroll) {   // (double-buffered load batches were measured slower: 150+ registers)
        VT a[kPsUnroll], x[kPsUnroll];
#pragma unroll
        for (int j = 0; j < kPsUnroll; ++j) {
            const int t = min(tb + j, t1 - 1);
            a[j] = __ldcs(A + (size_t)t * nvec);
            x[j] = __ldcs(X + (size_t)t * nvec);
        }
#pragma unroll
        for (int j = 0; j < kPsUnroll; ++j) {
            if (tb + j < t1) {
                h = Vec<V>::fma(a[j], h, x[j]);
                if (SUMMARY) P = Vec<V>::mul(P, a[j]);
                else __stcs(H + (size_t)(tb + j) * nvec, h);
            }
        }
    }
    if (SUMMARY) {
        const size_t o = ((size_t)b * p.nseg + seg) * p.DN;
        reinterpret_cast<VT *>(p.segP + o)[i] = P;
        reinterpret_cast<VT *>(p.segS + o)[i] = h;
    }
}

// ---- backward ----------------------------------------------------------------------------------------
// G(t) = A[t] * g[t] is the carry handed to step t-1;  g[t] = dH[t] + G(t+1).
template <int V, int U, bool SUMMARY>
__global__ void __launch_bounds__(128) pscan_bwd_kernel(PscanParams p) {
    constexpr int kPsUnroll = U;
    using VT = typename Vec<V>::type;
    const int64_t nvec = p.DN / V;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nvec) return;
    const int seg = SUMMARY ? blockIdx.y + 1 : blockIdx.y, b = blockIdx.z;
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);
    const VT *A = reinterpret_cast<const VT *>(p.A + (size_t)b * p.L * p.DN) + i;
    const VT *dH = reinterpret_cast<const VT *>(p.dH + (size_t)b * p.L * p.DN) + i;
    const VT *H = reinterpret_cast<const VT *>(p.H + (size_t)b * p.L * p.DN) + i;
    VT *dA = SUMMARY ? nullptr : reinterpret_cast<VT *>(p.dA + (size_t)b * p.L * p.DN) + i;
    VT *dX = SUMMARY ? nullptr : reinterpret_cast<VT *>(p.dX + (size_t)b * p.L * p.DN) + i;

    VT G = Vec<V>::zero(), P = Vec<V>::one();
    if (!SUMMARY) {
        for (int s = p.nseg - 1; s > seg; --s) {
            const size_t o = ((size_t)b * p.nseg + s) * p.DN;
            G = Vec<V>::fma(reinterpret_cast<const VT *>(p.segP + o)[i], G, reinterpret_cast<const VT *>(p.segS + o)[i]);
        }
    }
    // walk [t0, t1) backwards in blocks of kPsUnroll aligned to t0
    const int nblk = (t1 - t0 + kPsUnroll - 1) / kPsUnroll;
    for (int blk = nblk - 1; blk >= 0; --blk) {
        const int tb = t0 + blk * kPsUnroll;
        VT a[kPsUnroll], g[kPsUnroll], hp[kPsUnroll];
#pragma unroll
        for (int j = 0; j < kPsUnroll; ++j) {
            const int t = min(tb + j, t1 - 1);
            a[j] = __ldcs(A + (size_t)t * nvec);
            g[j] = __ldcs(dH + (size_t)t * nvec);
            if (!SUMMARY) hp[j] = t > 0 ? __ldcs(H + (size_t)(t - 1) * nvec) : Vec<V>::zero();
        }
#pragma unroll
        for (int j = kPsUnroll - 1; j >= 0; --j) {
            if (tb + j < t1) {
                const VT gt = Vec<V>::add(g[j], G);
                if (!SUMMARY) {
                    __stcs(dX + (size_t)(tb + j) * nvec, gt);
                    __stcs(dA + (size_t)(tb + j) * nvec, Vec<V>::mul(hp[j], gt));
                } else {
                    P = Vec<V>::mul(P, a[j]);
                }
                G = Vec<V>::mul(a[j], gt);
            }
        }
    }
    if (SUMMARY) {
        const size_t o = ((size_t)b * p.nseg + seg) * p.DN;
        reinterpret_cast<VT *>(p.segP + o)[i] = P;
        reinterpret_cast<VT *>(p.segS + o)[i] = G;
    }
}

// shared-memory accesses the compiler may neither cache in registers nor reorder across the ready flags
__device__ __forceinline__ float4 ps_ld_shared(const float4 *p) {
    float4 v;
    asm volatile("ld.volatile.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ float2 ps_ld_shared(const float2 *p) {
    float2 v;
    asm volatile("ld.volatile.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ float ps_ld_shared(const float *p) {
    float v;
    asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void ps_st_shared(float4 *p, float4 v) {
    asm volatile("st.volatile.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void ps_st_shared(float2 *p, float2 v) {
    asm volatile("st.volatile.shared.v2.f32 [%0], {%1, %2};" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void ps_st_shared(float *p, float v) {
    asm volatile("st.volatile.shared.f32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "f"(v) : "memory");
}

// ---- warp-chained single pass --------------------------------------------------------------------------------------
// The sequential kernels above keep one batch of U steps in flight per thread and wait out a full memory round trip per batch:
// with few columns (B * D * N / 4 threads) that is latency-, not bandwidth-bound (forward 47-65 % of the HBM peak, round 2).
// Here the W warps of a CTA share the same 32 * V columns and take the batches of U steps in turn (warp w: batches w, w + W,
// ...).  A warp loads its batch, scans it locally from a zero carry while keeping the running products (both in place of the
// loaded values), and only then needs the carry of the previous batch: it picks it up from shared memory, publishes its own end
// state -- one FMA later, so the serial chain per batch is a shared-memory hop instead of a memory round trip plus U dependent
// FMAs -- and fixes its U outputs up with one FMA each.  W batches per column are in flight, every element is still read and
// written exactly once, and nothing is recomputed.  (A shared-memory ring filled by cp.async.bulk -- one warp per 32 float4
// columns, 512-byte row pieces, up to 24 stages of 8 steps -- was measured as well: 71 % / 35 % of the HBM peak at B = 8 / 2
// against 77 % / 53 % for this kernel; many small bulk copies do not reach the memory-level parallelism of plain loads.)
template <int V, int U, int W>
__global__ void __launch_bounds__(32 * W) pscan_fwd_chain_kernel(PscanParams p) {
    using VT = typename Vec<V>::type;
    __shared__ VT s_carry[W][32];
    __shared__ int s_ready[W];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nvec = p.DN / V;
    const int64_t i = (int64_t)blockIdx.x * 32 + lane;
    const bool act = i < nvec;
    const int64_t ic = act ? i : nvec - 1;
    const int b = blockIdx.z;
    const VT *A = reinterpret_cast<const VT *>(p.A + (size_t)b * p.L * p.DN) + ic;
    const VT *X = reinterpret_cast<const VT *>(p.X + (size_t)b * p.L * p.DN) + ic;
    VT *H = reinterpret_cast<VT *>(p.Hout + (size_t)b * p.L * p.DN) + ic;
    if (lane == 0) s_ready[w] = -1;
    __syncthreads();
    const int nb = (p.L + U - 1) / U;
    const int wp = (w + W - 1) % W;
    volatile int *ready = s_ready;
    for (int k = w; k < nb; k += W) {
        const int tb = k * U;
        VT a[U], x[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int t = min(tb + j, p.L - 1);
            a[j] = __ldcs(A + (size_t)t * nvec);
            x[j] = __ldcs(X + (size_t)t * nvec);
        }
#pragma unroll
        for (int j = 1; j < U; ++j) {   // x[j] <- state after step j from a zero carry, a[j] <- a[0] ... a[j]
            x[j] = Vec<V>::fma(a[j], x[j - 1], x[j]);
            a[j] = Vec<V>::mul(a[j], a[j - 1]);
        }
        VT hin = Vec<V>::zero();
        if (k > 0) {
            while (ready[wp] != k - 1) { }
            __syncwarp();
            hin = ps_ld_shared(&s_carry[wp][lane]);
        }
        if (k + 1 < nb) {   // the end state of this batch, as early as possible
            ps_st_shared(&s_carry[w][lane], Vec<V>::fma(a[U - 1], hin, x[U - 1]));
            __syncwarp();
            if (lane == 0) { __threadfence_block(); ready[w] = k; }
        }
        if (act) {
#pragma unroll
            for (int j = 0; j < U; ++j)
                if (tb + j < p.L) __stcs(H + (size_t)(tb + j) * nvec, Vec<V>::fma(a[j], hin, x[j]));
        }
    }
}

// Reverse direction: gt[t] = dH[t] + A[t+1] gt[t+1], dX[t] = gt[t], dA[t] = H[t-1] gt[t]; the carry handed to the earlier batch
// is G = A[tb] gt[tb].  Within a batch gt[j] = gl[j] + Q[j] G_in with gl the local scan and Q[j] = A[j+1] ... A[U-1].
template <int V, int U, int W>
__global__ void __launch_bounds__(32 * W) pscan_bwd_chain_kernel(PscanParams p) {
    using VT = typename Vec<V>::type;
    __shared__ VT s_carry[W][32];
    __shared__ int s_ready[W];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nvec = p.DN / V;
    const int64_t i = (int64_t)blockIdx.x * 32 + lane;
    const bool act = i < nvec;
    const int64_t ic = act ? i : nvec - 1;
    const int b = blockIdx.z;
    const VT *A = reinterpret_cast<const VT *>(p.A + (size_t)b * p.L * p.DN) + ic;
    const VT *dH = reinterpret_cast<const VT *>(p.dH + (size_t)b * p.L * p.DN) + ic;
    const VT *H = reinterpret_cast<const VT *>(p.H + (size_t)b * p.L * p.DN) + ic;
    VT *dA = reinterpret_cast<VT *>(p.dA + (size_t)b * p.L * p.DN) + ic;
    VT *dX = reinterpret_cast<VT *>(p.dX + (size_t)b * p.L * p.DN) + ic;
    if (lane == 0) s_ready[w] = -1;
    __syncthreads();
    const int nb = (p.L + U - 1) / U;
    const int wp = (w + W - 1) % W;
    volatile int *ready = s_ready;
    for (int k = w; k < nb; k += W) {   // k-th batch in processing order = batch nb - 1 - k of the sequence
        const int tb = (nb - 1 - k) * U;
        VT a[U], g[U], hp[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int t = min(tb + j, p.L - 1);
            a[j] = __ldcs(A + (size_t)t * nvec);
            g[j] = tb + j < p.L ? __ldcs(dH + (size_t)t * nvec) : Vec<V>::zero();   // steps past the end contribute nothing
            hp[j] = t > 0 ? __ldcs(H + (size_t)(t - 1) * nvec) : Vec<V>::zero();
        }
        // g[j] <- local gt[j]; a[j + 1] <- Q[j] = a[j + 1] ... a[U - 1] (Q[U - 1] = 1 stays implicit); a[0] is kept for the carry
        VT q = Vec<V>::one();
#pragma unroll
        for (int j = U - 2; j >= 0; --j) {
            g[j] = Vec<V>::fma(a[j + 1], g[j + 1], g[j]);
            q = Vec<V>::mul(q, a[j + 1]);
            a[j + 1] = q;
        }
        VT gin = Vec<V>::zero();
        if (k > 0) {
            while (ready[wp] != k - 1) { }
            __syncwarp();
            gin = ps_ld_shared(&s_carry[wp][lane]);
        }
        if (k + 1 < nb) {   // G handed to the earlier batch: a[0] (gl[0] + Q[0] G_in)
            const VT q0 = U > 1 ? a[1] : Vec<V>::one();
            ps_st_shared(&s_carry[w][lane], Vec<V>::mul(a[0], Vec<V>::fma(q0, gin, g[0])));
            __syncwarp();
            if (lane == 0) { __threadfence_block(); ready[w] = k; }
        }
        if (act) {
#pragma unroll
            for (int j = 0; j < U; ++j) {
                if (tb + j < p.L) {
                    const VT gt = j + 1 < U ? Vec<V>::fma(a[j + 1], gin, g[j]) : Vec<V>::add(g[j], gin);
                    __stcs(dX + (size_t)(tb + j) * nvec, gt);
                    __stcs(dA + (size_t)(tb + j) * nvec, Vec<V>::mul(hp[j], gt));
                }
            }
        }
    }
}

// warps per CTA of the warp-chained kernels (batches in flight per column): forward 8, backward 4 (4 / 8 / 16 forward against
// 8 / 4 / 2 backward measured on three shapes, profiles/r02_chain_variants.txt)
constexpr int kPsChainFW = 8;
constexpr int kPsChainBW = 4;
constexpr int kPsChainU = 8;
static bool pscan_use_chain(int L, int nseg) { return nseg == 1 && L >= 4 * kPsChainU; }

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int pscan_check(const void *a, const void *b, const void *c, int B, int L, int D, int N) {
    if (!a || !b || !c) { set_error("pscan: NULL pointer"); return GFE_ERR_ARG; }
    if (B <= 0 || L <= 0 || D <= 0 || N <= 0) { set_error("pscan: non-positive shape"); return GFE_ERR_ARG; }
    if (B > 65535) { set_error("pscan: batch %d exceeds grid limit", B); return GFE_ERR_UNSUPPORTED; }
    return GFE_OK;
}

}  // namespace gfe

extern "C" {

GFE_API size_t gfe_pscan_workspace_bytes(int B, int L, int D, int N) {
    if (B <= 0 || L <= 0 || D <= 0 || N <= 0) return 0;
    const int64_t DN = (int64_t)D * N;
    const gfe::PscanPlan pl = gfe::pscan_plan(B, L, DN, 2);   // the forward plan never has fewer segments than the backward plan
    if (pl.nseg <= 1) return 0;
    return 2 * gfe::align_up((size_t)B * pl.nseg * DN * sizeof(float), 256);
}

GFE_API int gfe_pscan_fwd(const float *A, const float *X, float *H, int B, int L, int D, int N,
                          void *ws, size_t ws_bytes, void *stream) {
    using namespace gfe;
    int rc = pscan_check(A, X, H, B, L, D, N);
    if (rc != GFE_OK) return rc;
    const int64_t DN = (int64_t)D * N;
    const PscanPlan pl = pscan_plan(B, L, DN, 2);
    const size_t need = gfe_pscan_workspace_bytes(B, L, D, N);
    if (need > 0 && (ws == nullptr || ws_bytes < need)) { set_error("pscan_fwd: workspace too small (%zu < %zu)", ws ? ws_bytes : (size_t)0, need); return GFE_ERR_WORKSPACE; }
    PscanParams p{};
    p.A = A; p.X = X; p.Hout = H; p.B = B; p.L = L; p.DN = DN; p.nseg = pl.nseg; p.seg_len = pl.seg_len;
    p.segP = reinterpret_cast<float *>(ws);
    p.segS = reinterpret_cast<float *>(reinterpret_cast<char *>(ws) + need / 2);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const bool al = aligned16(A) && aligned16(X) && aligned16(H) && (need == 0 || aligned16(ws));
    // The plan only splits L once it has fallen to (1, 32), so the split runs the scalar kernels whatever the alignment;
    // otherwise (4, 16) when the operands allow it (rows of D*N fp32 keep 16-byte alignment when DN % 4 == 0)
    const int V = (al && pl.nseg == 1) ? pl.V : 1;
    const int64_t nvec = DN / V;
    const dim3 block(128), grid((unsigned)ceil_div64(nvec, 128), pl.nseg, B);
    if (pl.nseg > 1) {
        { ScopedKernelTimer tm(K_PSCAN_FWD_SUMMARY, st);
          pscan_fwd_kernel<1, 32, true><<<grid, block, 0, st>>>(p); }
        rc = check_launch("pscan_fwd_summary");
        if (rc != GFE_OK) return rc;
    }
    if (pscan_use_chain(L, pl.nseg)) {
        const int Vc = (al && DN % 4 == 0) ? 4 : 1;
        const dim3 gridc((unsigned)ceil_div64(DN / Vc, 32), 1, B);
        ScopedKernelTimer tm(K_PSCAN_FWD, st);
        if (Vc == 4) pscan_fwd_chain_kernel<4, kPsChainU, kPsChainFW><<<gridc, 32 * kPsChainFW, 0, st>>>(p);
        else pscan_fwd_chain_kernel<1, kPsChainU, kPsChainFW><<<gridc, 32 * kPsChainFW, 0, st>>>(p);
        return check_launch("pscan_fwd (chained)");
    }
    { ScopedKernelTimer tm(K_PSCAN_FWD, st);
      if (V == 4) pscan_fwd_kernel<4, 16, false><<<grid, block, 0, st>>>(p);
      else pscan_fwd_kernel<1, 32, false><<<grid, block, 0, st>>>(p); }
    return check_launch("pscan_fwd");
}

GFE_API int gfe_pscan_bwd(const float *A, const float *H, const float *dH, float *dA, float *dX,
                          int B, int L, int D, int N, void *ws, size_t ws_bytes, void *stream) {
    using namespace gfe;
    int rc = pscan_check(A, H, dH, B, L, D, N);
    if (rc != GFE_OK) return rc;
    if (!dA || !dX) { set_error("pscan_bwd: NULL output pointer"); return GFE_ERR_ARG; }
    const int64_t DN = (int64_t)D * N;
    const PscanPlan pl = pscan_plan(B, L, DN, 3);
    const size_t need = gfe_pscan_workspace_bytes(B, L, D, N);
    if (need > 0 && (ws == nullptr || ws_bytes < need)) { set_error("pscan_bwd: workspace too small (%zu < %zu)", ws ? ws_bytes : (size_t)0, need); return GFE_ERR_WORKSPACE; }
    PscanParams p{};
    p.A = A; p.H = H; p.dH = dH; p.dA = dA; p.dX = dX; p.B = B; p.L = L; p.DN = DN; p.nseg = pl.nseg; p.seg_len = pl.seg_len;
    p.segP = reinterpret_cast<float *>(ws);
    p.segS = reinterpret_cast<float *>(reinterpret_cast<char *>(ws) + need / 2);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const bool al = aligned16(A) && aligned16(H) && aligned16(dH) && aligned16(dA) && aligned16(dX) && (need == 0 || aligned16(ws));
    const int V = (al && pl.nseg == 1) ? pl.V : 1;   // as forward: the L-split only follows the fall to (1, 32)
    const int64_t nvec = DN / V;
    const dim3 block(128);
    if (pl.nseg > 1) {
        const dim3 grid((unsigned)ceil_div64(nvec, 128), pl.nseg - 1, B);
        { ScopedKernelTimer tm(K_PSCAN_BWD_SUMMARY, st);
          pscan_bwd_kernel<1, 32, true><<<grid, block, 0, st>>>(p); }
        rc = check_launch("pscan_bwd_summary");
        if (rc != GFE_OK) return rc;
    }
    if (pscan_use_chain(L, pl.nseg)) {
        const int Vc = (al && DN % 4 == 0) ? 4 : 1;
        const dim3 gridc((unsigned)ceil_div64(DN / Vc, 32), 1, B);
        ScopedKernelTimer tm(K_PSCAN_BWD, st);
        if (Vc == 4) pscan_bwd_chain_kernel<4, kPsChainU, kPsChainBW><<<gridc, 32 * kPsChainBW, 0, st>>>(p);
        else pscan_bwd_chain_kernel<1, kPsChainU, kPsChainBW><<<gridc, 32 * kPsChainBW, 0, st>>>(p);
        return check_launch("pscan_bwd (chained)");
    }
    const dim3 grid((unsigned)ceil_div64(nvec, 128), pl.nseg, B);
    { ScopedKernelTimer tm(K_PSCAN_BWD, st);
      if (V == 4) pscan_bwd_kernel<4, 8, false><<<grid, block, 0, st>>>(p);
      else if (V == 2) pscan_bwd_kernel<2, 16, false><<<grid, block, 0, st>>>(p);
      else pscan_bwd_kernel<1, 32, false><<<grid, block, 0, st>>>(p); }
    return check_launch("pscan_bwd");
}

}  // extern "C"
