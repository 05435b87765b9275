// selscan.cu -- fused selective scan, forward and backward, for sm_100a.
//
// Replaces MambaBlock.ssm / selective_scan (cross_atten/mamba.py:227-286) with the softplus+bias of
// mamba.py:255-256 and the silu(z) gate of mamba.py:220-222 fused in, without ever materialising the
// (B, L, ED, N) tensors the reference builds (mamba.py:275-280).
//
// Work decomposition (both directions)
//   lane  = one channel c of one batch row b; all N states of that channel (N = 16, 32 or 64, a template
//           argument of every kernel) live in the lane's registers as N / 2 float2 pairs so the recurrences run
//           as packed FFMA2/FMUL2;
//   warp  = 32 adjacent channels -> every global access is one coalesced 64/128-byte line per time step;
//   warps are fully independent (only __syncwarp), a CTA is just a scheduling container;
//   time  = chunks of kChunk = 16 steps.  Forward stores the state at every chunk start ("checkpoint",
//           4 N / 16 B per (t, c)); backward walks the chunks in reverse, re-derives the N states of a chunk
//           from its checkpoint, and keeps the 16-step history of ONE state pair at a time in registers
//           (state-pair-outer loop order), which is what makes a register-resident backward possible.
//   L-split: when B * ED / 32 warps cannot fill the GPU, L is cut into segments; a first cheap pass
//           computes each segment's (decay, local end state) summary and the main pass starts every
//           segment from the combined carry (plan_segments() in api.cu).  Same in reverse for backward.
//
// Cross-channel reductions (dB, dC are sums over ED): warp-transposed shuffle reduction (62 SHFL per
// 64 values), per-warp partial rows in the workspace, one small finalize kernel.  Parameter gradients
// (dA_log, dD, ddt_bias) are accumulated per lane over its whole segment, then reduced over (b, seg)
// by the second finalize kernel.  Everything is deterministic (no atomics).
#include "common.cuh"
#include "selscan_shared.cuh"

namespace gfe {


// Every kernel below is a template on the state size N in {16, 32, 64} (kernel-wide layout: lane = channel, all N states of
// the channel in the lane's registers as N / 2 float2 pairs).  Per time step a warp stages one B|C row of 2 N floats in
// shared memory, each lane 2 N / 32 of them.
template <int N> __host__ __device__ constexpr int bc_regs() { return 2 * N / 32; }            // B|C values one lane stages per step
template <int N> __host__ __device__ constexpr int row_regs() { return N > 32 ? N / 32 : 1; }  // B (or C) values one lane stages per step
template <int N> __host__ __device__ constexpr int row_stride() { return N > 32 ? N : 32; }    // shared row of the summaries' B (or C) tile
template <int N> __host__ __device__ constexpr int red_stride() { return 2 * N + 2; }          // padded row of the reduced dB|dC tile (bank-conflict free float2 writes)
__host__ __device__ constexpr int ilog2(int v) { return v <= 1 ? 0 : 1 + ilog2(v / 2); }

// lane stages element i = lane + 32 r of the B|C row (B[t][i] for i < N, C[t][i - N] otherwise) for the kChunk steps
// starting at tb: v[r * kChunk + j]
template <int N, typename T>
__device__ __forceinline__ void load_bc(float (&v)[kChunk * bc_regs<N>()], const T *Bb, const T *Cb, int64_t B_rs, int64_t C_rs,
                                        int tb, int t1, int lane) {
#pragma unroll
    for (int r = 0; r < bc_regs<N>(); ++r) {
        const int i = lane + 32 * r;
        const T *base = i < N ? Bb + i : Cb + (i - N);
        const int64_t rs = i < N ? B_rs : C_rs;
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const int t = tb + j;
            v[r * kChunk + j] = t < t1 ? to_f(__ldg(base + (int64_t)t * rs)) : 0.0f;
        }
    }
}

// one row of N values (B or C) for the kChunk steps starting at tb: lane stages element (lane mod N) + 32 r
template <int N, typename T>
__device__ __forceinline__ void load_row(float (&v)[kChunk * row_regs<N>()], const T *row, int64_t rs, int tb, int t1, int lane) {
#pragma unroll
    for (int r = 0; r < row_regs<N>(); ++r) {
        const T *base = row + (N < 32 ? (lane & (N - 1)) : lane) + 32 * r;
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const int t = tb + j;
            v[r * kChunk + j] = t < t1 ? to_f(__ldg(base + (int64_t)t * rs)) : 0.0f;
        }
    }
}

// lanes < N write their staged row values to a shared tile of row_stride<N>() floats per step
template <int N>
__device__ __forceinline__ void store_row(float *tile, const float (&v)[kChunk * row_regs<N>()], int lane) {
    if (lane < N) {
#pragma unroll
        for (int r = 0; r < row_regs<N>(); ++r) {
#pragma unroll
            for (int j = 0; j < kChunk; ++j) tile[j * row_stride<N>() + 32 * r + lane] = v[r * kChunk + j];
        }
    }
}

template <int N>
__device__ __forceinline__ void load_A2(float2 (&A2)[N / 2], const float *A_log, int c) {
    const float4 *row = reinterpret_cast<const float4 *>(A_log + (size_t)c * N);
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
        const float4 v = __ldg(row + q);
        A2[2 * q] = make_float2(-expf(v.x) * kLog2e, -expf(v.y) * kLog2e);
        A2[2 * q + 1] = make_float2(-expf(v.z) * kLog2e, -expf(v.w) * kLog2e);
    }
}

// The exp2 coefficients A2 = -exp(A_log) log2(e) of a lane's channel: in registers for N <= 32; for N = 64 in per-lane
// shared slots (one float2 per (pair, lane), read back by the lane that wrote it), since h and A2 together would take 128
// of the 255 registers and the kernels would spill.
template <int N> __host__ __device__ constexpr bool decay_in_smem() { return N > 32; }
template <int N> __host__ __device__ constexpr int decay_smem_floats() { return decay_in_smem<N>() ? N * 32 : 0; }

template <int N, bool SMEM = decay_in_smem<N>()> struct Decay;
template <int N> struct Decay<N, false> {
    float2 r[N / 2];
    __device__ __forceinline__ void load(const float *A_log, int c, float2 *, int) { load_A2<N>(r, A_log, c); }
    __device__ __forceinline__ float2 operator[](int q) const { return r[q]; }
};
template <int N> struct Decay<N, true> {
    const float2 *s;
    __device__ __forceinline__ void load(const float *A_log, int c, float2 *slots, int lane) {
        const float4 *row = reinterpret_cast<const float4 *>(A_log + (size_t)c * N);
#pragma unroll
        for (int q = 0; q < N / 4; ++q) {
            const float4 v = __ldg(row + q);
            slots[(2 * q) * 32 + lane] = make_float2(-expf(v.x) * kLog2e, -expf(v.y) * kLog2e);
            slots[(2 * q + 1) * 32 + lane] = make_float2(-expf(v.z) * kLog2e, -expf(v.w) * kLog2e);
        }
        s = slots + lane;
    }
    __device__ __forceinline__ float2 operator[](int q) const { return s[q * 32]; }
};

// per-warp shared memory (floats) of the summaries (B or C tile) and of the forward (double-buffered B|C tile), decay slots included
template <int N> __host__ __device__ constexpr int summary_smem_floats() { return kChunk * row_stride<N>() + decay_smem_floats<N>(); }
// (N = 64 adds per-lane slots of delta, u and z for the chunk's steps: its step loop is not unrolled, see selscan_fwd_kernel)
template <int N> __host__ __device__ constexpr int fwd_smem_floats() {
    return 2 * kChunk * 2 * N + decay_smem_floats<N>() + (decay_in_smem<N>() ? 3 * kChunk * 32 : 0);
}

// =====================================================================================================
// Forward
// =====================================================================================================

// Pass A (only when nseg > 1): segment-local end state from a zero start, and sum(delta) of the segment.
template <typename T, int N>
__global__ void __launch_bounds__(128) selscan_fwd_summary_kernel(ScanParams p) {
    constexpr int P = N / 2;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + warp;
    if (g * 32 >= p.ED) return;
    const int c_raw = g * 32 + lane;
    const bool active = c_raw < p.ED;
    const int c = active ? c_raw : p.ED - 1;
    const int seg = blockIdx.y, b = blockIdx.z;
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);
    float *sBC = smem + warp * summary_smem_floats<N>();
    float2 *sA2 = reinterpret_cast<float2 *>(sBC + kChunk * row_stride<N>());

    const T *ub = reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c;
    const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c;
    const T *Bb = reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    const float bias = p.dt_bias ? __ldg(p.dt_bias + c) : 0.0f;

    Decay<N> A2;
    float2 h[P];
    A2.load(p.A_log, c, sA2, lane);
#pragma unroll
    for (int q = 0; q < P; ++q) h[q] = make_float2(0.f, 0.f);
    float sd = 0.0f;

    for (int tb = t0; tb < t1; tb += kChunk) {
        float bc[kChunk * row_regs<N>()];
        load_row<N>(bc, Bb, p.B_rs, tb, t1, lane);   // only B is needed (N = 16: both half-warps load it)
        T ur[kChunk], dr[kChunk];
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const int t = min(tb + j, t1 - 1);
            ur[j] = ld_stream(ub + (int64_t)t * p.u_rs);
            dr[j] = ld_stream(db + (int64_t)t * p.d_rs);
        }
        __syncwarp();
        store_row<N>(sBC, bc, lane);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            float dl = 0.f, uj = 0.f;
            if (tb + j < t1) {
                dl = to_f(dr[j]) + bias;
                if (sp) dl = softplus_only(dl);
                uj = to_f(ur[j]);
            }
            sd += dl;
            const float2 dl2 = splat2(dl), du2 = splat2(dl * uj);
            const float4 *sb = reinterpret_cast<const float4 *>(sBC + j * row_stride<N>());
#pragma unroll
            for (int q = 0; q < N / 4; ++q) {
                const float4 Bq = sb[q];
                h[2 * q] = ffma2(ex2_2(fmul2(dl2, A2[2 * q])), h[2 * q], fmul2(du2, make_float2(Bq.x, Bq.y)));
                h[2 * q + 1] = ffma2(ex2_2(fmul2(dl2, A2[2 * q + 1])), h[2 * q + 1], fmul2(du2, make_float2(Bq.z, Bq.w)));
            }
        }
    }
    if (active) {
        float2 *dst = p.seg_h + ((size_t)(b * p.nseg + seg) * P) * p.ED + c;
#pragma unroll
        for (int q = 0; q < P; ++q) dst[(size_t)q * p.ED] = h[q];
        p.seg_sd[(size_t)(b * p.nseg + seg) * p.ED + c] = sd;
    }
}

// N = 16 prefetches: the next chunk's B|C, u, delta and z values are loaded into registers during the current chunk's
// math, and B|C go to the spare half of the double-buffered tile at the top of the next chunk.  N = 32 / 64 hold 2 N
// floats of state and decay per lane, next to which a prefetched chunk does not fit in 255 registers: they stage B|C into
// the tile at the top of each chunk, then load the chunk's u, delta and z, and let the other resident warps cover the
// load latency.
template <int N> __host__ __device__ constexpr bool bc_in_regs() { return N == 16; }

template <typename T, bool HAS_Z, int N>
__global__ void __launch_bounds__(128) selscan_fwd_kernel(ScanParams p) {
    constexpr int P = N / 2, NB = bc_regs<N>();
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + warp;
    if (g * 32 >= p.ED) return;   // warp-uniform; no block-level barrier is used anywhere
    const int c_raw = g * 32 + lane;
    const bool active = c_raw < p.ED;
    const int c = active ? c_raw : p.ED - 1;
    const int seg = blockIdx.y, b = blockIdx.z;
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);
    float *sBCw = smem + warp * fwd_smem_floats<N>();   // double buffered B|C tile
    float2 *sA2 = reinterpret_cast<float2 *>(sBCw + 2 * kChunk * 2 * N);
    float *sStep = sBCw + 2 * kChunk * 2 * N + decay_smem_floats<N>();   // N = 64: [delta | u | z][step][lane]

    const T *ub = reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c;
    const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c;
    const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c : nullptr;
    const T *Bb = reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;
    const T *Cb = reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs;
    T *ob = reinterpret_cast<T *>(p.out) + (int64_t)b * p.o_bs + c;
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    const float bias = p.dt_bias ? __ldg(p.dt_bias + c) : 0.0f;
    const float Dc = __ldg(p.D + c);

    Decay<N> A2;
    float2 h[P];
    A2.load(p.A_log, c, sA2, lane);
    if (p.h0 != nullptr) {   // the caller's state before token 0 (same layout as last_state)
        const float2 *src = reinterpret_cast<const float2 *>(p.h0 + ((size_t)b * p.ED + c) * N);
#pragma unroll
        for (int q = 0; q < P; ++q) h[q] = src[q];
    } else {
#pragma unroll
        for (int q = 0; q < P; ++q) h[q] = make_float2(0.f, 0.f);
    }

    // carry-in: combine the summaries of all earlier segments (exp of a delta prefix sum per state); the summaries are
    // zero-start locals, so a state h0 is carried through them like any other
#pragma unroll 4
    for (int s = 0; s < seg; ++s) {
        const float sd = p.seg_sd[(size_t)(b * p.nseg + s) * p.ED + c];
        const float2 *src = p.seg_h + ((size_t)(b * p.nseg + s) * P) * p.ED + c;
        const float2 sd2 = splat2(sd);
#pragma unroll
        for (int q = 0; q < P; ++q) h[q] = ffma2(ex2_2(fmul2(sd2, A2[q])), h[q], src[(size_t)q * p.ED]);
    }

    auto store_bc = [&](float *sBC, const float (&v)[kChunk * NB]) {
#pragma unroll
        for (int r = 0; r < NB; ++r) {
#pragma unroll
            for (int j = 0; j < kChunk; ++j) sBC[j * 2 * N + 32 * r + lane] = v[r * kChunk + j];
        }
    };
    T ur[kChunk], dr[kChunk], zr[kChunk];
    float bc[bc_in_regs<N>() ? kChunk * NB : 1];
    auto load_udz = [&](int tb) {
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const int t = min(tb + j, t1 - 1);
            ur[j] = ld_stream(ub + (int64_t)t * p.u_rs);
            dr[j] = ld_stream(db + (int64_t)t * p.d_rs);
            if (HAS_Z) zr[j] = ld_stream(zb + (int64_t)t * p.z_rs);
        }
    };
    auto load_chunk = [&](int tb) {   // N = 16 only
        if constexpr (bc_in_regs<N>()) load_bc<N>(bc, Bb, Cb, p.B_rs, p.C_rs, tb, t1, lane);
        load_udz(tb);
    };
    if constexpr (bc_in_regs<N>()) load_chunk(t0);

    int buf = 0;
    for (int tb = t0; tb < t1; tb += kChunk) {
        float *sBC = sBCw + buf * (kChunk * 2 * N);
        if constexpr (bc_in_regs<N>()) {
            store_bc(sBC, bc);
        } else {
            float v[kChunk * NB];
            load_bc<N>(v, Bb, Cb, p.B_rs, p.C_rs, tb, t1, lane);
            store_bc(sBC, v);
        }
        __syncwarp();
        if constexpr (!bc_in_regs<N>()) load_udz(tb);

        if (p.ckpt != nullptr && active) {   // state at the start of this chunk, for backward
            float2 *dst = p.ckpt + ((size_t)(b * p.nchunks + tb / kChunk) * P) * p.ED + c;
#pragma unroll
            for (int q = 0; q < P; ++q) dst[(size_t)q * p.ED] = h[q];
        }

        T uc[kChunk], dc[kChunk], zc[kChunk];
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            uc[j] = ur[j];
            dc[j] = dr[j];
            if (HAS_Z) zc[j] = zr[j];
        }
        if constexpr (bc_in_regs<N>()) {
            if (tb + kChunk < t1) load_chunk(tb + kChunk);   // next chunk's loads fly during this chunk's math
        }

        if constexpr (decay_in_smem<N>()) {
            // N = 64: an unrolled step loop lets the scheduler hoist many steps' B|C reads (2 N floats each) next to the
            // N floats of state, and the kernel spills.  Each lane parks its steps' delta, u and z in its own shared slots
            // and walks the steps in a rolled loop.
#pragma unroll
            for (int j = 0; j < kChunk; ++j) {
                float dl = 0.f, uj = 0.f;
                if (tb + j < t1) {
                    dl = to_f(dc[j]) + bias;
                    if (sp) dl = softplus_only(dl);
                    uj = to_f(uc[j]);
                }
                sStep[j * 32 + lane] = dl;
                sStep[(kChunk + j) * 32 + lane] = uj;
                if (HAS_Z) sStep[(2 * kChunk + j) * 32 + lane] = to_f(zc[j]);
            }
#pragma unroll 1
            for (int j = 0; j < kChunk; ++j) {
                const bool valid = tb + j < t1;
                const float dl = sStep[j * 32 + lane], uj = sStep[(kChunk + j) * 32 + lane];
                const float2 dl2 = splat2(dl), du2 = splat2(dl * uj);
                float2 y2 = make_float2(0.f, 0.f);
                const float4 *sb = reinterpret_cast<const float4 *>(sBC + j * 2 * N);
#pragma unroll
                for (int q = 0; q < N / 4; ++q) {
                    const float4 Bq = sb[q], Cq = sb[N / 4 + q];
                    h[2 * q] = ffma2(ex2_2(fmul2(dl2, A2[2 * q])), h[2 * q], fmul2(du2, make_float2(Bq.x, Bq.y)));
                    y2 = ffma2(h[2 * q], make_float2(Cq.x, Cq.y), y2);
                    h[2 * q + 1] = ffma2(ex2_2(fmul2(dl2, A2[2 * q + 1])), h[2 * q + 1], fmul2(du2, make_float2(Bq.z, Bq.w)));
                    y2 = ffma2(h[2 * q + 1], make_float2(Cq.z, Cq.w), y2);
                }
                float y = fmaf(Dc, uj, y2.x + y2.y);
                if (HAS_Z) {
                    const float zj = sStep[(2 * kChunk + j) * 32 + lane];
                    y *= zj * sigmoid_fast(zj);
                }
                if (valid && active) st_stream(ob + (int64_t)(tb + j) * p.o_rs, from_f<T>(y));
            }
            buf ^= 1;
            continue;
        }

#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const bool valid = tb + j < t1;   // warp-uniform; padded steps leave h untouched (a = 1, bx = 0)
            float dl = 0.f, uj = 0.f;
            if (valid) {
                dl = to_f(dc[j]) + bias;
                if (sp) dl = softplus_only(dl);
                uj = to_f(uc[j]);
            }
            const float2 dl2 = splat2(dl), du2 = splat2(dl * uj);
            float2 y2 = make_float2(0.f, 0.f);
            const float4 *sb = reinterpret_cast<const float4 *>(sBC + j * 2 * N);
#pragma unroll
            for (int q = 0; q < N / 4; ++q) {
                const float4 Bq = sb[q], Cq = sb[N / 4 + q];
                h[2 * q] = ffma2(ex2_2(fmul2(dl2, A2[2 * q])), h[2 * q], fmul2(du2, make_float2(Bq.x, Bq.y)));
                y2 = ffma2(h[2 * q], make_float2(Cq.x, Cq.y), y2);
                h[2 * q + 1] = ffma2(ex2_2(fmul2(dl2, A2[2 * q + 1])), h[2 * q + 1], fmul2(du2, make_float2(Bq.z, Bq.w)));
                y2 = ffma2(h[2 * q + 1], make_float2(Cq.z, Cq.w), y2);
            }
            float y = fmaf(Dc, uj, y2.x + y2.y);
            if (HAS_Z) {
                const float zj = to_f(zc[j]);
                y *= zj * sigmoid_fast(zj);
            }
            if (valid && active) st_stream(ob + (int64_t)(tb + j) * p.o_rs, from_f<T>(y));
        }
        buf ^= 1;
    }

    if (p.last_state != nullptr && seg == p.nseg - 1 && active) {
        float2 *dst = reinterpret_cast<float2 *>(p.last_state + ((size_t)b * p.ED + c) * N);
#pragma unroll
        for (int q = 0; q < P; ++q) dst[q] = h[q];
    }
}

// =====================================================================================================
// Backward
// =====================================================================================================

// Reduce 64 per-lane values across the 32 lanes of a warp; lane l ends with the totals of values
// 2l and 2l+1.  31+... = 62 shuffles: each step exchanges half of the remaining values.
template <int HALF>
__device__ __forceinline__ void transpose_reduce_step(float *v, int lane) {
    const bool up = (lane & (HALF / 2)) != 0;
#pragma unroll
    for (int i = 0; i < HALF; ++i) {
        const float a = v[i], b = v[i + HALF];
        const float send = up ? a : b;
        const float keep = up ? b : a;
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, HALF / 2);
    }
}

template <typename T, bool HAS_Z>
__device__ __forceinline__ void bwd_prep_step(float xraw, float uj, float zj, float doj, bool sp, bool valid,
                                              float &dl, float &dlu, float &dy, float &sg, float &f) {
    if (!valid) {
        dl = dlu = dy = f = 0.f;
        sg = 0.f;
        return;
    }
    if (sp) {
        dl = softplus_sig(xraw, sg);
    } else {
        dl = xraw;
        sg = 1.0f;
    }
    dlu = dl * uj;
    if (HAS_Z) {
        const float sz = sigmoid_fast(zj);
        dy = doj * (zj * sz);
        f = doj * sz * fmaf(zj, 1.0f - sz, 1.0f);   // dout * d silu(z)/dz ; dz = f * y
    } else {
        dy = doj;
        f = 0.f;
    }
}

// Pass A' (only when nseg > 1): reverse-scan carry a[t0]*g[t0] of a segment from a zero incoming carry,
// plus sum(delta) of the segment.
template <typename T, bool HAS_Z, int N>
__global__ void __launch_bounds__(128) selscan_bwd_summary_kernel(ScanParams p) {
    constexpr int P = N / 2;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + warp;
    if (g * 32 >= p.ED) return;
    const int c_raw = g * 32 + lane;
    const bool active = c_raw < p.ED;
    const int c = active ? c_raw : p.ED - 1;
    const int seg = blockIdx.y + 1, b = blockIdx.z;   // segment 0's carry-out is never needed
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);
    float *sBC = smem + warp * summary_smem_floats<N>();
    float2 *sA2 = reinterpret_cast<float2 *>(sBC + kChunk * row_stride<N>());

    const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c;
    const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c : nullptr;
    const T *gb = reinterpret_cast<const T *>(p.dout) + (int64_t)b * p.do_bs + c;
    const T *Cb = reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs;
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    const float bias = p.dt_bias ? __ldg(p.dt_bias + c) : 0.0f;

    Decay<N> A2;
    float2 G[P];
    A2.load(p.A_log, c, sA2, lane);
#pragma unroll
    for (int q = 0; q < P; ++q) G[q] = make_float2(0.f, 0.f);
    float sd = 0.0f;

    const int first_chunk = t0 / kChunk, last_chunk = (t1 - 1) / kChunk;
    for (int k = last_chunk; k >= first_chunk; --k) {
        const int tb = k * kChunk;
        float bc[kChunk * row_regs<N>()];
        load_row<N>(bc, Cb, p.C_rs, tb, t1, lane);
        T dr[kChunk], zr[kChunk], gr[kChunk];
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const int t = min(tb + j, t1 - 1);
            dr[j] = ld_stream(db + (int64_t)t * p.d_rs);
            gr[j] = ld_stream(gb + (int64_t)t * p.do_rs);
            if (HAS_Z) zr[j] = ld_stream(zb + (int64_t)t * p.z_rs);
        }
        __syncwarp();
        store_row<N>(sBC, bc, lane);
        __syncwarp();
#pragma unroll
        for (int j = kChunk - 1; j >= 0; --j) {
            float dl = 0.f, dy = 0.f;
            if (tb + j < t1 && active) {
                dl = to_f(dr[j]) + bias;
                if (sp) dl = softplus_only(dl);
                dy = to_f(gr[j]);
                if (HAS_Z) {
                    const float zj = to_f(zr[j]);
                    dy *= zj * sigmoid_fast(zj);
                }
            }
            sd += dl;
            const float2 dl2 = splat2(dl), dy2 = splat2(dy);
            const float4 *sc = reinterpret_cast<const float4 *>(sBC + j * row_stride<N>());
#pragma unroll
            for (int q = 0; q < N / 4; ++q) {
                const float4 Cq = sc[q];
                G[2 * q] = fmul2(ex2_2(fmul2(dl2, A2[2 * q])), ffma2(make_float2(Cq.x, Cq.y), dy2, G[2 * q]));
                G[2 * q + 1] = fmul2(ex2_2(fmul2(dl2, A2[2 * q + 1])), ffma2(make_float2(Cq.z, Cq.w), dy2, G[2 * q + 1]));
            }
        }
    }
    if (active) {
        float2 *dst = p.seg_h + ((size_t)(b * p.nseg + seg) * P) * p.ED + c;
#pragma unroll
        for (int q = 0; q < P; ++q) dst[(size_t)q * p.ED] = G[q];
        p.seg_sd[(size_t)(b * p.nseg + seg) * p.ED + c] = sd;
    }
}

// per-warp shared memory of the backward kernel (floats)
template <int N> struct BwdSmem {
    static constexpr int kBC = kChunk * 2 * N;                 // B|C tile
    static constexpr int kRed = kChunk * red_stride<N>();      // reduced dB|dC tile
    static constexpr int kPair = N / 2 * 32 * 2;               // one float2 per (pair, lane)
    static constexpr int kSlot = kChunk * 32;                  // one float per (step, lane)
    static constexpr int kFloats = kBC + kRed + 4 * kPair + 3 * kSlot;
};

template <typename T, bool HAS_Z, int N>
__global__ void __launch_bounds__(128) selscan_bwd_kernel(ScanParams p) {
    constexpr int P = N / 2, NB = bc_regs<N>(), RS = red_stride<N>();
    using SM = BwdSmem<N>;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + warp;
    if (g * 32 >= p.ED) return;
    const int c_raw = g * 32 + lane;
    const bool active = c_raw < p.ED;
    const int c = active ? c_raw : p.ED - 1;
    const int seg = blockIdx.y, b = blockIdx.z;
    const int t0 = seg * p.seg_len, t1 = min(p.L, t0 + p.seg_len);

    float *sw = smem + warp * SM::kFloats;
    float *sBC = sw;
    float *sRed = sBC + SM::kBC;
    float2 *sA = reinterpret_cast<float2 *>(sRed + SM::kRed);     // natural A = -exp(A_log)
    float2 *sG = sA + P * 32;                                     // reverse carry a[t+1] g[t+1]
    float2 *sdA = sG + P * 32;                                    // dA accumulators
    float2 *sH = sdA + P * 32;                                    // checkpointed state at the chunk start
    float *sU = reinterpret_cast<float *>(sH + P * 32);
    float *sF = sU + SM::kSlot;
    float *sSg = sF + SM::kSlot;

    const T *ub = reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c;
    const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c;
    const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c : nullptr;
    const T *gb = reinterpret_cast<const T *>(p.dout) + (int64_t)b * p.do_bs + c;
    const T *Bb = reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;
    const T *Cb = reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs;
    T *dub = reinterpret_cast<T *>(p.du) + (int64_t)b * p.du_bs + c;
    T *ddb = reinterpret_cast<T *>(p.ddelta) + (int64_t)b * p.dd_bs + c;
    T *dzb = HAS_Z ? reinterpret_cast<T *>(p.dz) + (int64_t)b * p.dz_bs + c : nullptr;
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    const float bias = p.dt_bias ? __ldg(p.dt_bias + c) : 0.0f;
    const float Dc = __ldg(p.D + c);

    // per-lane constants and carries
    {
        const float4 *row = reinterpret_cast<const float4 *>(p.A_log + (size_t)c * N);
#pragma unroll
        for (int q = 0; q < N / 4; ++q) {
            const float4 v = __ldg(row + q);
            sA[(2 * q) * 32 + lane] = make_float2(-expf(v.x), -expf(v.y));
            sA[(2 * q + 1) * 32 + lane] = make_float2(-expf(v.z), -expf(v.w));
        }
#pragma unroll
        for (int q = 0; q < P; ++q) {
            sG[q * 32 + lane] = make_float2(0.f, 0.f);
            sdA[q * 32 + lane] = make_float2(0.f, 0.f);
        }
        // carry-in from the later segments: G = P[s] * G + Gloc[s], s = nseg-1 .. seg+1 (N = 64: one segment's 32 pairs of
        // loads at a time, four would take the whole register file)
#pragma unroll(N > 32 ? 1 : 4)
        for (int s = p.nseg - 1; s > seg; --s) {
            const float sd = p.seg_sd[(size_t)(b * p.nseg + s) * p.ED + c];
            const float2 *src = p.seg_h + ((size_t)(b * p.nseg + s) * P) * p.ED + c;
            const float2 sd2 = splat2(sd * kLog2e);
#pragma unroll
            for (int q = 0; q < P; ++q)
                sG[q * 32 + lane] = ffma2(ex2_2(fmul2(sd2, sA[q * 32 + lane])), sG[q * 32 + lane], src[(size_t)q * p.ED]);
        }
    }
    float dD_acc = 0.f, dbias_acc = 0.f;

    const int first_chunk = t0 / kChunk, last_chunk = (t1 - 1) / kChunk;
    for (int k = last_chunk; k >= first_chunk; --k) {
        const int tb = k * kChunk;

        // ---- stage B|C, load and pre-process the 16 steps of this lane's channel ----
        float dl[kChunk], dlu[kChunk], dy[kChunk];
        if constexpr (N > 16) {   // B|C first: its 2 N values per lane are not held next to the chunk's other loads
            float bc[kChunk * NB];
            load_bc<N>(bc, Bb, Cb, p.B_rs, p.C_rs, tb, t1, lane);
            __syncwarp();   // previous chunk's readers of sBC / sRed are done
#pragma unroll
            for (int r = 0; r < NB; ++r) {
#pragma unroll
                for (int j = 0; j < kChunk; ++j) sBC[j * 2 * N + 32 * r + lane] = bc[r * kChunk + j];
            }
            __syncwarp();
        }
        if constexpr (N > 16) {   // this chunk's checkpoint -> per-lane shared slots, 8 pairs at a time
            const float2 *ck = p.ckpt + ((size_t)(b * p.nchunks + k) * P) * p.ED + c;
#pragma unroll
            for (int q0 = 0; q0 < P; q0 += 8) {
                float2 hk[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) hk[q] = __ldcs(ck + (size_t)(q0 + q) * p.ED);
#pragma unroll
                for (int q = 0; q < 8; ++q) sH[(q0 + q) * 32 + lane] = hk[q];
            }
        }
        {
            float bc[N > 16 ? 1 : kChunk * NB];
            if constexpr (N == 16) load_bc<N>(bc, Bb, Cb, p.B_rs, p.C_rs, tb, t1, lane);
            T ur[kChunk], dr[kChunk], zr[kChunk], gr[kChunk];
#pragma unroll
            for (int j = 0; j < kChunk; ++j) {
                const int t = min(tb + j, t1 - 1);
                ur[j] = ld_stream(ub + (int64_t)t * p.u_rs);
                dr[j] = ld_stream(db + (int64_t)t * p.d_rs);
                gr[j] = ld_stream(gb + (int64_t)t * p.do_rs);
                if (HAS_Z) zr[j] = ld_stream(zb + (int64_t)t * p.z_rs);
            }
            if constexpr (N == 16) {   // this chunk's checkpoint -> per-lane shared slots (the pair loop below is not unrolled)
                const float2 *ck = p.ckpt + ((size_t)(b * p.nchunks + k) * P) * p.ED + c;
                float2 hk[P];
#pragma unroll
                for (int q = 0; q < P; ++q) hk[q] = __ldcs(ck + (size_t)q * p.ED);
#pragma unroll
                for (int q = 0; q < P; ++q) sH[q * 32 + lane] = hk[q];
            }
            if (k > first_chunk) {   // pull the next (earlier) chunk towards L2 while this one is processed
#pragma unroll
                for (int j = 0; j < kChunk; ++j) {
                    const int64_t t = tb - kChunk + j;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(ub + t * p.u_rs));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(db + t * p.d_rs));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(gb + t * p.do_rs));
                    if (HAS_Z) asm volatile("prefetch.global.L2 [%0];" ::"l"(zb + t * p.z_rs));
                }
            }
            __syncwarp();   // previous chunk's readers of sBC / sRed are done
            if constexpr (N == 16) {
#pragma unroll
                for (int j = 0; j < kChunk; ++j) sBC[j * 32 + lane] = bc[j];
            }
#pragma unroll
            for (int j = 0; j < kChunk; ++j) {
                const bool valid = (tb + j < t1) && active;
                const float uj = to_f(ur[j]);
                float sg, f;
                bwd_prep_step<T, HAS_Z>(to_f(dr[j]) + bias, uj, HAS_Z ? to_f(zr[j]) : 0.f, to_f(gr[j]), sp, valid,
                                        dl[j], dlu[j], dy[j], sg, f);
                sU[j * 32 + lane] = valid ? uj : 0.f;
                sF[j * 32 + lane] = f;
                sSg[j * 32 + lane] = sg;
            }
            __syncwarp();
        }

        float S1[kChunk], S2[kChunk], yv[kChunk];
#pragma unroll
        for (int j = 0; j < kChunk; ++j) S1[j] = S2[j] = yv[j] = 0.f;

        // ---- one state pair at a time: forward sweep (recompute), reverse sweep (gradients) ----
#pragma unroll 1
        for (int q = 0; q < P; ++q) {
            const float2 Aq = sA[q * 32 + lane];
            const float2 A2q = fmul2(Aq, splat2(kLog2e));
            float2 h = sH[q * 32 + lane];
            float2 a[kChunk], hp[kChunk];
#pragma unroll
            for (int j = 0; j < kChunk; ++j) {
                const float2 Bq = *reinterpret_cast<const float2 *>(sBC + j * 2 * N + 2 * q);
                const float2 Cq = *reinterpret_cast<const float2 *>(sBC + j * 2 * N + N + 2 * q);
                a[j] = ex2_2(fmul2(splat2(dl[j]), A2q));
                hp[j] = h;
                h = ffma2(a[j], h, fmul2(splat2(dlu[j]), Bq));
                yv[j] = fmaf(h.x, Cq.x, fmaf(h.y, Cq.y, yv[j]));
            }
            float2 G = sG[q * 32 + lane];
            float2 dA = sdA[q * 32 + lane];
            float v[64];   // [0,32): dB contributions (step-major, pair element minor); [32,64): dC
#pragma unroll
            for (int j = kChunk - 1; j >= 0; --j) {
                const float2 Bq = *reinterpret_cast<const float2 *>(sBC + j * 2 * N + 2 * q);
                const float2 Cq = *reinterpret_cast<const float2 *>(sBC + j * 2 * N + N + 2 * q);
                const float2 gg = ffma2(Cq, splat2(dy[j]), G);          // g[t] = C dy + a[t+1] g[t+1]
                const float2 dc = fmul2(splat2(dy[j]), h);              // dC_t[n] += dy * h[t]
                const float2 dbv = fmul2(gg, splat2(dlu[j]));           // dB_t[n] += g * delta * u
                v[2 * j] = dbv.x;
                v[2 * j + 1] = dbv.y;
                v[32 + 2 * j] = dc.x;
                v[32 + 2 * j + 1] = dc.y;
                S1[j] = fmaf(gg.x, Bq.x, fmaf(gg.y, Bq.y, S1[j]));      // sum_n g B
                G = fmul2(a[j], gg);                                    // a[t] g[t]
                const float2 t1v = fmul2(G, hp[j]);                     // g a h[t-1]  (= d a * a)
                S2[j] = fmaf(t1v.x, Aq.x, fmaf(t1v.y, Aq.y, S2[j]));    // sum_n (da a) A
                dA = ffma2(t1v, splat2(dl[j]), dA);                     // dA[c,n] += (da a) delta
                h = hp[j];
            }
            sG[q * 32 + lane] = G;
            sdA[q * 32 + lane] = dA;

            transpose_reduce_step<32>(v, lane);
            transpose_reduce_step<16>(v, lane);
            transpose_reduce_step<8>(v, lane);
            transpose_reduce_step<4>(v, lane);
            transpose_reduce_step<2>(v, lane);
            // lane l now owns values 2l, 2l+1: kind = l >> 4 (0: dB, 1: dC), step = l & 15, states 2q, 2q+1
            *reinterpret_cast<float2 *>(sRed + (lane & 15) * RS + (lane >> 4) * N + 2 * q) = make_float2(v[0], v[1]);
        }
        __syncwarp();

        // ---- per-warp partial rows of dB|dC (N > 16: after the outputs below, whose 5 x 16 per-step values are then dead) ----
        auto write_part_bc = [&]() {
            float *dst = p.part_bc + (((size_t)g * p.B + b) * p.L + tb) * (2 * N) + lane;
#pragma unroll
            for (int j = 0; j < kChunk; ++j)
                if (tb + j < t1) {
#pragma unroll
                    for (int r = 0; r < NB; ++r) dst[(size_t)j * (2 * N) + 32 * r] = sRed[j * RS + 32 * r + lane];
                }
        };
        if constexpr (N == 16) write_part_bc();

        // ---- per-(t, c) outputs ----
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            if (tb + j < t1 && active) {
                const float uj = sU[j * 32 + lane];
                const float ddl = fmaf(S1[j], uj, S2[j]);               // d delta
                const float draw = ddl * sSg[j * 32 + lane];            // through softplus
                st_stream(dub + (int64_t)(tb + j) * p.du_rs, from_f<T>(fmaf(dl[j], S1[j], Dc * dy[j])));
                st_stream(ddb + (int64_t)(tb + j) * p.dd_rs, from_f<T>(draw));
                if (HAS_Z) st_stream(dzb + (int64_t)(tb + j) * p.dz_rs, from_f<T>(sF[j * 32 + lane] * fmaf(Dc, uj, yv[j])));
                dD_acc = fmaf(dy[j], uj, dD_acc);
                dbias_acc += draw;
            }
        }
        if constexpr (N > 16) write_part_bc();
    }

    if (active) {
        float *dst = p.part_par + ((size_t)(b * p.nseg + seg) * (N + 2)) * p.ED + c;
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const float2 dA = sdA[q * 32 + lane];
            dst[(size_t)(2 * q) * p.ED] = dA.x;
            dst[(size_t)(2 * q + 1) * p.ED] = dA.y;
        }
        dst[(size_t)N * p.ED] = dD_acc;
        dst[(size_t)(N + 1) * p.ED] = dbias_acc;
    }
}

// dB|dC = sum over the G channel groups of the per-warp partial rows
template <typename T, int N>
__global__ void __launch_bounds__(256) selscan_bwd_finalize_bc_kernel(ScanParams p) {
    constexpr int W = 2 * N;   // one partial row: dB|dC of one token
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (row, n of the 2N)
    const int64_t rows = (int64_t)p.B * p.L;
    if (idx >= rows * W) return;
    const int64_t row = idx >> ilog2(W);
    const int n = (int)(idx & (W - 1));
    float acc = 0.f;
    const int64_t rbase = idx & ~(int64_t)(W - 1);
    const float *src = p.part_bc + (p.bc_interleaved ? rbase + 2 * (n & (N - 1)) + (n >> ilog2(N)) : idx);
    for (int g = 0; g < p.G; ++g) acc += __ldcs(src + (size_t)g * rows * W);
    const int64_t b = row / p.L, t = row % p.L;
    if (n < N)
        reinterpret_cast<T *>(p.dBm)[b * p.dB_bs + t * p.dB_rs + n] = from_f<T>(acc);
    else
        reinterpret_cast<T *>(p.dCm)[b * p.dC_bs + t * p.dC_rs + (n - N)] = from_f<T>(acc);
}

// dA_log = A * sum_{b,seg} dA ; dD, ddt_bias = sums
template <int N>
__global__ void __launch_bounds__(128) selscan_bwd_finalize_par_kernel(ScanParams p) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int q = blockIdx.y;   // 0..N+1
    if (c >= p.ED) return;
    float acc = 0.f;
    const int nbs = p.B * p.nseg;
    for (int i = 0; i < nbs; ++i) acc += p.part_par[((size_t)i * (N + 2) + q) * p.ED + c];
    if (q < N) {
        p.dA_log[(size_t)c * N + q] = acc * -expf(p.A_log[(size_t)c * N + q]);
    } else if (q == N) {
        p.dD[c] = acc;
    } else if (p.ddt_bias != nullptr) {
        p.ddt_bias[c] = acc;
    }
}

// =====================================================================================================
// Host side
// =====================================================================================================

struct WsLayout {
    size_t seg_h, seg_sd, part_bc, part_par, total;
};

static WsLayout fwd_ws_layout(int B, int L, int ED, int N, const SegPlan &sp) {
    WsLayout w{};
    size_t off = 0;
    w.seg_h = off;
    off += align_up(sp.nseg > 1 ? (size_t)B * sp.nseg * (N / 2) * ED * sizeof(float2) : 0, 256);
    w.seg_sd = off;
    off += align_up(sp.nseg > 1 ? (size_t)B * sp.nseg * ED * sizeof(float) : 0, 256);
    w.total = off;
    (void)L;
    return w;
}

static WsLayout bwd_ws_layout(int B, int L, int ED, int N, const SegPlan &sp) {
    WsLayout w = fwd_ws_layout(B, L, ED, N, sp);
    size_t off = w.total;
    const size_t G = (ED + 31) / 32;   // one dB|dC row (2 N floats) per warp (32 channels) and token
    w.part_bc = off;
    off += align_up(G * B * L * 2 * N * sizeof(float), 256);
    w.part_par = off;                  // dA[N] | dD | ddt_bias per (b, segment) and channel
    off += align_up((size_t)B * sp.nseg * (N + 2) * ED * sizeof(float), 256);
    w.total = off;
    return w;
}

static size_t ckpt_state_bytes(int B, int L, int ED, int N) {   // [b][chunk][pair][ED] float2
    const size_t nchunks = (L + kChunk - 1) / kChunk;
    return (size_t)B * nchunks * ED * N * sizeof(float);
}

static int validate_common(const gfe_selscan_args *a, bool bwd) {
    if (a == nullptr) { set_error("selscan: args is NULL"); return GFE_ERR_ARG; }
    if (a->batch <= 0 || a->seqlen <= 0 || a->d_inner <= 0) { set_error("selscan: non-positive shape"); return GFE_ERR_ARG; }
    if (!fused_d_state(a->d_state)) {
        set_error("selscan: d_state=%d unsupported by the fused kernel (compiled for 16, 32 and 64)", a->d_state);
        return GFE_ERR_UNSUPPORTED;
    }
    if (a->dtype != GFE_F32 && a->dtype != GFE_BF16 && a->dtype != GFE_F16) { set_error("selscan: bad dtype %d", a->dtype); return GFE_ERR_DTYPE; }
    if (!a->u || !a->delta || !a->Bm || !a->Cm || !a->A_log || !a->D) { set_error("selscan: NULL input pointer"); return GFE_ERR_ARG; }
    if ((reinterpret_cast<uintptr_t>(a->A_log) & 15) != 0) { set_error("selscan: A_log must be 16-byte aligned"); return GFE_ERR_ARG; }
    if (!bwd && !a->out) { set_error("selscan_fwd: out is NULL"); return GFE_ERR_ARG; }
    if (bwd) {
        if (!a->dout || !a->du || !a->ddelta || !a->dBm || !a->dCm || !a->dA_log || !a->dD) { set_error("selscan_bwd: NULL gradient pointer"); return GFE_ERR_ARG; }
        if ((a->z != nullptr) != (a->dz != nullptr)) { set_error("selscan_bwd: dz must be given iff z is"); return GFE_ERR_ARG; }
        if (!a->ckpt) { set_error("selscan_bwd: checkpoints from the forward pass are required"); return GFE_ERR_WORKSPACE; }
    }
    if (a->ckpt && a->ckpt_bytes < gfe_selscan_ckpt_bytes_dt(a->batch, a->seqlen, a->d_inner, a->d_state, a->dtype)) {
        set_error("selscan: checkpoint buffer too small (%zu < %zu)", a->ckpt_bytes,
                  gfe_selscan_ckpt_bytes_dt(a->batch, a->seqlen, a->d_inner, a->d_state, a->dtype));
        return GFE_ERR_WORKSPACE;
    }
    if (a->ckpt && (reinterpret_cast<uintptr_t>(a->ckpt) & 7) != 0) { set_error("selscan: ckpt must be 8-byte aligned"); return GFE_ERR_ARG; }
    return GFE_OK;
}

static void fill_common(ScanParams &p, const gfe_selscan_args *a, const SegPlan &sp) {
    p.B = a->batch; p.L = a->seqlen; p.ED = a->d_inner;
    p.nseg = sp.nseg; p.seg_len = sp.seg_len; p.nchunks = sp.nchunks;
    p.flags = a->flags;
    p.u = a->u; p.delta = a->delta; p.z = a->z; p.Bm = a->Bm; p.Cm = a->Cm;
    p.u_bs = a->u_bs; p.u_rs = a->u_rs; p.d_bs = a->delta_bs; p.d_rs = a->delta_rs;
    p.z_bs = a->z_bs; p.z_rs = a->z_rs; p.B_bs = a->B_bs; p.B_rs = a->B_rs; p.C_bs = a->C_bs; p.C_rs = a->C_rs;
    p.A_log = a->A_log; p.D = a->D; p.dt_bias = a->dt_bias;
    p.ckpt = reinterpret_cast<float2 *>(a->ckpt);
    p.ysave = a->ckpt ? reinterpret_cast<char *>(a->ckpt) + ckpt_state_bytes(a->batch, a->seqlen, a->d_inner, a->d_state) : nullptr;
    p.G = (a->d_inner + 31) / 32;
}

template <typename K>
static void launch_fast(K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, const ScanParams &p) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kernel<<<grid, block, smem, st>>>(p);
}

template <typename T, int N>
static int launch_fwd(const gfe_selscan_args *a, const float *h0, cudaStream_t st) {
    const SegPlan sp = plan_segments(a->batch, a->seqlen, a->d_inner);
    const WsLayout wl = fwd_ws_layout(a->batch, a->seqlen, a->d_inner, N, sp);
    if (wl.total > 0 && (a->ws == nullptr || a->ws_bytes < wl.total)) {
        set_error("selscan_fwd: workspace too small (%zu < %zu)", a->ws ? a->ws_bytes : (size_t)0, wl.total);
        return GFE_ERR_WORKSPACE;
    }
    ScanParams p{};
    fill_common(p, a, sp);
    p.out = a->out; p.o_bs = a->out_bs; p.o_rs = a->out_rs; p.last_state = a->last_state; p.h0 = h0;
    char *ws = reinterpret_cast<char *>(a->ws);
    p.seg_h = reinterpret_cast<float2 *>(ws + wl.seg_h);
    p.seg_sd = reinterpret_cast<float *>(ws + wl.seg_sd);

    const dim3 block(32);   // one warp per CTA
    const dim3 grid(p.G, sp.nseg, a->batch);
    if (sp.nseg > 1) {
        { ScopedKernelTimer tm(K_SELSCAN_FWD_SUMMARY, st);
          selscan_fwd_summary_kernel<T, N><<<grid, block, summary_smem_floats<N>() * sizeof(float), st>>>(p); }
        int rc = check_launch("selscan_fwd_summary");
        if (rc != GFE_OK) return rc;
    }
    {
        const size_t smem = fwd_smem_floats<N>() * sizeof(float);
        ScopedKernelTimer tm(K_SELSCAN_FWD, st);
        if (a->z != nullptr) selscan_fwd_kernel<T, true, N><<<grid, block, smem, st>>>(p);
        else selscan_fwd_kernel<T, false, N><<<grid, block, smem, st>>>(p);
    }
    return check_launch("selscan_fwd");
}

template <typename T, int N>
static int launch_finalize_t(const gfe_selscan_args *a, ScanParams &p, cudaStream_t st);

template <typename T, bool HAS_Z, int N>
static int launch_bwd_z(const gfe_selscan_args *a, ScanParams &p, const SegPlan &sp, cudaStream_t st) {
    const dim3 block(32);   // one warp per CTA
    if (sp.nseg > 1) {
        const dim3 grid(p.G, sp.nseg - 1, a->batch);
        { ScopedKernelTimer tm(K_SELSCAN_BWD_SUMMARY, st);
          selscan_bwd_summary_kernel<T, HAS_Z, N><<<grid, block, summary_smem_floats<N>() * sizeof(float), st>>>(p); }
        int rc = check_launch("selscan_bwd_summary");
        if (rc != GFE_OK) return rc;
    }
    const dim3 grid(p.G, sp.nseg, a->batch);
    {
        const size_t smem = BwdSmem<N>::kFloats * sizeof(float);
        ScopedKernelTimer tm(K_SELSCAN_BWD, st);
        launch_fast(selscan_bwd_kernel<T, HAS_Z, N>, grid, block, smem, st, p);
    }
    int rc = check_launch("selscan_bwd");
    if (rc != GFE_OK) return rc;
    return launch_finalize_t<T, N>(a, p, st);
}

// dB|dC and parameter-gradient finalize kernels, shared with the chained backward (selscan_chain_bwd.cu)
template <typename T, int N>
static int launch_finalize_t(const gfe_selscan_args *a, ScanParams &p, cudaStream_t st) {
    const int64_t nbc = (int64_t)a->batch * a->seqlen * 2 * N;
    { ScopedKernelTimer tm(K_SELSCAN_BWD_FIN_BC, st);
      selscan_bwd_finalize_bc_kernel<T, N><<<(unsigned)ceil_div64(nbc, 256), 256, 0, st>>>(p); }
    int rc = check_launch("selscan_bwd_finalize_bc");
    if (rc != GFE_OK) return rc;
    { ScopedKernelTimer tm(K_SELSCAN_BWD_FIN_PAR, st);
      selscan_bwd_finalize_par_kernel<N><<<dim3((a->d_inner + 127) / 128, N + 2), 128, 0, st>>>(p); }
    return check_launch("selscan_bwd_finalize_par");
}

// (the chained backward serves d_state = kNState only)
void launch_bwd_finalize(const gfe_selscan_args *a, ScanParams &p, cudaStream_t st, int &rc) {
    switch (a->dtype) {
        case GFE_F32: rc = launch_finalize_t<float, kNState>(a, p, st); break;
        case GFE_BF16: rc = launch_finalize_t<__nv_bfloat16, kNState>(a, p, st); break;
        default: rc = launch_finalize_t<__half, kNState>(a, p, st); break;
    }
}

template <typename T, int N>
static int launch_bwd(const gfe_selscan_args *a, cudaStream_t st) {
    const SegPlan sp = plan_segments(a->batch, a->seqlen, a->d_inner);
    const WsLayout wl = bwd_ws_layout(a->batch, a->seqlen, a->d_inner, N, sp);
    if (a->ws == nullptr || a->ws_bytes < wl.total) {
        set_error("selscan_bwd: workspace too small (%zu < %zu)", a->ws ? a->ws_bytes : (size_t)0, wl.total);
        return GFE_ERR_WORKSPACE;
    }
    ScanParams p{};
    fill_common(p, a, sp);
    char *ws = reinterpret_cast<char *>(a->ws);
    p.seg_h = reinterpret_cast<float2 *>(ws + wl.seg_h);
    p.seg_sd = reinterpret_cast<float *>(ws + wl.seg_sd);
    p.part_bc = reinterpret_cast<float *>(ws + wl.part_bc);
    p.part_par = reinterpret_cast<float *>(ws + wl.part_par);
    p.dout = a->dout; p.do_bs = a->dout_bs; p.do_rs = a->dout_rs;
    p.du = a->du; p.du_bs = a->du_bs; p.du_rs = a->du_rs;
    p.ddelta = a->ddelta; p.dd_bs = a->ddelta_bs; p.dd_rs = a->ddelta_rs;
    p.dz = a->dz; p.dz_bs = a->dz_bs; p.dz_rs = a->dz_rs;
    p.dBm = a->dBm; p.dB_bs = a->dB_bs; p.dB_rs = a->dB_rs;
    p.dCm = a->dCm; p.dC_bs = a->dC_bs; p.dC_rs = a->dC_rs;
    p.dA_log = a->dA_log; p.dD = a->dD; p.ddt_bias = a->ddt_bias;
    if (a->z != nullptr) return launch_bwd_z<T, true, N>(a, p, sp, st);
    return launch_bwd_z<T, false, N>(a, p, sp, st);
}

// generic kernels by state size (validate_common has checked fused_d_state)
template <typename T>
static int launch_fwd_n(const gfe_selscan_args *a, const float *h0, cudaStream_t st) {
    switch (a->d_state) {
        case 16: return launch_fwd<T, 16>(a, h0, st);
        case 32: return launch_fwd<T, 32>(a, h0, st);
        default: return launch_fwd<T, 64>(a, h0, st);
    }
}

template <typename T>
static int launch_bwd_n(const gfe_selscan_args *a, cudaStream_t st) {
    switch (a->d_state) {
        case 16: return launch_bwd<T, 16>(a, st);
        case 32: return launch_bwd<T, 32>(a, st);
        default: return launch_bwd<T, 64>(a, st);
    }
}

// forward dispatch of gfe_selscan_fwd / gfe_selscan_fwd_state (arguments validated); h0 NULL = zero start
static int launch_fwd_any(const gfe_selscan_args *a, const float *h0, cudaStream_t st) {
    if (chain_applicable(a->batch, a->seqlen, a->d_inner, a->d_state)) return chain_launch_fwd(a, h0, st);
    switch (a->dtype) {
        case GFE_F32: return launch_fwd_n<float>(a, h0, st);
        case GFE_BF16: return launch_fwd_n<__nv_bfloat16>(a, h0, st);
        default: return launch_fwd_n<__half>(a, h0, st);
    }
}

}  // namespace gfe

extern "C" {

GFE_API size_t gfe_selscan_ckpt_bytes_dt(int B, int L, int ED, int N, int dtype) {
    if (B <= 0 || L <= 0 || ED <= 0 || !gfe::fused_d_state(N)) return 0;
    if (dtype != GFE_F32 && dtype != GFE_BF16 && dtype != GFE_F16) return 0;
    // segment-start states (fp32) + y before the gate in the activation dtype
    const size_t ybytes = (size_t)B * L * ED * (dtype == GFE_F32 ? 4 : 2);
    if (gfe::chain_applicable(B, L, ED, N)) return gfe::chain_ckpt_state_bytes(B, L, ED, dtype) + ybytes;
    return gfe::ckpt_state_bytes(B, L, ED, N) + ybytes;
}

GFE_API size_t gfe_selscan_ckpt_bytes(int B, int L, int ED, int N) {   // upper bound over the activation dtypes
    return gfe_selscan_ckpt_bytes_dt(B, L, ED, N, GFE_F32);
}

GFE_API size_t gfe_selscan_fwd_workspace_bytes(int B, int L, int ED, int N) {
    if (B <= 0 || L <= 0 || ED <= 0 || !gfe::fused_d_state(N)) return 0;
    if (gfe::chain_applicable(B, L, ED, N)) return gfe::chain_fwd_workspace_bytes(B, L, ED);
    return gfe::fwd_ws_layout(B, L, ED, N, gfe::plan_segments(B, L, ED)).total;
}

GFE_API size_t gfe_selscan_bwd_workspace_bytes(int B, int L, int ED, int N) {
    if (B <= 0 || L <= 0 || ED <= 0 || !gfe::fused_d_state(N)) return 0;
    if (gfe::chain_applicable(B, L, ED, N)) return gfe::chain_bwd_workspace_bytes(B, L, ED);
    return gfe::bwd_ws_layout(B, L, ED, N, gfe::plan_segments(B, L, ED)).total;
}

GFE_API int gfe_selscan_fwd(const gfe_selscan_args *a, void *stream) {
    int rc = gfe::validate_common(a, false);
    if (rc != GFE_OK) return rc;
    return gfe::launch_fwd_any(a, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

GFE_API int gfe_selscan_fwd_state(const gfe_selscan_args *a, const float *h0, void *stream) {
    if (a != nullptr && a->ckpt != nullptr) {
        gfe::set_error("selscan_fwd_state: ckpt must be NULL (a forward from a carried state has no backward)");
        return GFE_ERR_ARG;
    }
    int rc = gfe::validate_common(a, false);
    if (rc != GFE_OK) return rc;
    if (h0 != nullptr) {
        if ((reinterpret_cast<uintptr_t>(h0) & 15) != 0) { gfe::set_error("selscan_fwd_state: h0 must be 16-byte aligned"); return GFE_ERR_ARG; }
        const size_t n = (size_t)a->batch * a->d_inner * a->d_state;
        if (a->last_state != nullptr && a->last_state < h0 + n && h0 < a->last_state + n) {
            gfe::set_error("selscan_fwd_state: h0 and last_state overlap");
            return GFE_ERR_ARG;
        }
    }
    return gfe::launch_fwd_any(a, h0, reinterpret_cast<cudaStream_t>(stream));
}

GFE_API int gfe_selscan_bwd(const gfe_selscan_args *a, void *stream) {
    int rc = gfe::validate_common(a, true);
    if (rc != GFE_OK) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (gfe::chain_applicable(a->batch, a->seqlen, a->d_inner, a->d_state)) return gfe::chain_launch_bwd(a, st);
    switch (a->dtype) {
        case GFE_F32: return gfe::launch_bwd_n<float>(a, st);
        case GFE_BF16: return gfe::launch_bwd_n<__nv_bfloat16>(a, st);
        default: return gfe::launch_bwd_n<__half>(a, st);
    }
}

}  // extern "C"
