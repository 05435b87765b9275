// selscan_v4_fwd.cu -- fused selective-scan forward, "v4": two channels x four states per lane.
// Replaces mamba.py:255-256, 275-284, 220-222 of the reference (softplus -> discretise -> scan -> C.h -> D skip -> gate).
//
// What the profile of the first chained forward (one channel x four states per lane, profiles/r01_ab_*) said: it was bound by
// the shared-memory data pipe and by issue slots, not by HBM.  An LDS.128 costs ~2 pipe clocks whatever its address pattern
// (tools/microbench_lds.cu), so the number of LDS per state-step is what matters, and half of its instructions were spent
// outside the recurrence.  Here
//   * a lane owns the states 4q..4q+3 of TWO adjacent channels: the B and C quads it fetches feed eight state-steps
//     instead of four, and {delta, delta*u} of both channels arrive in one LDS.128 (no splatted copies: ptxas folds a
//     scalar operand of FFMA2/FMUL2 into the R.F32 broadcast form);
//   * a CTA of 128 threads serves 64 channels; every thread stages exactly one 16-byte piece per tile with offsets
//     computed once per unit, and the per-(t, channel pair) scalar work runs once per pair in the item mapping;
//   * per lane and step: 3 LDS.128 + 16 packed FP32 ops + 8 exp2 (every other step 2 of them on the FMA pipe) + 1 STS.64 for 8
//     state-steps (one channel per lane: 3 LDS.128 + 8 + 4 + 1 for 4); the slot loads run two steps ahead of their use;
//   * the item phases work on packed FP32 over the channel pair, slots are laid out in pair order {dl0, dl1, dl0 u0, dl1 u1},
//     rows are masked only in a ragged last chunk, paired stores are a compile-time property of the cp.async instantiation.
// Segments are chained (ChainSched) or independent (carries from selscan_seg.cu); checkpoints [b][t/8][c][16] (fp32, bf16 for bf16 activations) and the saved y are what
// selscan_chain_bwd.cu consumes.
#include <type_traits>

#include "common.cuh"
#include "selscan_shared.cuh"

namespace gfe {

// CPC = channels per CTA (64 or 32); 2 * CPC threads: lane (pair, quad) owns 2 channels x 4 states.
template <typename T, bool HAS_Z, int CPC>
struct FwdV4Smem {
    static constexpr int kV4CPC = CPC;
    static constexpr int kYPlane = CPC / 2 + 4;   // float2 per (t, quad) plane of the partial C.h: CPC / 2 pairs + 32 B skew (conflict-free STS.64)
    static constexpr int kStages = sizeof(T) == 4 ? 2 : 3;
    static constexpr int kNTile = HAS_Z ? 3 : 2;
    static constexpr int kTile = kChunk * kV4CPC * (int)sizeof(T);      // one of u, delta, z
    static constexpr int kBCRaw = kChunk * kNState * (int)sizeof(T);     // one of B, C
    static constexpr int kStage = kNTile * kTile + 2 * kBCRaw;
    static constexpr int kOffDD = kStages * kStage;                      // float2 [16][64] {dl, dl*u}
    static constexpr int kOffBC = kOffDD + kChunk * kV4CPC * 8;          // float4 [16][8]  B quads | C quads
    static constexpr int kOffY = kOffBC + kChunk * 8 * 16;               // float2 [16][4][36] partial C.h of a channel pair
    static constexpr int kTotal = kOffY + kChunk * 4 * kYPlane * 8;
};

// The 16 recurrence steps of one chunk, with the slot loads software-pipelined by hand: neither nvcc nor ptxas moves the
// three LDS of step j + 1 above the partial-sum STS of step j (may-alias shared addresses; __restrict__ does not reach
// ptxas), so in source order every step waited out a full LDS latency before its first FMUL2 (seen in the SASS).
template <int CPC, typename CK>
__device__ __forceinline__ void v4_recur_chunk(const float4 *__restrict__ dd_r, const float4 *__restrict__ bc_r,
                                               float2 *__restrict__ y_w, const float2 (&A2)[2][2], float2 (&h)[2][2],
                                               CK *__restrict__ ckq, size_t ck_step, int tb, int t1) {
    constexpr int kV4YPlane = CPC / 2 + 4;
    // slot loads are issued PF steps ahead of their use, BEFORE the stores of the steps between (1 / 2 / 3 / 4 steps measured on
    // cfg3 and cfg5: 2 within 1 % of the best on both, profiles/r02_chain_variants.txt)
    constexpr int PF = 2;
    float4 dd_q[PF + 1], B_q[PF + 1], C_q[PF + 1];
#pragma unroll
    for (int i = 0; i < PF; ++i) { dd_q[i] = dd_r[i * (CPC / 2)]; B_q[i] = bc_r[i * 8]; C_q[i] = bc_r[i * 8 + 4]; }
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
        if (j + PF < kChunk) {
            dd_q[PF] = dd_r[(j + PF) * (CPC / 2)];
            B_q[PF] = bc_r[(j + PF) * 8];
            C_q[PF] = bc_r[(j + PF) * 8 + 4];
        }
        if (j % kCkptV2 == 0 && ckq != nullptr && tb + j < t1) {   // states before step tb + j, for backward
            CK *dst = ckq + (size_t)((tb + j) / kCkptV2) * ck_step;
            ckpt_store(dst, make_float4(h[0][0].x, h[0][0].y, h[0][1].x, h[0][1].y));
            ckpt_store(dst + kNState, make_float4(h[1][0].x, h[1][0].y, h[1][1].x, h[1][1].y));
        }
        const float4 dd = dd_q[0], B4 = B_q[0], C4 = C_q[0];
#pragma unroll
        for (int i = 0; i < PF; ++i) { dd_q[i] = dd_q[i + 1]; B_q[i] = B_q[i + 1]; C_q[i] = C_q[i + 1]; }
        const float2 B01 = make_float2(B4.x, B4.y), B23 = make_float2(B4.z, B4.w);
        const float2 C01 = make_float2(C4.x, C4.y), C23 = make_float2(C4.z, C4.w);
        float yv[2];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            const float dl = ch ? dd.y : dd.x, du = ch ? dd.w : dd.z;
            const float2 x0 = fmul2(splat2(dl), A2[ch][0]), x1 = fmul2(splat2(dl), A2[ch][1]);
            // on odd steps one exp2 pair of 4 runs as a polynomial on the FMA pipe instead of MUFU.EX2 (0 / 1 / 2 pairs measured
            // on cfg3: 1 fastest, profiles/r02_chain_variants.txt)
            const float2 a0 = (ch == 0 && (j & 1)) ? ex2_poly2(x0) : ex2_2(x0);
            const float2 a1 = ex2_2(x1);
            h[ch][0] = ffma2(a0, h[ch][0], fmul2(splat2(du), B01));
            h[ch][1] = ffma2(a1, h[ch][1], fmul2(splat2(du), B23));
            const float2 y2 = ffma2(h[ch][1], C23, fmul2(h[ch][0], C01));
            yv[ch] = y2.x + y2.y;
        }
        y_w[j * (4 * kV4YPlane)] = make_float2(yv[0], yv[1]);
    }
}

#ifdef GFE_PHASE_CLOCKS   // development only: cycles per phase, summed over warp leaders (tools/dbg/phase_clocks.py)
__device__ unsigned long long g_fwd_phase_clk[8];
#define GFE_CLK(i) do { const long long now_ = clock64(); if ((threadIdx.x & 31) == 0) clk_acc[i] += now_ - clk_last; clk_last = now_; } while (0)
#else
#define GFE_CLK(i) do { } while (0)
#endif

template <typename T, bool HAS_Z, int CPB, int CPC>
__global__ void __launch_bounds__(2 * CPC, kFwdMinBlocks * (64 / CPC)) selscan_fwd_v4_kernel(ScanParams p, ChainSched cs) {
#ifdef GFE_PHASE_CLOCKS
    long long clk_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, clk_last = clock64();
#endif
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_unit;
    using SM = FwdV4Smem<T, HAS_Z, CPC>;
    constexpr int NT = 2 * CPC, NP = CPC / 2, NST = SM::kStages, NTILE = SM::kNTile;
    constexpr int kV4YPlane = SM::kYPlane;
    constexpr int RB = CPC * (int)sizeof(T);          // bytes per tile row
    constexpr int PPT = kChunk * RB / 16 / NT;        // 16-byte pieces per thread per activation tile (1 bf16, 2 fp32)
    constexpr int BCP = kChunk * kNState * (int)sizeof(T) / 16;   // pieces per B (or C) tile: 32 bf16, 64 fp32
    const int tid = threadIdx.x;
    const int rp = tid >> 2, rq = tid & 3;     // recurrence mapping: channel pair in block (0..31), state quad
    const int ip = tid % NP, ir = tid / NP;    // item mapping: channel pair, rows ir + 4 i

    float4 *sDD = reinterpret_cast<float4 *>(smem + SM::kOffDD);   // [t][pair] {dl0, dl0*u0, dl1, dl1*u1}
    float4 *sBC = reinterpret_cast<float4 *>(smem + SM::kOffBC);
    float2 *sY = reinterpret_cast<float2 *>(smem + SM::kOffY);
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    constexpr bool vec = CPB == 16;   // the cp.async instantiation also requires pair-aligned outputs (chain_launch_fwd)
    const int per_seg = p.B * cs.nblk;

    const float4 *dd_r = sDD + rp;
    const float4 *bc_r = sBC + rq;
    float2 *y_w = sY + rq * kV4YPlane + rp;

    // staging geometry of this thread (fixed): activation tiles and B|C tiles
    const int srow = (tid * PPT) / (RB / 16), spiece = (tid * PPT) % (RB / 16);   // PPT consecutive pieces of one row
    constexpr int BCI = (2 * BCP + NT - 1) / NT;   // B|C pieces per thread: piece i of this thread is tid + i * NT of [B pieces | C pieces]

    for (;;) {
        __syncthreads();   // every thread is done with the previous unit's shared memory
        if (tid == 0) s_unit = atomicAdd(cs.counter, 1);
        __syncthreads();
        const int unit = s_unit;
        if (unit >= cs.total) break;
        const int seg = unit / per_seg;
        const int rem = unit - seg * per_seg;
        const int b = rem / cs.nblk;
        const int c0 = (rem - b * cs.nblk) * CPC;
        const int t0 = seg * cs.seg_len, t1 = min(p.L, t0 + cs.seg_len);
        const int nch = (t1 - t0 + kChunk - 1) / kChunk;

        const T *ub = reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c0;
        const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c0;
        const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c0 : nullptr;
        const T *Bb = reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;
        const T *Cb = reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs;
        T *ob = reinterpret_cast<T *>(p.out) + (int64_t)b * p.o_bs + c0 + 2 * ip;
        T *yb = p.ysave ? reinterpret_cast<T *>(p.ysave) + (int64_t)b * p.L * p.ED + c0 + 2 * ip : nullptr;
        // checkpoints [b][t / 8][c][16] fp32: this lane's quads of channels 2 rp and 2 rp + 1
        using CK = typename CkptOf<T>::type;
        CK *ckq = p.ckpt ? reinterpret_cast<CK *>(p.ckpt) + ((size_t)b * p.nchunks * p.ED + c0 + 2 * rp) * kNState + 4 * rq : nullptr;
        const size_t ck_step = (size_t)p.ED * kNState;   // elements between consecutive checkpoints

        // per-thread source pointers of the staged pieces of the NEXT chunk to issue (chunks are issued strictly in order)
        const char *su = nullptr, *sd = nullptr, *sz = nullptr, *sbc[BCI];
        int bcrow[BCI];
        if constexpr (CPB == 16) {
            su = reinterpret_cast<const char *>(ub + (int64_t)(t0 + srow) * p.u_rs) + spiece * 16;
            sd = reinterpret_cast<const char *>(db + (int64_t)(t0 + srow) * p.d_rs) + spiece * 16;
            if (HAS_Z) sz = reinterpret_cast<const char *>(zb + (int64_t)(t0 + srow) * p.z_rs) + spiece * 16;
#pragma unroll
            for (int i = 0; i < BCI; ++i) {
                const int pc = tid + i * NT;                    // < 2 * BCP checked at issue time
                const int sel = pc / BCP, within = pc % BCP;    // 0: B, 1: C
                bcrow[i] = within / (BCP / kChunk);
                const int64_t rs = sel ? p.C_rs : p.B_rs;
                sbc[i] = reinterpret_cast<const char *>((sel ? Cb : Bb) + (int64_t)(t0 + bcrow[i]) * rs) + (within % (BCP / kChunk)) * 16;
            }
        }
        const uint32_t dst_act = smem_u32(smem) + srow * RB + spiece * 16;
        const uint32_t dst_bc = smem_u32(smem) + NTILE * SM::kTile + tid * 16;   // the raw B tile is followed by the raw C tile

        auto issue = [&](int k, int stage) {   // chunk k of this segment -> stage k % NST
            if (k < nch) {
                const int tb = t0 + k * kChunk;
                const int nrows = min(kChunk, t1 - tb);
                const uint32_t so = stage * SM::kStage;
                if constexpr (CPB == 16) {
                    if (srow < nrows) {
#pragma unroll
                        for (int i = 0; i < PPT; ++i) {
                            cp_async16(dst_act + so + i * 16, su + i * 16);
                            cp_async16(dst_act + so + SM::kTile + i * 16, sd + i * 16);
                            if (HAS_Z) cp_async16(dst_act + so + 2 * SM::kTile + i * 16, sz + i * 16);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < BCI; ++i)
                        if (tid + i * NT < 2 * BCP && bcrow[i] < nrows) cp_async16(dst_bc + so + i * NT * 16, sbc[i]);
                    constexpr int64_t sz_t = (int64_t)sizeof(T) * kChunk;
                    su += p.u_rs * sz_t; sd += p.d_rs * sz_t;
                    if (HAS_Z) sz += p.z_rs * sz_t;
#pragma unroll
                    for (int i = 0; i < BCI; ++i) sbc[i] += ((tid + i * NT) / BCP ? p.C_rs : p.B_rs) * sz_t;
                } else {
                    unsigned char *s = smem + so;
                    stage_tile<T, CPC, NT>(s, ub + (int64_t)tb * p.u_rs, p.u_rs, nrows, tid);
                    stage_tile<T, CPC, NT>(s + SM::kTile, db + (int64_t)tb * p.d_rs, p.d_rs, nrows, tid);
                    if (HAS_Z) stage_tile<T, CPC, NT>(s + 2 * SM::kTile, zb + (int64_t)tb * p.z_rs, p.z_rs, nrows, tid);
                    stage_tile<T, kNState, NT>(s + NTILE * SM::kTile, Bb + (int64_t)tb * p.B_rs, p.B_rs, nrows, tid);
                    stage_tile<T, kNState, NT>(s + NTILE * SM::kTile + SM::kBCRaw, Cb + (int64_t)tb * p.C_rs, p.C_rs, nrows, tid);
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int k = 0; k < NST; ++k) issue(k, k);

        // per-thread constants: A of both channels (recurrence mapping), D and bias (item mapping)
        float2 A2[2][2], h[2][2];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(p.A_log + (size_t)(c0 + 2 * rp + ch) * kNState) + rq);
            A2[ch][0] = make_float2(-expf(v.x) * kLog2e, -expf(v.y) * kLog2e);
            A2[ch][1] = make_float2(-expf(v.z) * kLog2e, -expf(v.w) * kLog2e);
        }
        const float2 Dc = __ldg(reinterpret_cast<const float2 *>(p.D + c0) + ip);
        const float2 bias = p.dt_bias ? __ldg(reinterpret_cast<const float2 *>(p.dt_bias + c0) + ip) : make_float2(0.f, 0.f);

        // carry-in: the state our predecessor segment left behind
        float *carry = cs.independent ? cs.segc + (((size_t)(seg > 0 ? seg - 1 : 0) * p.B + b) * p.ED + c0 + 2 * rp) * kNState + 4 * rq
                                      : cs.carry + ((size_t)b * p.ED + c0 + 2 * rp) * kNState + 4 * rq;
        if (seg > 0) {
            if (!cs.independent) {
                if (tid == 0) {
                    const int *f = cs.flags + (unit - per_seg);
                    while (ld_acquire(f) == 0) __nanosleep(100);
                }
                __syncthreads();
            }
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                const float4 v = __ldcg(reinterpret_cast<const float4 *>(carry + ch * kNState));
                h[ch][0] = make_float2(v.x, v.y);
                h[ch][1] = make_float2(v.z, v.w);
            }
        } else if (p.h0 != nullptr) {   // the caller's state before token 0, in the lane layout of the last_state store below
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(p.h0 + ((size_t)b * p.ED + c0 + 2 * rp + ch) * kNState) + rq);
                h[ch][0] = make_float2(v.x, v.y);
                h[ch][1] = make_float2(v.z, v.w);
            }
        } else {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) h[ch][0] = h[ch][1] = make_float2(0.f, 0.f);
        }

        float2 Du[4], gate[4];
        // FULL: all 16 rows of the chunk lie inside the sequence (every chunk but a ragged last one): no row masking.
        auto phase_a = [&](int k, int stage, auto full_c) {   // per-(t, channel pair) scalars of chunk k -> shared slots; B|C rows -> fp32 quads
            constexpr bool FULL = decltype(full_c)::value;
            const int tb = t0 + k * kChunk;
            const unsigned char *s = smem + stage * SM::kStage;
            const T *sU = reinterpret_cast<const T *>(s);
            const T *sD = reinterpret_cast<const T *>(s + SM::kTile);
            const T *sZ = reinterpret_cast<const T *>(s + 2 * SM::kTile);
            const T *sBr = reinterpret_cast<const T *>(s + NTILE * SM::kTile);   // B rows then C rows
            float2 dl[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) dl[i] = fadd2(lds_pair(sD + (ir + 4 * i) * CPC, ip), bias);
            if (sp) {   // branch-free packed softplus (selscan_shared.cuh)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float2 sg2;
                    dl[i] = softplus_pair<false>(dl[i], sg2);
                }
            }
            float2 uq[4], zq[4];   // every load of the phase before its first store (an LDS is never moved above an STS)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                uq[i] = lds_pair(sU + (ir + 4 * i) * CPC, ip);
                if (HAS_Z) zq[i] = lds_pair(sZ + (ir + 4 * i) * CPC, ip);
            }
            constexpr int BCC = kChunk * 8 / NT;   // fp32 quads this thread converts (16 rows x 8 quads over the CTA)
            float4 bcv[BCC];
#pragma unroll
            for (int i = 0; i < BCC; ++i) {   // B|C rows -> fp32 quads: [t][B quads 0..3 | C quads 0..3]
                const int e = tid + i * NT, t = e >> 3, q8 = e & 7;
                bcv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (FULL || tb + t < t1) bcv[i] = lds_quad(sBr + (q8 < 4 ? 0 : kChunk * 16) + t * 16 + 4 * (q8 & 3));
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int t = ir + 4 * i;
                float2 u2 = uq[i], dl2 = dl[i];
                if (!FULL && tb + t >= t1) u2 = dl2 = make_float2(0.f, 0.f);   // padded step: a = 1, bx = 0
                const float2 dlu = fmul2(dl2, u2);
                sDD[t * NP + ip] = make_float4(dl2.x, dl2.y, dlu.x, dlu.y);
                Du[i] = fmul2(Dc, u2);
                if (HAS_Z) {
                    const float2 z2 = zq[i];
                    const float2 den = fadd2(ex2_2(fmul2(z2, splat2(-kLog2e))), splat2(1.0f));
                    gate[i] = fmul2(z2, make_float2(rcp_approx(den.x), rcp_approx(den.y)));
                }
            }
#pragma unroll
            for (int i = 0; i < BCC; ++i) sBC[tid + i * NT] = bcv[i];
        };
        auto phase_a_any = [&](int k, int stage) {
            if (t0 + (k + 1) * kChunk <= t1) phase_a(k, stage, std::true_type{});
            else phase_a(k, stage, std::false_type{});
        };

        GFE_CLK(0);   // unit set-up (incl. waiting for the predecessor segment)
        cp_async_wait<NST - 1>();
        __syncthreads();
        phase_a_any(0, 0);
        GFE_CLK(5);
        // running output pointers of this thread's item rows (row ir of the current chunk)
        T *op = ob + (int64_t)(t0 + ir) * p.o_rs;
        T *yp_g = yb != nullptr ? yb + (int64_t)(t0 + ir) * p.ED : nullptr;
        const int64_t o_step = 4 * p.o_rs, y_step = (int64_t)4 * p.ED;

        int stage = 0;   // k % NST
        for (int k = 0; k < nch; ++k) {
            const int tb = t0 + k * kChunk;
            __syncthreads();   // (1) slots of chunk k are complete
            GFE_CLK(1);
            v4_recur_chunk<CPC, CK>(dd_r, bc_r, y_w, A2, h, ckq, ck_step, tb, t1);   // 16 steps of this lane's 2 x 4 states
            GFE_CLK(2);
            cp_async_wait<NST - 2>();   // chunk k + 1 has landed (this thread's pieces)
            __syncthreads();            // (2) partial sums complete; chunk k + 1 visible; stage k % NST free
            GFE_CLK(3);
            issue(k + NST, stage);
            stage = stage + 1 == NST ? 0 : stage + 1;
            GFE_CLK(7);   // (debug build: the refill alone)

            // ---- per-(t, channel pair) epilogue of chunk k: sum the 4 quads, D skip, gate, store ----
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int t = ir + 4 * i;
                if (tb + t < t1) {
                    const float2 *yp = sY + (t * 4) * kV4YPlane + ip;
                    const float2 p0 = yp[0], p1 = yp[kV4YPlane], p2 = yp[2 * kV4YPlane], p3 = yp[3 * kV4YPlane];
                    float2 y2 = fadd2(fadd2(fadd2(p0, p1), fadd2(p2, p3)), Du[i]);
                    if (yp_g != nullptr) stg_pair<T>(yp_g, y2.x, y2.y, true);
                    if (HAS_Z) y2 = fmul2(y2, gate[i]);
                    stg_pair<T>(op, y2.x, y2.y, vec);
                }
                op += o_step;
                if (yp_g != nullptr) yp_g += y_step;
            }
            GFE_CLK(4);
            if (k + 1 < nch) phase_a_any(k + 1, stage);
            GFE_CLK(5);
        }

        // carry-out / final state
        if (seg == cs.nseg - 1) {
            if (p.last_state != nullptr) {
#pragma unroll
                for (int ch = 0; ch < 2; ++ch)
                    *(reinterpret_cast<float4 *>(p.last_state + ((size_t)b * p.ED + c0 + 2 * rp + ch) * kNState) + rq) =
                        make_float4(h[ch][0].x, h[ch][0].y, h[ch][1].x, h[ch][1].y);
            }
        } else if (!cs.independent) {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch)
                __stcg(reinterpret_cast<float4 *>(carry + ch * kNState), make_float4(h[ch][0].x, h[ch][0].y, h[ch][1].x, h[ch][1].y));
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release(cs.flags + unit, 1);
        }
        cp_async_wait<0>();
        GFE_CLK(6);
    }
#ifdef GFE_PHASE_CLOCKS
    if ((threadIdx.x & 31) == 0)
        for (int i = 0; i < 8; ++i) atomicAdd(&g_fwd_phase_clk[i], (unsigned long long)clk_acc[i]);
#endif
}

#ifdef GFE_PHASE_CLOCKS
extern "C" __attribute__((visibility("default"))) int gfe_debug_fwd_phase_clocks(unsigned long long *out, int reset) {
    if (out) cudaMemcpyFromSymbol(out, g_fwd_phase_clk, sizeof(g_fwd_phase_clk));
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_fwd_phase_clk, z, sizeof(z)); }
    return 0;
}
#endif

// ---------------------------------------------------------------------------------------------------- host
template <typename T, bool HAS_Z, int CPB, int CPC>
static void launch_fwd_v4_inst(const ScanParams &p, const ChainSched &cs, cudaStream_t st) {
    constexpr size_t smem = FwdV4Smem<T, HAS_Z, CPC>::kTotal;
    const int grid = persistent_grid<selscan_fwd_v4_kernel<T, HAS_Z, CPB, CPC>>(2 * CPC, smem, cs.total);
    selscan_fwd_v4_kernel<T, HAS_Z, CPB, CPC><<<grid, 2 * CPC, smem, st>>>(p, cs);
}

template <typename T, int CPC>
static void launch_fwd_v4_cpc(const ScanParams &p, const ChainSched &cs, bool has_z, int cpb, cudaStream_t st) {
    if (has_z) {
        if (cpb == 16) launch_fwd_v4_inst<T, true, 16, CPC>(p, cs, st);
        else launch_fwd_v4_inst<T, true, 0, CPC>(p, cs, st);
    } else {
        if (cpb == 16) launch_fwd_v4_inst<T, false, 16, CPC>(p, cs, st);
        else launch_fwd_v4_inst<T, false, 0, CPC>(p, cs, st);
    }
}

// called by the chained-kernel dispatch (selscan_chain_host.cu) with cpc = cs.nblk's channel-block width
template <typename T>
void v4_launch_fwd_kernel(const ScanParams &p, const ChainSched &cs, int cpc, bool has_z, int cpb, cudaStream_t st) {
    if (cpc == 64) launch_fwd_v4_cpc<T, 64>(p, cs, has_z, cpb, st);
    else launch_fwd_v4_cpc<T, 32>(p, cs, has_z, cpb, st);   // (16-channel blocks measured slower; not instantiated)
}
template void v4_launch_fwd_kernel<float>(const ScanParams &, const ChainSched &, int, bool, int, cudaStream_t);
template void v4_launch_fwd_kernel<__nv_bfloat16>(const ScanParams &, const ChainSched &, int, bool, int, cudaStream_t);
template void v4_launch_fwd_kernel<__half>(const ScanParams &, const ChainSched &, int, bool, int, cudaStream_t);

}  // namespace gfe
