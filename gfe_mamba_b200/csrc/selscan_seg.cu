// selscan_seg.cu -- independent L-segments for the chained selective-scan kernels (small B * ED: one long sequence, the
// production shape B = 2, a channel shard of an N-GPU run).  Replaces, for those shapes, the same reference lines as the
// chained kernels (mamba.py:255-256, 275-284 and PScan.backward, pscan.py:189-224).
//
// When B * ED / 64 chains cannot fill the GPU, waiting on a predecessor segment (ChainSched) would leave most SMs idle.
// Instead every segment gets its carry-in BEFORE the main pass:
//   1. summary pass (this file): per (segment, batch row, channel block) the recurrence alone, from a zero carry -- forward
//      h = a h + delta u B (segments 0 .. S-2), reverse G = a (G + C dy) (segments S-1 .. 1) -- in the lane layout of the
//      chained kernels (two channels x four states per lane, item mapping through shared slots), plus sum(delta) of the
//      segment.  No C.h, no outputs, no checkpoints, no cross-lane reduction: 2 packed FP32 ops and 2 exp2 per state pair
//      and step; one exp2 pair of four runs as a polynomial on the FMA pipe, because this loop is MUFU-bound.
//   2. combine pass: carry[s + 1] = exp2(A sum_delta[s]) carry[s] + local[s] over the segments, as a two-level scan (32 runs of
//      up to 8 segments per (b, c, n) element, chained through shared memory); carry[0] is the caller's state h0 (forward from
//      a carried state, gfe_selscan_fwd_state / _fwd_carry) or zero; in reverse the chain starts from the gradient of the
//      final state, dlast (gfe_selscan_bwd_carry), or zero.
//   3. main pass: the chained kernels with ChainSched::independent = 1 (selscan_v4_fwd.cu, selscan_chain_bwd.cu).
#include "common.cuh"
#include "selscan_shared.cuh"

namespace gfe {

template <typename T, bool HAS_Z, int CPC>
struct SegSumSmem {
    static constexpr int kStages = 3;                                    // (2, 3 and 4 stages measure the same)
    static constexpr int kNTile = HAS_Z ? 3 : 2;                         // x (u forward | dout reverse), delta, [z]
    static constexpr int kTile = kChunk * CPC * (int)sizeof(T);
    static constexpr int kBCRaw = kChunk * kNState * (int)sizeof(T);     // B rows (forward) | C rows (reverse)
    static constexpr int kStage = kNTile * kTile + kBCRaw;
    static constexpr int kOffDD = kStages * kStage;                      // float4 [16][CPC / 2] {dl0, v0, dl1, v1}
    static constexpr int kOffBC = kOffDD + kChunk * (CPC / 2) * 16;      // float4 [16][4] state quads of B | C
    static constexpr int kTotal = kOffBC + kChunk * 4 * 16;
};

// REV = false: forward aggregate of segments 0 .. nseg-2 (slot = segment);  v = delta u,        h = a h + v B
// REV = true : reverse aggregate of segments 1 .. nseg-1 (slot = segment - 1);  v = dout silu(z), G = a (G + v C)
// SLOT0 = 0 with REV: every segment, slot = segment (the summary of a whole range, seg_launch_total)
template <typename T, bool HAS_Z, int CPB, int CPC, bool REV, int SLOT0 = REV ? 1 : 0>
__global__ void __launch_bounds__(2 * CPC, 4 * (64 / CPC)) selscan_seg_summary_kernel(ScanParams p, ChainSched cs) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_unit;
    using SM = SegSumSmem<T, HAS_Z, CPC>;
    constexpr int NT = 2 * CPC, NP = CPC / 2, NST = SM::kStages, NTILE = SM::kNTile;
    constexpr int RB = CPC * (int)sizeof(T);
    constexpr int PPT = kChunk * RB / 16 / NT;                    // 16-byte pieces per thread per activation tile
    constexpr int BCP = kChunk * kNState * (int)sizeof(T) / 16;   // pieces of the B (C) tile: 32 (16-bit) / 64 (fp32) <= NT
    const int tid = threadIdx.x;
    const int rp = tid >> 2, rq = tid & 3;     // recurrence mapping: channel pair in block, state quad
    const int ip = tid % NP, ir = tid / NP;    // item mapping: channel pair, rows ir + 4 i

    float4 *sDD = reinterpret_cast<float4 *>(smem + SM::kOffDD);
    float4 *sBC = reinterpret_cast<float4 *>(smem + SM::kOffBC);
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    const int per_seg = p.B * cs.nblk;
    const float4 *dd_r = sDD + rp;
    const float4 *bc_r = sBC + rq;
    const int srow = (tid * PPT) / (RB / 16), spiece = (tid * PPT) % (RB / 16);
    const int bcrow = tid / (BCP / kChunk), bcpiece = tid % (BCP / kChunk);

    for (;;) {
        __syncthreads();
        if (tid == 0) s_unit = atomicAdd(cs.counter, 1);
        __syncthreads();
        const int unit = s_unit;
        if (unit >= cs.total) break;
        const int slot = unit / per_seg;
        const int seg = slot + SLOT0;
        const int rem = unit - slot * per_seg;
        const int b = rem / cs.nblk;
        const int c0 = (rem - b * cs.nblk) * CPC;
        const int t0 = seg * cs.seg_len, t1 = min(p.L, t0 + cs.seg_len);
        const int nch = (t1 - t0 + kChunk - 1) / kChunk;

        const int64_t x_rs = REV ? p.do_rs : p.u_rs, bc_rs = REV ? p.C_rs : p.B_rs;
        const T *xb = REV ? reinterpret_cast<const T *>(p.dout) + (int64_t)b * p.do_bs + c0 : reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c0;
        const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c0;
        const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c0 : nullptr;
        const T *BCb = REV ? reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs : reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;

        const uint32_t dst_act = smem_u32(smem) + srow * RB + spiece * 16;
        const uint32_t dst_bc = smem_u32(smem) + NTILE * SM::kTile + tid * 16;
        auto issue = [&](int i, int stage) {   // i-th chunk in processing order -> stage i % NST
            if (i < nch) {
                const int tb = t0 + (REV ? nch - 1 - i : i) * kChunk;
                const int nrows = min(kChunk, t1 - tb);
                const uint32_t so = stage * SM::kStage;
                if constexpr (CPB == 16) {
                    if (srow < nrows) {
                        const char *su = reinterpret_cast<const char *>(xb + (int64_t)(tb + srow) * x_rs) + spiece * 16;
                        const char *sd = reinterpret_cast<const char *>(db + (int64_t)(tb + srow) * p.d_rs) + spiece * 16;
#pragma unroll
                        for (int q = 0; q < PPT; ++q) {
                            cp_async16(dst_act + so + q * 16, su + q * 16);
                            cp_async16(dst_act + so + SM::kTile + q * 16, sd + q * 16);
                        }
                        if (HAS_Z) {
                            const char *sz = reinterpret_cast<const char *>(zb + (int64_t)(tb + srow) * p.z_rs) + spiece * 16;
#pragma unroll
                            for (int q = 0; q < PPT; ++q) cp_async16(dst_act + so + 2 * SM::kTile + q * 16, sz + q * 16);
                        }
                    }
                    if (tid < BCP && bcrow < nrows)
                        cp_async16(dst_bc + so, reinterpret_cast<const char *>(BCb + (int64_t)(tb + bcrow) * bc_rs) + bcpiece * 16);
                } else {
                    unsigned char *s = smem + so;
                    stage_tile<T, CPC, NT>(s, xb + (int64_t)tb * x_rs, x_rs, nrows, tid);
                    stage_tile<T, CPC, NT>(s + SM::kTile, db + (int64_t)tb * p.d_rs, p.d_rs, nrows, tid);
                    if (HAS_Z) stage_tile<T, CPC, NT>(s + 2 * SM::kTile, zb + (int64_t)tb * p.z_rs, p.z_rs, nrows, tid);
                    stage_tile<T, kNState, NT>(s + NTILE * SM::kTile, BCb + (int64_t)tb * bc_rs, bc_rs, nrows, tid);
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int i = 0; i < NST; ++i) issue(i, i);

        float2 A2[2][2], h[2][2];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(p.A_log + (size_t)(c0 + 2 * rp + ch) * kNState) + rq);
            A2[ch][0] = make_float2(-expf(v.x) * kLog2e, -expf(v.y) * kLog2e);
            A2[ch][1] = make_float2(-expf(v.z) * kLog2e, -expf(v.w) * kLog2e);
            h[ch][0] = h[ch][1] = make_float2(0.f, 0.f);
        }
        const float2 bias = p.dt_bias ? __ldg(reinterpret_cast<const float2 *>(p.dt_bias + c0) + ip) : make_float2(0.f, 0.f);
        float2 sdl = make_float2(0.f, 0.f);   // sum of delta over the segment, both channels

        auto phase_a = [&](int i, int stage) {   // per-(t, channel pair) scalars of the i-th chunk -> slots; B | C rows -> fp32 quads
            const int tb = t0 + (REV ? nch - 1 - i : i) * kChunk;
            const unsigned char *s = smem + stage * SM::kStage;
            const T *sX = reinterpret_cast<const T *>(s);
            const T *sD = reinterpret_cast<const T *>(s + SM::kTile);
            const T *sZ = reinterpret_cast<const T *>(s + 2 * SM::kTile);
            const T *sBr = reinterpret_cast<const T *>(s + NTILE * SM::kTile);
            float2 dl[4], xq[4], zq[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int t = ir + 4 * q;
                const float2 x = fadd2(lds_pair(sD + t * CPC, ip), bias);
                float2 sg2;
                const float2 v = softplus_pair<false>(x, sg2);
                dl[q] = sp ? v : x;
                xq[q] = lds_pair(sX + t * CPC, ip);
                if (HAS_Z) zq[q] = lds_pair(sZ + t * CPC, ip);
            }
            float4 bcv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (tid < kChunk * 4 && tb + (tid >> 2) < t1) {
                const T *src = sBr + (tid >> 2) * 16 + 4 * (tid & 3);
                const float2 lo = lds_pair(src, 0), hi = lds_pair(src, 1);
                bcv = make_float4(lo.x, lo.y, hi.x, hi.y);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int t = ir + 4 * q;
                const bool valid = tb + t < t1;   // padded step: a = 1, v = 0
                const float dl0 = valid ? dl[q].x : 0.f, dl1 = valid ? dl[q].y : 0.f;
                float v0 = valid ? xq[q].x : 0.f, v1 = valid ? xq[q].y : 0.f;
                if (REV) {
                    if (HAS_Z) {
                        const float z0 = valid ? zq[q].x : 0.f, z1 = valid ? zq[q].y : 0.f;
                        v0 *= z0 * sigmoid_fast(z0);
                        v1 *= z1 * sigmoid_fast(z1);
                    }
                } else {
                    v0 *= dl0;
                    v1 *= dl1;
                }
                sDD[t * NP + ip] = make_float4(dl0, v0, dl1, v1);
            }
            if (tid < kChunk * 4) sBC[tid] = bcv;
        };

        cp_async_wait<NST - 1>();
        __syncthreads();
        phase_a(0, 0);
        int stage = 0;
        for (int i = 0; i < nch; ++i) {
            __syncthreads();   // (1) slots of this chunk are complete
#pragma unroll
            for (int jj = 0; jj < kChunk; ++jj) {
                const int j = REV ? kChunk - 1 - jj : jj;
                const float4 dd = dd_r[j * NP], B4 = bc_r[j * 4];
                const float2 B01 = make_float2(B4.x, B4.y), B23 = make_float2(B4.z, B4.w);
#pragma unroll
                for (int ch = 0; ch < 2; ++ch) {
                    const float dl = ch ? dd.z : dd.x, v = ch ? dd.w : dd.y;
                    const float2 x0 = fmul2(splat2(dl), A2[ch][0]), x1 = fmul2(splat2(dl), A2[ch][1]);
                    // one exp2 pair of 4 on the FMA pipe (0 / 1 / 2 pairs measured on cfg4: 1 fastest, profiles/r02_chain_variants.txt)
                    const float2 a0 = ch == 0 ? ex2_poly2(x0) : ex2_2(x0);
                    const float2 a1 = ex2_2(x1);
                    if (REV) {
                        h[ch][0] = fmul2(a0, ffma2(B01, splat2(v), h[ch][0]));
                        h[ch][1] = fmul2(a1, ffma2(B23, splat2(v), h[ch][1]));
                    } else {
                        h[ch][0] = ffma2(a0, h[ch][0], fmul2(splat2(v), B01));
                        h[ch][1] = ffma2(a1, h[ch][1], fmul2(splat2(v), B23));
                    }
                }
                sdl.x += dd.x;
                sdl.y += dd.z;
            }
            cp_async_wait<NST - 2>();
            __syncthreads();   // (2) every thread is done with the slots; the next chunk's tiles are visible; this stage is free
            issue(i + NST, stage);
            stage = stage + 1 == NST ? 0 : stage + 1;
            if (i + 1 < nch) phase_a(i + 1, stage);
        }

        float *dst = cs.segc + (((size_t)slot * p.B + b) * p.ED + c0 + 2 * rp) * kNState + 4 * rq;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch)
            *reinterpret_cast<float4 *>(dst + ch * kNState) = make_float4(h[ch][0].x, h[ch][0].y, h[ch][1].x, h[ch][1].y);
        if (rq == 0) *reinterpret_cast<float2 *>(cs.segsd + ((size_t)slot * p.B + b) * p.ED + c0 + 2 * rp) = sdl;
        cp_async_wait<0>();
    }
}

// carry[slot] <- exp2(A sum_delta[slot]) carry[previous slot] + local[slot], in place; forward: slots ascending (the result is
// the carry-in of segment slot + 1), reverse: slots descending (the reverse carry-in of segment slot).  The carry before the
// first slot in processing order is h0[(b, c, n)] ((B, ED, 16), the element index) when h0 is not NULL, else zero: the
// caller's initial state (forward) or the gradient of the final state, dlast (reverse).
// A CTA of 32 x 32 threads serves 32 consecutive (b, c, n) elements: thread (x, y) owns element x and the y-th run of K <= 8
// consecutive slots (in processing order).  It loads its run (all loads in flight at once), reduces it to one (P, S) pair,
// row y = 0 chains the 32 pairs through shared memory, and every thread replays its run from the carry it was handed.
constexpr int kCombK = (kMaxSeg + 31) / 32;
__global__ void __launch_bounds__(1024) selscan_seg_combine_kernel(float *__restrict__ segc, const float *__restrict__ segsd,
                                                                   const float *__restrict__ A_log, const float *__restrict__ h0,
                                                                   int nslots, int B, int ED, int rev) {
    __shared__ float sP[32][33], sS[32][33];
    const int x = threadIdx.x, y = threadIdx.y;
    const int64_t n_el = (int64_t)B * ED * kNState;
    const int64_t idx = (int64_t)blockIdx.x * 32 + x;
    const bool act = idx < n_el;
    const int64_t ic = act ? idx : n_el - 1;
    const int64_t bc = ic >> 4;
    const float a2 = -expf(__ldg(A_log + (size_t)(bc % ED) * kNState + (ic & 15))) * kLog2e;
    const int K = (nslots + 31) / 32;          // slots per run (<= kCombK)
    const int s0 = y * K;
    float S[kCombK], Pd[kCombK];
#pragma unroll
    for (int u = 0; u < kCombK; ++u) {
        const int s = s0 + u;
        S[u] = 0.f; Pd[u] = 1.f;
        if (u < K && s < nslots) {
            const int64_t slot = rev ? nslots - 1 - s : s;
            S[u] = __ldcg(segc + slot * n_el + ic);
            Pd[u] = ex2_approx(a2 * __ldcg(segsd + slot * (n_el >> 4) + bc));
        }
    }
    float P = 1.f, H = 0.f;                    // the run as one step: H_out = P H_in + H
#pragma unroll
    for (int u = 0; u < kCombK; ++u) { H = fmaf(Pd[u], H, S[u]); P *= Pd[u]; }
    sP[y][x] = P; sS[y][x] = H;
    __syncthreads();
    if (y == 0) {
        float h = h0 != nullptr ? __ldg(h0 + ic) : 0.f;
        for (int r = 0; r < 32; ++r) {          // carry INTO run r
            const float pr = sP[r][x], sr = sS[r][x];
            sS[r][x] = h;
            h = fmaf(pr, h, sr);
        }
    }
    __syncthreads();
    H = sS[y][x];
    if (act) {
#pragma unroll
        for (int u = 0; u < kCombK; ++u) {
            const int s = s0 + u;
            if (u < K && s < nslots) {
                const int64_t slot = rev ? nslots - 1 - s : s;
                H = fmaf(Pd[u], H, S[u]);
                segc[slot * n_el + ic] = H;
            }
        }
    }
}

// The same for a few segments (<= 32, e.g. the production shape): one thread per element walks the slots, 8 loads in flight.
__global__ void __launch_bounds__(256) selscan_seg_combine_seq_kernel(float *__restrict__ segc, const float *__restrict__ segsd,
                                                                      const float *__restrict__ A_log, const float *__restrict__ h0,
                                                                      int nslots, int B, int ED, int rev) {
    const int64_t n_el = (int64_t)B * ED * kNState;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= n_el) return;
    const int64_t bc = idx >> 4;
    const float a2 = -expf(__ldg(A_log + (size_t)(bc % ED) * kNState + (idx & 15))) * kLog2e;
    float H = h0 != nullptr ? __ldg(h0 + idx) : 0.f;
    constexpr int U = 8;
    for (int s0 = 0; s0 < nslots; s0 += U) {
        float S[U], sd[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (s0 + u < nslots) {
                const int64_t slot = rev ? nslots - 1 - (s0 + u) : s0 + u;
                S[u] = __ldcg(segc + slot * n_el + idx);
                sd[u] = __ldcg(segsd + slot * (n_el >> 4) + bc);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (s0 + u < nslots) {
                const int64_t slot = rev ? nslots - 1 - (s0 + u) : s0 + u;
                H = fmaf(ex2_approx(a2 * sd[u]), H, S[u]);
                segc[slot * n_el + idx] = H;
            }
        }
    }
}

// Fold of per-segment summaries into the summary of a whole range (gfe_selscan_summary_fwd / _bwd): for every (b, c, n)
// element, out = the carry chain over all nseg segments from a zero carry, carry = exp2(A sum_delta[s]) carry + local[s],
// segments ascending (forward) or descending (reverse); sum_delta (may be NULL) = the sum over s of sum_delta[s].  The
// segment summaries are in the chained layout (GEN = false: local [s][B][ED][16], sum_delta [s][B][ED]) or in the generic
// one (GEN = true: local [B][s][N / 2][ED] float2, sum_delta [B][s][ED]).  out: (B, ED, N); sum_delta: (B, ED).
template <int N, bool GEN>
__global__ void __launch_bounds__(256) selscan_summary_total_kernel(const float *__restrict__ loc, const float *__restrict__ segsd,
                                                                    const float *__restrict__ A_log, float *__restrict__ out,
                                                                    float *__restrict__ sum_delta, int nseg, int B, int ED, int rev) {
    const int64_t n_el = (int64_t)B * ED * N;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= n_el) return;
    const int n = (int)(idx % N);
    const int64_t bc = idx / N;
    const int64_t b = bc / ED, c = bc % ED;
    const float a2 = -expf(__ldg(A_log + c * N + n)) * kLog2e;
    float H = 0.f, S = 0.f;
    for (int i = 0; i < nseg; ++i) {
        const int64_t s = rev ? nseg - 1 - i : i;
        const int64_t si = GEN ? (b * nseg + s) * ED + c : (s * B + b) * ED + c;
        const int64_t li = GEN ? (((b * nseg + s) * (N / 2) + n / 2) * ED + c) * 2 + (n & 1) : s * n_el + idx;
        const float sd = __ldcg(segsd + si);
        H = fmaf(ex2_approx(a2 * sd), H, __ldcg(loc + li));
        S += sd;
    }
    out[idx] = H;
    if (sum_delta != nullptr && n == 0) sum_delta[bc] = S;
}

int launch_summary_total(const float *loc, const float *segsd, const float *A_log, float *out, float *sum_delta, int nseg, int B,
                         int ED, int N, bool generic, bool rev, cudaStream_t st) {
    const unsigned grid = (unsigned)ceil_div64((int64_t)B * ED * N, 256);
    const int r = rev ? 1 : 0;
    if (!generic) selscan_summary_total_kernel<kNState, false><<<grid, 256, 0, st>>>(loc, segsd, A_log, out, sum_delta, nseg, B, ED, r);
    else if (N == 16) selscan_summary_total_kernel<16, true><<<grid, 256, 0, st>>>(loc, segsd, A_log, out, sum_delta, nseg, B, ED, r);
    else if (N == 32) selscan_summary_total_kernel<32, true><<<grid, 256, 0, st>>>(loc, segsd, A_log, out, sum_delta, nseg, B, ED, r);
    else selscan_summary_total_kernel<64, true><<<grid, 256, 0, st>>>(loc, segsd, A_log, out, sum_delta, nseg, B, ED, r);
    return check_launch("selscan summary total");
}

// ---------------------------------------------------------------------------------------------------- host
template <typename T, bool HAS_Z, int CPB, int CPC, bool REV, int SLOT0>
static void launch_summary_inst(const ScanParams &p, const ChainSched &cs, cudaStream_t st) {
    constexpr size_t smem = SegSumSmem<T, HAS_Z, CPC>::kTotal;
    const int grid = persistent_grid<selscan_seg_summary_kernel<T, HAS_Z, CPB, CPC, REV, SLOT0>>(2 * CPC, smem, cs.total);
    selscan_seg_summary_kernel<T, HAS_Z, CPB, CPC, REV, SLOT0><<<grid, 2 * CPC, smem, st>>>(p, cs);
}

// RSLOT0: slot of segment 0 in reverse (1: segments 1 .. nseg-1 for the carries, 0: every segment for a total)
template <typename T, int CPC, int RSLOT0>
static void launch_summary_cpc(const ScanParams &p, const ChainSched &cs, bool rev, bool has_z, int cpb, cudaStream_t st) {
    if (!rev) {   // the forward aggregate never needs z
        if (cpb == 16) launch_summary_inst<T, false, 16, CPC, false, 0>(p, cs, st);
        else launch_summary_inst<T, false, 0, CPC, false, 0>(p, cs, st);
    } else if (has_z) {
        if (cpb == 16) launch_summary_inst<T, true, 16, CPC, true, RSLOT0>(p, cs, st);
        else launch_summary_inst<T, true, 0, CPC, true, RSLOT0>(p, cs, st);
    } else {
        if (cpb == 16) launch_summary_inst<T, false, 16, CPC, true, RSLOT0>(p, cs, st);
        else launch_summary_inst<T, false, 0, CPC, true, RSLOT0>(p, cs, st);
    }
}

template <int RSLOT0>
static int launch_summaries(const ScanParams &p, const ChainSched &s, int dtype, int cpc, bool rev, bool has_z, int cpb, cudaStream_t st) {
    switch (dtype) {
        case GFE_F32:
            if (cpc == 64) launch_summary_cpc<float, 64, RSLOT0>(p, s, rev, has_z, cpb, st);
            else launch_summary_cpc<float, 32, RSLOT0>(p, s, rev, has_z, cpb, st);
            break;
        case GFE_BF16:
            if (cpc == 64) launch_summary_cpc<__nv_bfloat16, 64, RSLOT0>(p, s, rev, has_z, cpb, st);
            else launch_summary_cpc<__nv_bfloat16, 32, RSLOT0>(p, s, rev, has_z, cpb, st);
            break;
        default:
            if (cpc == 64) launch_summary_cpc<__half, 64, RSLOT0>(p, s, rev, has_z, cpb, st);
            else launch_summary_cpc<__half, 32, RSLOT0>(p, s, rev, has_z, cpb, st);
            break;
    }
    return check_launch(rev ? "selscan_bwd segment summary" : "selscan_fwd segment summary");
}

// Summary + combine for the independent segments of `cs` (cs.nseg > 1): fills cs.segc with every segment's carry-in.
// `cs.counter + 16` is the summary pass's own unit counter (zeroed with the main one by chain_fill_sched).
int seg_launch_carries(const ScanParams &p, const ChainSched &cs, int dtype, int cpc, bool rev, bool has_z, int cpb, cudaStream_t st) {
    ChainSched s = cs;
    s.counter = cs.counter + 16;
    s.total = (cs.nseg - 1) * p.B * cs.nblk;
    int rc = launch_summaries<1>(p, s, dtype, cpc, rev, has_z, cpb, st);
    if (rc != GFE_OK) return rc;
    const int64_t n_el = (int64_t)p.B * p.ED * kNState;
    const float *h0 = rev ? p.dlast : p.h0;   // the carry entering the first slot in processing order
    if (cs.nseg - 1 <= 32)
        selscan_seg_combine_seq_kernel<<<(unsigned)ceil_div64(n_el, 256), 256, 0, st>>>(cs.segc, cs.segsd, p.A_log, h0, cs.nseg - 1, p.B, p.ED, rev ? 1 : 0);
    else
        selscan_seg_combine_kernel<<<(unsigned)ceil_div64(n_el, 32), dim3(32, 32), 0, st>>>(cs.segc, cs.segsd, p.A_log, h0, cs.nseg - 1, p.B, p.ED, rev ? 1 : 0);
    return check_launch("selscan segment combine");
}

// The summary of the whole range [0, L) (gfe_selscan_summary_fwd / _bwd) for the chained family: every segment of `cs`
// from a zero carry (slot = segment; cs.segc / cs.segsd hold cs.nseg slots, *cs.counter is zero), folded into out (B, ED, 16)
// and, forward, sum_delta (B, ED).
int seg_launch_total(const ScanParams &p, const ChainSched &cs, int dtype, int cpc, bool rev, bool has_z, int cpb, float *out,
                     float *sum_delta, cudaStream_t st) {
    ChainSched s = cs;
    s.total = cs.nseg * p.B * cs.nblk;
    int rc = launch_summaries<0>(p, s, dtype, cpc, rev, has_z, cpb, st);
    if (rc != GFE_OK) return rc;
    return launch_summary_total(cs.segc, cs.segsd, p.A_log, out, sum_delta, cs.nseg, p.B, p.ED, kNState, false, rev, st);
}

}  // namespace gfe
