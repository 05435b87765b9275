// selscan_chain_bwd.cu -- fused selective-scan backward, chained L-segments, two channels x four states per lane.
// Replaces autograd through mamba.py:255-256, 275-284, 220-222 and PScan.backward (pscan.py:189-224).
//
// Same lane layout as the forward kernel (selscan_v4_fwd.cu): a CTA of 2 * CPC threads serves CPC adjacent channels of
// one batch row; lane (pair, quad) owns the states 4q..4q+3 of channels 2p and 2p + 1 as four float2 pairs.  Against the
// first chained backward (one channel x four states per lane, profiles/r02_chain_variants.txt) every B|C quad fetched from
// shared memory feeds eight state-steps instead of four, the first level of the cross-channel dB|dC sums is an FFMA in the
// lane, the shuffle reduction runs over half as many values, and the per-(t, channel) sums over states leave the lane as
// ONE 16-byte store.  Per lane and step (8 state-steps): 6 LDS + 48 packed FP32 + 16 exp2 + 7 SHFL + 1 STS.128.
//
// Per unit = (L-segment, batch row, channel block), segments walked last to first (ChainSched, see selscan_shared.cuh; the
// segments are either chained through flags or independent, their carries then coming from selscan_seg.cu):
//   chunks of 16 steps are staged by cp.async (u, delta, dout, [y, z], B, C and the two checkpoints) and walked in reverse:
//   phase A  (item mapping, thread per (t, channel pair), packed FP32 over the pair): softplus and its derivative,
//            dy = dout * silu(z), dz, the slots {dl0, dl1, dl0 u0, dl1 u1}, {dy0, dy1}, {u0, u1, sg0, sg1}; B|C rows -> fp32
//            quads (natural and pair-swapped plane).  Rows are masked only in a ragged last chunk (template flag);
//   phase B  (recurrence mapping): a forward sweep re-derives the 8 states and decay factors of steps 8..15 from their
//            checkpoint into registers; then the reverse sweep of steps 8..15 (g[t] = C dy + a[t+1] g[t+1], every
//            contraction as packed FP32 ops; dB|dC reduced over the 8 pairs of the warp in groups of 2 steps: 14 SHFL per 16
//            values, the first level without selects because odd pairs hold their state pairs swapped) runs INTERLEAVED
//            with the forward sweep of steps 0..7 -- one is bound by FP32 operand delivery, the other by MUFU, and the
//            histories hand their registers over step by step -- followed by the reverse sweep of steps 0..7;
//   phase C  (warp-local item mapping, right after each reverse sweep: only __syncwarp, packed FP32): du, ddelta from the
//            four quads' partials; dD / ddt_bias accumulation;
//   then the warps' dB|dC rows are added and leave as one row per (CTA, t) for selscan_bwd_finalize_bc.
#include <type_traits>

#include "common.cuh"
#include "selscan_shared.cuh"

namespace gfe {

int chain_fill_sched(ChainSched &cs, char *ws, int B, int ED, const ChainPlan &pl, cudaStream_t st);
size_t chain_bytes(int B, int ED, const ChainPlan &pl);
int seg_launch_carries(const ScanParams &p, const ChainSched &cs, int dtype, int cpc, bool rev, bool has_z, int cpb, cudaStream_t st);   // selscan_seg.cu
void chain_fill_params(ScanParams &p, const gfe_selscan_args *a);
int chain_cpb(const gfe_selscan_args *a, bool bwd);
bool chain_pair_stores(const gfe_selscan_args *a, bool bwd);
int chain_check_alignment(const gfe_selscan_args *a);
void launch_bwd_finalize(const gfe_selscan_args *a, ScanParams &p, cudaStream_t st, int &rc);   // selscan.cu

constexpr int kCRedRow = 36;   // padded row (floats) of the per-warp dB|dC tile: [t][n]{dB, dC}
constexpr int kCBCPlane = kChunk * 8 + 4;   // float4 per B|C plane; the 64 B skew keeps the natural and the pair-swapped plane
                                            // (read by the even / odd pairs of one quarter-warp) on disjoint banks

template <typename T, bool HAS_Z, int CPC>
struct BwdChainSmem {
    static constexpr int kStages = 2;
    static constexpr int NP = CPC / 2;
    static constexpr int NW = CPC / 16;                                 // warps per CTA
    static constexpr int kTile = kChunk * CPC * (int)sizeof(T);         // one of u, delta, dout, y, z
    static constexpr int kNTile = HAS_Z ? 5 : 3;
    static constexpr int kBCRaw = kChunk * kNState * (int)sizeof(T);     // one of B, C
    using CK = typename CkptOf<T>::type;
    static constexpr int kCk = CPC * kNState * (int)sizeof(CK);          // the checkpoints of one half chunk: [c][16]
    static constexpr int kOffCk = kNTile * kTile + 2 * kBCRaw;           // inside a stage: both halves' checkpoints
    static constexpr int kStage = kOffCk + 2 * kCk;
    static constexpr int kSPlane = NP + 2;                               // float4 per (t, quad) plane of the partials (+32 B skew)
    static constexpr int kOffDD = kStages * kStage;                      // float4 [16][NP] {dl0, dl0 u0, dl1, dl1 u1}
    static constexpr int kOffDY = kOffDD + kChunk * NP * 16;             // float2 [16][NP] {dy0, dy1}
    static constexpr int kOffEpi = kOffDY + kChunk * NP * 8;             // float4 [16][NP] {u0, softplus'0, u1, softplus'1}
    static constexpr int kOffBC = kOffEpi + kChunk * NP * 16;            // float4 [2][16][8] (+64 B skew) B quads | C quads
    static constexpr int kOffS = kOffBC + 2 * kCBCPlane * 16;            // float4 [8][4][NP + 2] {S1_0, S2_0, S1_1, S2_1} of one half chunk
    static constexpr int kOffRed = kOffS + kCkptV2 * 4 * kSPlane * 16;   // float  [NW][16][36] per-warp dB|dC rows
    static constexpr int kTotal = kOffRed + NW * kChunk * kCRedRow * 4;
};

#ifdef GFE_PHASE_CLOCKS   // development only: cycles per phase, summed over warp leaders (tools/dbg/phase_clocks.py)
__device__ unsigned long long g_bwd_phase_clk[8];
#define GFE_CLK(i) do { const long long now_ = clock64(); if ((threadIdx.x & 31) == 0) clk_acc[i] += now_ - clk_last; clk_last = now_; } while (0)
#else
#define GFE_CLK(i) do { } while (0)
#endif

template <typename T, bool HAS_Z, int CPB, int CPC>
__global__ void __launch_bounds__(2 * CPC, kBwdMinBlocks * (64 / CPC)) selscan_bwd_chain_kernel(ScanParams p, ChainSched cs) {
#ifdef GFE_PHASE_CLOCKS
    long long clk_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, clk_last = clock64();
#endif
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_unit;
    using SM = BwdChainSmem<T, HAS_Z, CPC>;
    constexpr int NT = 2 * CPC, NP = SM::NP, NW = SM::NW, NST = SM::kStages, NTILE = SM::kNTile;
    constexpr int RB = CPC * (int)sizeof(T);          // bytes per activation tile row
    constexpr int PPT = kChunk * RB / 16 / NT;        // 16-byte pieces per thread per activation tile (1 for 16-bit, 2 for fp32)
    constexpr int BCP = kChunk * kNState * (int)sizeof(T) / 16;   // pieces per B (or C) tile: 32 (16-bit), 64 (fp32)
    constexpr int BCI = (2 * BCP + NT - 1) / NT;      // B|C pieces per thread
    constexpr int BCC = kChunk * 8 / NT;              // fp32 B|C quads converted per thread
    using CK = typename SM::CK;
    constexpr int CKP = 2 * SM::kCk / 16 / NT;        // 16-byte checkpoint pieces per thread and chunk (4 fp32, 2 bf16)
    constexpr int SPL = SM::kSPlane;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rp = tid >> 2, rq = tid & 3;     // recurrence mapping: channel pair in block, state quad
    const int sw = rp & 1;                     // odd pairs hold their state pairs swapped (select-free first reduce level)
    const int ip = tid % NP, ir = tid / NP;    // phase A mapping: channel pair, rows ir + 4 i
    const int cp = warp * 8 + (lane & 7), cr = lane >> 3;   // phase C mapping (warp-local): channel pair, rows cr + 4 i of a half

    float4 *sDD = reinterpret_cast<float4 *>(smem + SM::kOffDD);
    float2 *sDY = reinterpret_cast<float2 *>(smem + SM::kOffDY);
    float4 *sEpi = reinterpret_cast<float4 *>(smem + SM::kOffEpi);
    float4 *sBC = reinterpret_cast<float4 *>(smem + SM::kOffBC);
    float4 *sS = reinterpret_cast<float4 *>(smem + SM::kOffS);
    float *sRed = reinterpret_cast<float *>(smem + SM::kOffRed);
    const bool sp = p.flags & GFE_FLAG_DELTA_SOFTPLUS;
    constexpr bool vec = CPB == 16;   // the cp.async instantiation also requires pair-aligned outputs (chain_launch_bwd)
    const int per_seg = p.B * cs.nblk;

    // recurrence-side shared pointers (fixed for the whole kernel)
    const float4 *dd_r = sDD + rp;
    const float2 *dy_r = sDY + rp;
    const float4 *bc_r = sBC + sw * kCBCPlane + rq;
    float4 *s_w = sS + rq * SPL + rp;
    const bool up8 = (lane & 8) != 0, up16 = (lane & 16) != 0;
    float *red_w = sRed + warp * (kChunk * kCRedRow) + (up16 ? kCRedRow : 0) + 2 * (4 * rq + (up8 ? 2 : 0) + sw);

    // staging geometry of this thread (fixed)
    const int srow = (tid * PPT) / (RB / 16), spiece = (tid * PPT) % (RB / 16);   // PPT consecutive pieces of one row

    for (;;) {
        __syncthreads();
        if (tid == 0) s_unit = atomicAdd(cs.counter, 1);
        __syncthreads();
        const int unit = s_unit;
        if (unit >= cs.total) break;
        const int rseg = unit / per_seg;           // processing order: last time segment first
        const int seg = cs.nseg - 1 - rseg;
        const int rem = unit - rseg * per_seg;
        const int b = rem / cs.nblk;
        const int blk = rem - b * cs.nblk;
        const int c0 = blk * CPC;
        const int t0 = seg * cs.seg_len, t1 = min(p.L, t0 + cs.seg_len);
        const int kfirst = t0 / kChunk, klast = (t1 - 1) / kChunk;   // global chunk indices, walked klast .. kfirst
        const int nch = klast - kfirst + 1;

        const T *ub = reinterpret_cast<const T *>(p.u) + (int64_t)b * p.u_bs + c0;
        const T *db = reinterpret_cast<const T *>(p.delta) + (int64_t)b * p.d_bs + c0;
        const T *gb = reinterpret_cast<const T *>(p.dout) + (int64_t)b * p.do_bs + c0;
        const T *yb = reinterpret_cast<const T *>(p.ysave) + (int64_t)b * p.L * p.ED + c0;
        const T *zb = HAS_Z ? reinterpret_cast<const T *>(p.z) + (int64_t)b * p.z_bs + c0 : nullptr;
        const T *Bb = reinterpret_cast<const T *>(p.Bm) + (int64_t)b * p.B_bs;
        const T *Cb = reinterpret_cast<const T *>(p.Cm) + (int64_t)b * p.C_bs;
        // checkpoints [b][t / 8][c][16] fp32: the block's CPC channels of one half chunk are contiguous (staged with the tiles)
        const char *ckb = reinterpret_cast<const char *>(reinterpret_cast<const CK *>(p.ckpt) +
                                                         ((size_t)b * p.nchunks * p.ED + c0) * kNState);
        const size_t ck_step = (size_t)p.ED * kNState * sizeof(CK);      // bytes between consecutive checkpoints
        T *dub = reinterpret_cast<T *>(p.du) + (int64_t)b * p.du_bs + c0 + 2 * cp;
        T *ddb = reinterpret_cast<T *>(p.ddelta) + (int64_t)b * p.dd_bs + c0 + 2 * cp;
        T *dzb = HAS_Z ? reinterpret_cast<T *>(p.dz) + (int64_t)b * p.dz_bs + c0 + 2 * ip : nullptr;

        // per-thread source pointers of the staged pieces of the NEXT chunk to issue (cp.async path): chunks are issued strictly in
        // processing order (klast, klast - 1, ...), so every pointer just steps back by one chunk after each issue
        const char *su = nullptr, *sd = nullptr, *sg_ = nullptr, *sy = nullptr, *sz = nullptr, *sbc[BCI], *sck = nullptr;
        int bcrow[BCI];
        constexpr int PH = SM::kCk / 16;      // 16-byte pieces per half-chunk checkpoint block: NT (16-bit states) or 2 NT (fp32)
        static_assert(PH % NT == 0 && CKP == 2 * (PH / NT), "checkpoint staging layout");
        sck = ckb + (size_t)(2 * klast) * ck_step + tid * 16;
        if constexpr (CPB == 16) {
            const int64_t r0 = (int64_t)klast * kChunk + srow;
            su = reinterpret_cast<const char *>(ub + r0 * p.u_rs) + spiece * 16;
            sd = reinterpret_cast<const char *>(db + r0 * p.d_rs) + spiece * 16;
            sg_ = reinterpret_cast<const char *>(gb + r0 * p.do_rs) + spiece * 16;
            if (HAS_Z) {
                sy = reinterpret_cast<const char *>(yb + r0 * p.ED) + spiece * 16;
                sz = reinterpret_cast<const char *>(zb + r0 * p.z_rs) + spiece * 16;
            }
#pragma unroll
            for (int i = 0; i < BCI; ++i) {
                const int pc = tid + i * NT;
                const int sel = pc / BCP, within = pc % BCP;    // 0: B, 1: C
                bcrow[i] = within / (BCP / kChunk);
                const int64_t rs = sel ? p.C_rs : p.B_rs;
                sbc[i] = reinterpret_cast<const char *>((sel ? Cb : Bb) + ((int64_t)klast * kChunk + bcrow[i]) * rs) + (within % (BCP / kChunk)) * 16;
            }
        }
        const uint32_t dst_act = smem_u32(smem) + srow * RB + spiece * 16;
        const uint32_t dst_bc = smem_u32(smem) + NTILE * SM::kTile + tid * 16;   // raw B tile followed by raw C tile
        const uint32_t dst_ck = smem_u32(smem) + SM::kOffCk + tid * 16;

        auto issue = [&](int i, int stage) {   // i-th chunk in processing order (global chunk klast - i) -> stage i % NST
            if (i < nch) {
                const int tb = (klast - i) * kChunk;
                const int nrows = min(kChunk, t1 - tb);
                const uint32_t so = stage * SM::kStage;
                {   // both halves' checkpoints (states before steps tb and tb + 8); always 16-byte aligned
                    const int nhalf = tb + kCkptV2 < t1 ? 2 : 1;
#pragma unroll
                    for (int q = 0; q < CKP; ++q) {   // piece tid + q NT of [half][c][16]
                        constexpr int QH = PH / NT;    // pieces per thread and half
                        if (q / QH < nhalf) cp_async16(dst_ck + so + q * NT * 16, sck + (size_t)(q / QH) * ck_step + (q % QH) * NT * 16);
                        else *reinterpret_cast<float4 *>(smem + so + SM::kOffCk + (tid + q * NT) * 16) = make_float4(0.f, 0.f, 0.f, 0.f);   // identity half
                    }
                    sck -= 2 * ck_step;
                }
                if constexpr (CPB == 16) {
                    if (srow < nrows) {
#pragma unroll
                        for (int q = 0; q < PPT; ++q) {
                            cp_async16(dst_act + so + q * 16, su + q * 16);
                            cp_async16(dst_act + so + SM::kTile + q * 16, sd + q * 16);
                            cp_async16(dst_act + so + 2 * SM::kTile + q * 16, sg_ + q * 16);
                            if (HAS_Z) {
                                cp_async16(dst_act + so + 3 * SM::kTile + q * 16, sy + q * 16);
                                cp_async16(dst_act + so + 4 * SM::kTile + q * 16, sz + q * 16);
                            }
                        }
                    }
#pragma unroll
                    for (int q = 0; q < BCI; ++q)
                        if (tid + q * NT < 2 * BCP && bcrow[q] < nrows) cp_async16(dst_bc + so + q * NT * 16, sbc[q]);
                    constexpr int64_t sz_t = (int64_t)sizeof(T) * kChunk;
                    su -= p.u_rs * sz_t; sd -= p.d_rs * sz_t; sg_ -= p.do_rs * sz_t;
                    if (HAS_Z) { sy -= (int64_t)p.ED * sz_t; sz -= p.z_rs * sz_t; }
#pragma unroll
                    for (int q = 0; q < BCI; ++q) sbc[q] -= ((tid + q * NT) / BCP ? p.C_rs : p.B_rs) * sz_t;
                } else {
                    unsigned char *s = smem + so;
                    stage_tile<T, CPC, NT>(s, ub + (int64_t)tb * p.u_rs, p.u_rs, nrows, tid);
                    stage_tile<T, CPC, NT>(s + SM::kTile, db + (int64_t)tb * p.d_rs, p.d_rs, nrows, tid);
                    stage_tile<T, CPC, NT>(s + 2 * SM::kTile, gb + (int64_t)tb * p.do_rs, p.do_rs, nrows, tid);
                    if (HAS_Z) {
                        stage_tile<T, CPC, NT>(s + 3 * SM::kTile, yb + (int64_t)tb * p.ED, p.ED, nrows, tid);
                        stage_tile<T, CPC, NT>(s + 4 * SM::kTile, zb + (int64_t)tb * p.z_rs, p.z_rs, nrows, tid);
                    }
                    unsigned char *sb = s + NTILE * SM::kTile;
                    stage_tile<T, kNState, NT>(sb, Bb + (int64_t)tb * p.B_rs, p.B_rs, nrows, tid);
                    stage_tile<T, kNState, NT>(sb + SM::kBCRaw, Cb + (int64_t)tb * p.C_rs, p.C_rs, nrows, tid);
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int i = 0; i < NST; ++i) issue(i, i);

        // per-thread constants (state pairs swapped when sw)
        float2 A2[2][2], G[2][2], dA[2][2];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(p.A_log + (size_t)(c0 + 2 * rp + ch) * kNState) + rq);
            const float a0 = -expf(v.x) * kLog2e, a1 = -expf(v.y) * kLog2e, a2 = -expf(v.z) * kLog2e, a3 = -expf(v.w) * kLog2e;
            A2[ch][0] = sw ? make_float2(a1, a0) : make_float2(a0, a1);
            A2[ch][1] = sw ? make_float2(a3, a2) : make_float2(a2, a3);
            dA[ch][0] = dA[ch][1] = make_float2(0.f, 0.f);
        }
        const float2 bias = p.dt_bias ? __ldg(reinterpret_cast<const float2 *>(p.dt_bias + c0) + ip) : make_float2(0.f, 0.f);   // phase A pair
        const float2 Dc = __ldg(reinterpret_cast<const float2 *>(p.D + c0) + cp);                                                // phase C pair
        float2 dD_acc = make_float2(0.f, 0.f), dbias_acc = make_float2(0.f, 0.f);

        float *carry = cs.independent ? cs.segc + (((size_t)(rseg > 0 ? seg : 0) * p.B + b) * p.ED + c0 + 2 * rp) * kNState + 4 * rq
                                      : cs.carry + ((size_t)b * p.ED + c0 + 2 * rp) * kNState + 4 * rq;
        if (rseg > 0) {
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
                G[ch][0] = sw ? make_float2(v.y, v.x) : make_float2(v.x, v.y);
                G[ch][1] = sw ? make_float2(v.w, v.z) : make_float2(v.z, v.w);
            }
        } else {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) G[ch][0] = G[ch][1] = make_float2(0.f, 0.f);
        }

        // FULL: all 16 rows of the chunk lie inside the sequence (every chunk but a ragged last one): no row masking at all.
        // Slot layouts follow the packed register pairs: {dl0, dl1, dl0 u0, dl1 u1}, {dy0, dy1}, {u0, u1, softplus'0, softplus'1}.
        auto phase_a = [&](int i, int stage, auto full_c) {
            constexpr bool FULL = decltype(full_c)::value;
            const int tb = (klast - i) * kChunk;
            const unsigned char *s = smem + stage * SM::kStage;
            const T *sU = reinterpret_cast<const T *>(s);
            const T *sD = reinterpret_cast<const T *>(s + SM::kTile);
            const T *sDo = reinterpret_cast<const T *>(s + 2 * SM::kTile);
            const T *sY = reinterpret_cast<const T *>(s + 3 * SM::kTile);
            const T *sZ = reinterpret_cast<const T *>(s + 4 * SM::kTile);
            const T *sBr = reinterpret_cast<const T *>(s + NTILE * SM::kTile);
            float2 dl[4], sg[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {   // branch-free packed softplus + sigmoid (selscan_shared.cuh)
                dl[q] = fadd2(lds_pair(sD + (ir + 4 * q) * CPC, ip), bias);
                sg[q] = make_float2(1.0f, 1.0f);
            }
            if (sp) {
#pragma unroll
                for (int q = 0; q < 4; ++q) dl[q] = softplus_pair<true>(dl[q], sg[q]);
            }
            float2 uq[4], gq[4], zq[4], yq[4];   // every load of the phase before its first store (an LDS is never moved above an STS)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int t = ir + 4 * q;
                uq[q] = lds_pair(sU + t * CPC, ip);
                gq[q] = lds_pair(sDo + t * CPC, ip);
                if (HAS_Z) {
                    zq[q] = lds_pair(sZ + t * CPC, ip);
                    yq[q] = lds_pair(sY + t * CPC, ip);
                }
            }
            float4 bcv[BCC];
#pragma unroll
            for (int q = 0; q < BCC; ++q) {
                const int e = tid + q * NT, t = e >> 3, q8 = e & 7;
                bcv[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (FULL || tb + t < t1) bcv[q] = lds_quad(sBr + (q8 < 4 ? 0 : kChunk * 16) + t * 16 + 4 * (q8 & 3));
            }
            T *dzp = HAS_Z ? dzb + ((int64_t)tb + ir) * p.dz_rs : nullptr;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int t = ir + 4 * q;
                const bool valid = FULL || tb + t < t1;
                float2 u2 = uq[q], do2 = gq[q], dl2 = dl[q];
                if (!FULL && !valid) u2 = do2 = dl2 = make_float2(0.f, 0.f);   // padded step: a = 1, bx = 0, dy = 0
                float2 dy2 = do2;
                if (HAS_Z) {
                    float2 z2 = zq[q];
                    if (!FULL && !valid) z2 = make_float2(0.f, 0.f);
                    const float2 ez = ex2_2(fmul2(z2, splat2(-kLog2e)));
                    const float2 den = fadd2(ez, splat2(1.0f));
                    const float2 sz2 = make_float2(rcp_approx(den.x), rcp_approx(den.y));   // sigmoid(z)
                    const float2 zs = fmul2(z2, sz2);                                        // silu(z)
                    dy2 = fmul2(do2, zs);
                    if (valid) {   // dz = dout * d silu(z)/dz * y needs nothing from the sweeps: d silu = sz (1 + z - z sz)
                        const float2 w = fadd2(fadd2(z2, splat2(1.0f)), make_float2(-zs.x, -zs.y));
                        const float2 f = fmul2(fmul2(do2, sz2), fmul2(w, yq[q]));
                        stg_pair<T>(dzp, f.x, f.y, vec);
                    }
                    dzp += 4 * p.dz_rs;
                }
                const float2 dlu = fmul2(dl2, u2);
                sDD[t * NP + ip] = make_float4(dl2.x, dl2.y, dlu.x, dlu.y);
                sDY[t * NP + ip] = dy2;
                sEpi[t * NP + ip] = make_float4(u2.x, u2.y, sg[q].x, sg[q].y);
            }
            // B|C rows as fp32 quads, natural and pair-swapped order: [sw][t][B quads 0..3 | C quads 0..3]
#pragma unroll
            for (int q = 0; q < BCC; ++q) {
                sBC[tid + q * NT] = bcv[q];
                sBC[kCBCPlane + tid + q * NT] = make_float4(bcv[q].y, bcv[q].x, bcv[q].w, bcv[q].z);
            }
        };
        auto phase_a_any = [&](int i, int stage) {
            if ((klast - i) * kChunk + kChunk <= t1) phase_a(i, stage, std::true_type{});
            else phase_a(i, stage, std::false_type{});
        };

        GFE_CLK(0);   // unit set-up (incl. waiting for the successor segment's carry)
        cp_async_wait<NST - 1>();
        __syncthreads();
        phase_a_any(0, 0);
        GFE_CLK(5);

        int stage = 0;   // i % NST
        for (int i = 0; i < nch; ++i) {
            const int k = klast - i;
            const int tb = k * kChunk;
            __syncthreads();   // (1) slots of this chunk are complete
            GFE_CLK(1);

            // ------------------------------------------------------------ phase B + C
            // Both halves of the chunk are always walked (a half beyond the sequence consists of identity steps: delta = 0,
            // dy = 0, a zeroed checkpoint).  The reverse sweep of steps 8..15 and the forward sweep of steps 0..7 are
            // independent -- one is bound by FP32 operand delivery, the other by MUFU -- and run interleaved in one
            // instruction stream; the histories of the two halves hand their registers over step by step.
            float2 hA0[2][kCkptV2 + 1], hA1[2][kCkptV2 + 1], eA0[2][kCkptV2], eA1[2][kCkptV2];   // steps 8..15
            float2 hB0[2][kCkptV2 + 1], hB1[2][kCkptV2 + 1], eB0[2][kCkptV2], eB1[2][kCkptV2];   // steps 0..7
            const unsigned char *ckbase = smem + stage * SM::kStage + SM::kOffCk;
            auto load_ck = [&](float2 (&h0)[2][kCkptV2 + 1], float2 (&h1)[2][kCkptV2 + 1], int half) {
#pragma unroll
                for (int ch = 0; ch < 2; ++ch) {
                    const float4 ck = ckpt_load_smem(reinterpret_cast<const CK *>(ckbase + half * SM::kCk) + (2 * rp + ch) * kNState + 4 * rq);
                    h0[ch][0] = sw ? make_float2(ck.y, ck.x) : make_float2(ck.x, ck.y);
                    h1[ch][0] = sw ? make_float2(ck.w, ck.z) : make_float2(ck.z, ck.w);
                }
            };
            auto fwd_step = [&](float2 (&h0)[2][kCkptV2 + 1], float2 (&h1)[2][kCkptV2 + 1], float2 (&e0h)[2][kCkptV2],
                                float2 (&e1h)[2][kCkptV2], const float4 dd, const float4 B4, int j) {
                const float2 B01 = make_float2(B4.x, B4.y), B23 = make_float2(B4.z, B4.w);
#pragma unroll
                for (int ch = 0; ch < 2; ++ch) {
                    const float2 dl2 = splat2(ch ? dd.y : dd.x), du2 = splat2(ch ? dd.w : dd.z);   // scalar-broadcast operands
                    const float2 e0 = ex2_2(fmul2(dl2, A2[ch][0])), e1 = ex2_2(fmul2(dl2, A2[ch][1]));
                    e0h[ch][j] = e0; e1h[ch][j] = e1;
                    h0[ch][j + 1] = ffma2(e0, h0[ch][j], fmul2(du2, B01));
                    h1[ch][j + 1] = ffma2(e1, h1[ch][j], fmul2(du2, B23));
                }
            };
            // one group of two reverse steps (jb + 1, jb) of the half at row offset jo, with the slot loads of the following
            // step issued ahead (neither nvcc nor ptxas moves an LDS above a may-alias STS)
            float4 dd_n, B_n, C_n;
            float2 dy_n;
            auto rev_prime = [&](int jo) {
                dd_n = dd_r[(jo + kCkptV2 - 1) * NP]; B_n = bc_r[(jo + kCkptV2 - 1) * 8]; C_n = bc_r[(jo + kCkptV2 - 1) * 8 + 4];
                dy_n = dy_r[(jo + kCkptV2 - 1) * NP];
            };
            auto rev_group = [&](float2 (&h0)[2][kCkptV2 + 1], float2 (&h1)[2][kCkptV2 + 1], float2 (&e0h)[2][kCkptV2],
                                 float2 (&e1h)[2][kCkptV2], int jo, int jb) {
                const float4 *dd_p = dd_r + jo * NP;
                const float2 *dy_p = dy_r + jo * NP;
                const float4 *bc_p = bc_r + jo * 8;
                float v[16];   // [kind (dB, dC)][step in group (2)][state in quad (4)], summed over the lane's two channels
#pragma unroll
                for (int jj = 1; jj >= 0; --jj) {
                    const int j = jb + jj;
                    const float4 dd = dd_n, B4 = B_n, C4 = C_n;
                    const float2 dyv = dy_n;
                    if (j > 0) {
                        dd_n = dd_p[(j - 1) * NP]; B_n = bc_p[(j - 1) * 8]; C_n = bc_p[(j - 1) * 8 + 4];
                        dy_n = dy_p[(j - 1) * NP];
                    }
                    const float2 B01 = make_float2(B4.x, B4.y), B23 = make_float2(B4.z, B4.w);
                    const float2 C01 = make_float2(C4.x, C4.y), C23 = make_float2(C4.z, C4.w);
                    float2 dc0, dc1, db0, db1;
                    float4 part;
#pragma unroll
                    for (int ch = 0; ch < 2; ++ch) {
                        const float2 dl2 = splat2(ch ? dd.y : dd.x), du2 = splat2(ch ? dd.w : dd.z), dy2 = splat2(ch ? dyv.y : dyv.x);
                        const float2 gg0 = ffma2(C01, dy2, G[ch][0]);   // g[t] = C dy + a[t+1] g[t+1]
                        const float2 gg1 = ffma2(C23, dy2, G[ch][1]);
                        if (ch == 0) {
                            dc0 = fmul2(dy2, h0[ch][j + 1]); dc1 = fmul2(dy2, h1[ch][j + 1]);   // dC_t[n] += dy h[t]
                            db0 = fmul2(gg0, du2); db1 = fmul2(gg1, du2);                       // dB_t[n] += g delta u
                        } else {
                            dc0 = ffma2(dy2, h0[ch][j + 1], dc0); dc1 = ffma2(dy2, h1[ch][j + 1], dc1);
                            db0 = ffma2(gg0, du2, db0); db1 = ffma2(gg1, du2, db1);
                        }
                        const float2 sb = ffma2(gg1, B23, fmul2(gg0, B01));                      // sum_n g B
                        G[ch][0] = fmul2(e0h[ch][j], gg0);                                       // a[t] g[t]
                        G[ch][1] = fmul2(e1h[ch][j], gg1);
                        const float2 w0 = fmul2(G[ch][0], h0[ch][j]), w1 = fmul2(G[ch][1], h1[ch][j]);   // (d a) a = g a h[t-1]
                        const float2 sa = ffma2(w1, A2[ch][1], fmul2(w0, A2[ch][0]));            // sum_n (da a) A log2e
                        dA[ch][0] = ffma2(w0, dl2, dA[ch][0]);                                   // dA[c,n] += (da a) delta
                        dA[ch][1] = ffma2(w1, dl2, dA[ch][1]);
                        if (ch == 0) { part.x = sb.x + sb.y; part.z = sa.x + sa.y; }   // {S1_0, S1_1, S2_0, S2_1}
                        else { part.y = sb.x + sb.y; part.w = sa.x + sa.y; }
                    }
                    s_w[j * (4 * SPL)] = part;
                    v[4 * jj] = db0.x; v[4 * jj + 1] = db0.y; v[4 * jj + 2] = db1.x; v[4 * jj + 3] = db1.y;
                    v[8 + 4 * jj] = dc0.x; v[8 + 4 * jj + 1] = dc0.y; v[8 + 4 * jj + 2] = dc1.x; v[8 + 4 * jj + 3] = dc1.y;
                }
                // reduce the 16 values over the 8 lanes that share this quad (lane bits 2, 3, 4)
                float r1[8];   // [kind][jj][m]: state 4 rq + 2 m + sw (odd pairs hold their state pairs swapped)
#pragma unroll
                for (int m = 0; m < 8; ++m) r1[m] = v[2 * m] + __shfl_xor_sync(0xffffffffu, v[2 * m + 1], 4);
                float r2[4];   // [kind][jj]: exchange on m
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const float keep = up8 ? r1[2 * m + 1] : r1[2 * m];
                    const float send = up8 ? r1[2 * m] : r1[2 * m + 1];
                    r2[m] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                }
                float r3[2];   // [kind]: exchange on jj
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    const float keep = up16 ? r2[2 * m + 1] : r2[2 * m];
                    const float send = up16 ? r2[2 * m] : r2[2 * m + 1];
                    r3[m] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                }
                *reinterpret_cast<float2 *>(red_w + (jo + jb) * kCRedRow) = make_float2(r3[0], r3[1]);   // {dB, dC} of (step, state)
            };
            auto phase_c = [&](int jo) {   // this warp's 8 pairs x 8 steps
                __syncwarp();
                T *dup = dub + ((int64_t)tb + jo + cr) * p.du_rs, *ddp = ddb + ((int64_t)tb + jo + cr) * p.dd_rs;
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int tl = cr + 4 * q, t = jo + tl;
                    if (tb + t < t1) {
                        const float4 *sp4 = sS + (tl * 4) * SPL + cp;   // {S1_0, S1_1, S2_0, S2_1}, one plane per quad
                        const float4 p0 = sp4[0], p1 = sp4[SPL], p2 = sp4[2 * SPL], p3 = sp4[3 * SPL];
                        const float4 dd = sDD[t * NP + cp];
                        const float2 dy = sDY[t * NP + cp];
                        const float4 e4 = sEpi[t * NP + cp];
                        const float2 s1 = fadd2(fadd2(make_float2(p0.x, p0.y), make_float2(p1.x, p1.y)), fadd2(make_float2(p2.x, p2.y), make_float2(p3.x, p3.y)));
                        const float2 s2 = fmul2(fadd2(fadd2(make_float2(p0.z, p0.w), make_float2(p1.z, p1.w)), fadd2(make_float2(p2.z, p2.w), make_float2(p3.z, p3.w))), splat2(kLn2));
                        const float2 u2 = make_float2(e4.x, e4.y);
                        const float2 draw = fmul2(ffma2(s1, u2, s2), make_float2(e4.z, e4.w));   // d delta through softplus
                        const float2 du = ffma2(make_float2(dd.x, dd.y), s1, fmul2(Dc, dy));
                        stg_pair<T>(dup, du.x, du.y, vec);
                        stg_pair<T>(ddp, draw.x, draw.y, vec);
                        dD_acc = ffma2(dy, u2, dD_acc);
                        dbias_acc = fadd2(dbias_acc, draw);
                    }
                    dup += 4 * p.du_rs;
                    ddp += 4 * p.dd_rs;
                }
                __syncwarp();   // the next half overwrites the partial planes
            };

            load_ck(hA0, hA1, 1);
#pragma unroll
            for (int j = 0; j < kCkptV2; ++j) fwd_step(hA0, hA1, eA0, eA1, dd_r[(kCkptV2 + j) * NP], bc_r[(kCkptV2 + j) * 8], j);
            load_ck(hB0, hB1, 0);
            rev_prime(kCkptV2);
#pragma unroll
            for (int g = 0; g < kCkptV2 / 2; ++g) {
                const float4 ddf0 = dd_r[(2 * g) * NP], Bf0 = bc_r[(2 * g) * 8];             // forward-step slots, before the group's stores
                const float4 ddf1 = dd_r[(2 * g + 1) * NP], Bf1 = bc_r[(2 * g + 1) * 8];
                rev_group(hA0, hA1, eA0, eA1, kCkptV2, kCkptV2 - 2 - 2 * g);
                fwd_step(hB0, hB1, eB0, eB1, ddf0, Bf0, 2 * g);
                fwd_step(hB0, hB1, eB0, eB1, ddf1, Bf1, 2 * g + 1);
            }
            GFE_CLK(2);
            phase_c(kCkptV2);
            rev_prime(0);
#pragma unroll
            for (int g = 0; g < kCkptV2 / 2; ++g) rev_group(hB0, hB1, eB0, eB1, 0, kCkptV2 - 2 - 2 * g);
            phase_c(0);
            GFE_CLK(6);

            cp_async_wait<NST - 2>();
            __syncthreads();   // (2) per-warp dB|dC rows complete; next chunk visible; this chunk's stage free
            GFE_CLK(3);
            issue(i + NST, stage);
            stage = stage + 1 == NST ? 0 : stage + 1;
            GFE_CLK(7);   // (debug build: the refill alone; the unit tail is not clocked then)
            // dB|dC rows of this CTA: add the warps' tiles; row layout {dB[n], dC[n]} interleaved
#pragma unroll
            for (int q = 0; q < BCC; ++q) {
                const int e = tid + q * NT, t = e >> 3, q8 = e & 7;
                if (tb + t < t1) {
                    const float4 *r = reinterpret_cast<const float4 *>(sRed + t * kCRedRow) + q8;
                    constexpr int W4 = kChunk * kCRedRow / 4;
                    float4 acc = r[0];
#pragma unroll
                    for (int w = 1; w < NW; ++w) {
                        const float4 x = r[w * W4];
                        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
                    }
                    __stcs(reinterpret_cast<float4 *>(p.part_bc + (((size_t)blk * p.B + b) * p.L + tb + t) * 32) + q8, acc);
                }
            }
            GFE_CLK(4);
            if (i + 1 < nch) phase_a_any(i + 1, stage);
            GFE_CLK(5);
        }

        // ---- end of unit: parameter-gradient partials, carry-out ----
        {
            float *dst = p.part_par + ((size_t)(b * cs.nseg + seg) * 18) * p.ED + c0 + 2 * rp;
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                dst[(size_t)(4 * rq + sw) * p.ED + ch] = dA[ch][0].x;
                dst[(size_t)(4 * rq + 1 - sw) * p.ED + ch] = dA[ch][0].y;
                dst[(size_t)(4 * rq + 2 + sw) * p.ED + ch] = dA[ch][1].x;
                dst[(size_t)(4 * rq + 3 - sw) * p.ED + ch] = dA[ch][1].y;
            }
        }
        // dD, ddt_bias: add the four item rows (cr) of each pair inside the warp
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
            dD_acc.x += __shfl_xor_sync(0xffffffffu, dD_acc.x, o);
            dD_acc.y += __shfl_xor_sync(0xffffffffu, dD_acc.y, o);
            dbias_acc.x += __shfl_xor_sync(0xffffffffu, dbias_acc.x, o);
            dbias_acc.y += __shfl_xor_sync(0xffffffffu, dbias_acc.y, o);
        }
        if (cr == 0) {
            float *dst = p.part_par + ((size_t)(b * cs.nseg + seg) * 18) * p.ED + c0 + 2 * cp;
            *reinterpret_cast<float2 *>(dst + (size_t)16 * p.ED) = dD_acc;
            *reinterpret_cast<float2 *>(dst + (size_t)17 * p.ED) = dbias_acc;
        }
        if (seg > 0 && !cs.independent) {
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                const float4 gv = sw ? make_float4(G[ch][0].y, G[ch][0].x, G[ch][1].y, G[ch][1].x)
                                     : make_float4(G[ch][0].x, G[ch][0].y, G[ch][1].x, G[ch][1].y);
                __stcg(reinterpret_cast<float4 *>(carry + ch * kNState), gv);
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) st_release(cs.flags + unit, 1);
        }
        cp_async_wait<0>();
        GFE_CLK(0);
    }
#ifdef GFE_PHASE_CLOCKS
    if ((threadIdx.x & 31) == 0)
        for (int i = 0; i < 8; ++i) atomicAdd(&g_bwd_phase_clk[i], (unsigned long long)clk_acc[i]);
#endif
}

#ifdef GFE_PHASE_CLOCKS
extern "C" __attribute__((visibility("default"))) int gfe_debug_bwd_phase_clocks(unsigned long long *out, int reset) {
    if (out) cudaMemcpyFromSymbol(out, g_bwd_phase_clk, sizeof(g_bwd_phase_clk));
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_bwd_phase_clk, z, sizeof(z)); }
    return 0;
}
#endif

// ---------------------------------------------------------------------------------------------------- host
struct BwdWs {
    size_t part_bc, part_par, total;
};
static BwdWs bwd_ws(int B, int L, int ED) {
    const ChainPlan pl = chain_bwd_plan(B, L, ED);
    BwdWs w{};
    size_t off = chain_bytes(B, ED, pl);
    w.part_bc = off;
    off += align_up((size_t)pl.nblk * B * L * 32 * sizeof(float), 256);
    w.part_par = off;
    off += align_up((size_t)B * pl.nseg * 18 * ED * sizeof(float), 256);
    w.total = off;
    return w;
}

size_t chain_bwd_workspace_bytes(int B, int L, int ED) { return bwd_ws(B, L, ED).total; }

template <typename T, bool HAS_Z, int CPB, int CPC>
static void launch_bwd_chain_inst(const ScanParams &p, const ChainSched &cs, cudaStream_t st) {
    constexpr size_t smem = BwdChainSmem<T, HAS_Z, CPC>::kTotal;
    const int grid = persistent_grid<selscan_bwd_chain_kernel<T, HAS_Z, CPB, CPC>>(2 * CPC, smem, cs.total);
    selscan_bwd_chain_kernel<T, HAS_Z, CPB, CPC><<<grid, 2 * CPC, smem, st>>>(p, cs);
}

template <typename T, int CPC>
static void launch_bwd_chain_cpc(const ScanParams &p, const ChainSched &cs, bool has_z, int cpb, cudaStream_t st) {
    if (has_z) {
        if (cpb == 16) launch_bwd_chain_inst<T, true, 16, CPC>(p, cs, st);
        else launch_bwd_chain_inst<T, true, 0, CPC>(p, cs, st);
    } else {
        if (cpb == 16) launch_bwd_chain_inst<T, false, 16, CPC>(p, cs, st);
        else launch_bwd_chain_inst<T, false, 0, CPC>(p, cs, st);
    }
}

template <typename T>
static int launch_bwd_chain_t(const gfe_selscan_args *a, cudaStream_t st) {
    const ChainPlan pl = chain_bwd_plan(a->batch, a->seqlen, a->d_inner);
    const int cpc = pl.cpc, nblk = pl.nblk, nseg = pl.nseg;
    const BwdWs w = bwd_ws(a->batch, a->seqlen, a->d_inner);
    if (a->ws == nullptr || a->ws_bytes < w.total) {
        set_error("selscan_bwd: workspace too small (%zu < %zu)", a->ws ? a->ws_bytes : (size_t)0, w.total);
        return GFE_ERR_WORKSPACE;
    }
    int rc = chain_check_alignment(a);
    if (rc != GFE_OK) return rc;
    ScanParams p{};
    chain_fill_params(p, a);
    char *ws = reinterpret_cast<char *>(a->ws);
    p.part_bc = reinterpret_cast<float *>(ws + w.part_bc);
    p.part_par = reinterpret_cast<float *>(ws + w.part_par);
    p.dout = a->dout; p.do_bs = a->dout_bs; p.do_rs = a->dout_rs;
    p.du = a->du; p.du_bs = a->du_bs; p.du_rs = a->du_rs;
    p.ddelta = a->ddelta; p.dd_bs = a->ddelta_bs; p.dd_rs = a->ddelta_rs;
    p.dz = a->dz; p.dz_bs = a->dz_bs; p.dz_rs = a->dz_rs;
    p.dBm = a->dBm; p.dB_bs = a->dB_bs; p.dB_rs = a->dB_rs;
    p.dCm = a->dCm; p.dC_bs = a->dC_bs; p.dC_rs = a->dC_rs;
    p.dA_log = a->dA_log; p.dD = a->dD; p.ddt_bias = a->ddt_bias;
    p.nseg = nseg;   // finalize_par sums over B * nseg partial rows
    p.G = nblk;      // finalize_bc sums one row per channel block
    p.bc_interleaved = 1;
    ChainSched cs{};
    rc = chain_fill_sched(cs, ws, a->batch, a->d_inner, pl, st);
    if (rc != GFE_OK) return rc;
    const int cpb = (chain_cpb(a, true) == 16 && chain_pair_stores(a, true)) ? 16 : 0;   // 16: cp.async staging AND paired stores
    if (pl.independent && nseg > 1) {
        ScopedKernelTimer tm(K_SELSCAN_BWD_SUMMARY, st);
        rc = seg_launch_carries(p, cs, a->dtype, cpc, true, a->z != nullptr, cpb, st);
        if (rc != GFE_OK) return rc;
    }
    {
        ScopedKernelTimer tm(K_SELSCAN_BWD, st);
        const bool hz = a->z != nullptr;
        if (cpc == 64) launch_bwd_chain_cpc<T, 64>(p, cs, hz, cpb, st);
        else launch_bwd_chain_cpc<T, 32>(p, cs, hz, cpb, st);   // (16-channel blocks measured slower; not instantiated)
    }
    rc = check_launch("selscan_bwd (chained)");
    if (rc != GFE_OK) return rc;
    launch_bwd_finalize(a, p, st, rc);
    return rc;
}

int chain_launch_bwd(const gfe_selscan_args *a, cudaStream_t st) {
    switch (a->dtype) {
        case GFE_F32: return launch_bwd_chain_t<float>(a, st);
        case GFE_BF16: return launch_bwd_chain_t<__nv_bfloat16>(a, st);
        default: return launch_bwd_chain_t<__half>(a, st);
    }
}

}  // namespace gfe
