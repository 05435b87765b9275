// selscan_chain_host.cu -- host side of the chained selective-scan kernels (selscan_v4_fwd.cu, selscan_chain_bwd.cu):
// the launch plan (channel-block width, L-segments), the workspace layout of the chain scheduler, argument checks and
// the forward dispatch.  Everything here is a pure function of the shape and the current device, so the size queries of
// the C ABI and the launches always agree.
#include "common.cuh"
#include "selscan_shared.cuh"

namespace gfe {

template <typename T>
void v4_launch_fwd_kernel(const ScanParams &p, const ChainSched &cs, int cpc, bool has_z, int cpb, cudaStream_t st);   // selscan_v4_fwd.cu

int seg_launch_carries(const ScanParams &p, const ChainSched &cs, int dtype, int cpc, bool rev, bool has_z, int cpb, cudaStream_t st);   // selscan_seg.cu
int seg_launch_total(const ScanParams &p, const ChainSched &cs, int dtype, int cpc, bool rev, bool has_z, int cpb, float *out,
                     float *sum_delta, cudaStream_t st);   // selscan_seg.cu

// L is cut into chained segments, ~12 units per resident CTA: the units of a chain interleave with those of the others and
// hop between SMs, which evens out SMs that host 2 and 3 working CTAs (measured on cfg3, profiles/r02_chain_variants.txt:
// 10-16 segments beat 1, 4 and 32 by 2-4 %).  Independent segments (too few chains to fill the GPU) only need enough units
// for the dynamic scheduler to balance the resident CTAs: 2 per CTA (2 / 3 / 6 measured on cfg4, 2 fastest by 1-3 %).
static void chain_plan(int B, int L, int nblk, int ctas_per_sm, bool independent, int &nseg, int &seg_len) {
    const int64_t slots = (int64_t)sm_count() * ctas_per_sm;
    int64_t want = ceil_div64((independent ? 2 : 12) * slots, (int64_t)B * nblk);
    const int64_t max_by_len = L / (8 * kChunk) > 0 ? L / (8 * kChunk) : 1;   // >= 128 steps per segment
    if (want > max_by_len) want = max_by_len;
    if (want > kMaxSeg) want = kMaxSeg;
    if (want < 1) want = 1;
    seg_len = (int)ceil_div64(ceil_div64(L, want), kChunk) * kChunk;
    nseg = (L + seg_len - 1) / seg_len;
}

// Channel-block width of both directions: 64 when it divides ED, else 32 (16 / 32 / 64 measured on cfg3 and cfg5: 64 is
// never slower, profiles/r02_chain_variants.txt).
static int chain_cpc(int ED) { return ED % 64 == 0 ? 64 : 32; }

// Chains wait for their predecessor segment when B * ED alone fills the GPU (plan_segments: at least half the schedulers
// get a warp without splitting L); otherwise the segments are made independent by a summary + combine pass.
static bool chain_independent(int B, int L, int ED) { return plan_segments(B, L, ED).nseg > 1; }

ChainPlan chain_fwd_plan(int B, int L, int ED) {
    ChainPlan pl{};
    pl.cpc = chain_cpc(ED);
    pl.nblk = ED / pl.cpc;
    pl.independent = chain_independent(B, L, ED) ? 1 : 0;
    chain_plan(B, L, pl.nblk, kFwdMinBlocks * (64 / pl.cpc), pl.independent, pl.nseg, pl.seg_len);
    return pl;
}
ChainPlan chain_bwd_plan(int B, int L, int ED) {
    ChainPlan pl{};
    pl.cpc = chain_cpc(ED);
    pl.nblk = ED / pl.cpc;
    pl.independent = chain_independent(B, L, ED) ? 1 : 0;
    chain_plan(B, L, pl.nblk, kBwdMinBlocks * (64 / pl.cpc), pl.independent, pl.nseg, pl.seg_len);
    return pl;
}

// The chained kernels serve every shape with d_state = 16 and ED % 32 == 0 (other widths and state sizes take the generic
// kernels in selscan.cu).
bool chain_applicable(int B, int L, int ED, int N) {
    (void)B; (void)L;
    return N == kNState && ED % 32 == 0;
}

struct ChainLayout {
    size_t counter, flags, carry, segsd, total;
};
static ChainLayout chain_layout(int B, int ED, const ChainPlan &pl) {
    ChainLayout c{};
    size_t off = 0;
    c.counter = off;   // [0]: main pass, [16]: summary pass
    off += 256;
    c.flags = off;
    off += align_up(pl.independent ? 0 : (size_t)pl.nseg * B * pl.nblk * sizeof(int), 256);
    c.carry = off;     // chained: [B][ED][16]; independent: [nseg - 1][B][ED][16] followed by sum(delta) [nseg - 1][B][ED]
    off += align_up((size_t)(pl.independent ? pl.nseg - 1 : 1) * B * ED * kNState * sizeof(float), 256);
    c.segsd = off;
    off += align_up(pl.independent ? (size_t)(pl.nseg - 1) * B * ED * sizeof(float) : 0, 256);
    c.total = off;
    return c;
}

size_t chain_bytes(int B, int ED, const ChainPlan &pl) { return chain_layout(B, ED, pl).total; }

size_t chain_fwd_workspace_bytes(int B, int L, int ED) { return chain_layout(B, ED, chain_fwd_plan(B, L, ED)).total; }

int chain_fill_sched(ChainSched &cs, char *ws, int B, int ED, const ChainPlan &pl, cudaStream_t st) {
    const ChainLayout cl = chain_layout(B, ED, pl);
    cs.counter = reinterpret_cast<int *>(ws + cl.counter);
    cs.flags = reinterpret_cast<int *>(ws + cl.flags);
    cs.carry = reinterpret_cast<float *>(ws + cl.carry);
    cs.nseg = pl.nseg;
    cs.seg_len = pl.seg_len;
    cs.nblk = pl.nblk;
    cs.total = pl.nseg * B * pl.nblk;
    cs.independent = pl.independent;
    cs.segc = cs.carry;
    cs.segsd = reinterpret_cast<float *>(ws + cl.segsd);
    if (cudaMemsetAsync(ws, 0, cl.carry, st) != cudaSuccess) return check_launch("selscan chain memset");
    return GFE_OK;
}

// the chained kernels read D / dt_bias two channels at a time and the checkpoints as float4
int chain_check_alignment(const gfe_selscan_args *a) {
    if ((reinterpret_cast<uintptr_t>(a->D) & 7) != 0 || (a->dt_bias && (reinterpret_cast<uintptr_t>(a->dt_bias) & 7) != 0)) {
        set_error("selscan: D and dt_bias must be 8-byte aligned");
        return GFE_ERR_ARG;
    }
    if (a->ckpt && (reinterpret_cast<uintptr_t>(a->ckpt) & 15) != 0) {
        set_error("selscan: ckpt must be 16-byte aligned");
        return GFE_ERR_ARG;
    }
    if (a->last_state && (reinterpret_cast<uintptr_t>(a->last_state) & 15) != 0) {
        set_error("selscan: last_state must be 16-byte aligned");
        return GFE_ERR_ARG;
    }
    return GFE_OK;
}

size_t chain_ckpt_state_bytes(int B, int L, int ED, int dtype) {   // [b][t / 8][c][16], fp32 (bf16 for bf16 activations), 256-byte padded
    const size_t el = dtype == GFE_BF16 ? 2 : 4;
    return align_up((size_t)B * ((L + kCkptV2 - 1) / kCkptV2) * ED * kNState * el, 256);
}

void chain_fill_params(ScanParams &p, const gfe_selscan_args *a) {
    p.B = a->batch; p.L = a->seqlen; p.ED = a->d_inner;
    p.nseg = 1; p.seg_len = a->seqlen; p.nchunks = (a->seqlen + kCkptV2 - 1) / kCkptV2;   // number of checkpoints: [b][t / 8][c][16]
    p.flags = a->flags;
    p.u = a->u; p.delta = a->delta; p.z = a->z; p.Bm = a->Bm; p.Cm = a->Cm;
    p.u_bs = a->u_bs; p.u_rs = a->u_rs; p.d_bs = a->delta_bs; p.d_rs = a->delta_rs;
    p.z_bs = a->z_bs; p.z_rs = a->z_rs; p.B_bs = a->B_bs; p.B_rs = a->B_rs; p.C_bs = a->C_bs; p.C_rs = a->C_rs;
    p.A_log = a->A_log; p.D = a->D; p.dt_bias = a->dt_bias;
    p.ckpt = reinterpret_cast<float2 *>(a->ckpt);
    p.ysave = a->ckpt ? reinterpret_cast<char *>(a->ckpt) + chain_ckpt_state_bytes(a->batch, a->seqlen, a->d_inner, a->dtype) : nullptr;
    p.G = a->d_inner / 32;
}

// 16 when every staged tensor can be moved in 16-byte cp.async pieces, else 0 (plain loads)
int chain_cpb(const gfe_selscan_args *a, bool bwd) {
    const int64_t s = a->dtype == GFE_F32 ? 4 : 2;
    const void *ptrs[6] = {a->u, a->delta, a->z, a->Bm, a->Cm, bwd ? a->dout : nullptr};
    const int64_t strides[12] = {a->u_bs, a->u_rs, a->delta_bs, a->delta_rs, a->z ? a->z_bs : 0, a->z ? a->z_rs : 0,
                                 a->B_bs, a->B_rs, a->C_bs, a->C_rs, bwd ? a->dout_bs : 0, bwd ? a->dout_rs : 0};
    bool ok = true;
    for (const void *q : ptrs) ok &= (reinterpret_cast<uintptr_t>(q) & 15) == 0;
    for (int64_t stv : strides) ok &= (stv * s) % 16 == 0;
    if (a->ckpt) ok &= (reinterpret_cast<uintptr_t>(a->ckpt) & 15) == 0;
    return ok ? 16 : 0;
}

// outputs may be written two channels at a time when every base and stride keeps the pair aligned
bool chain_pair_stores(const gfe_selscan_args *a, bool bwd) {
    const int64_t s = a->dtype == GFE_F32 ? 4 : 2;
    const int64_t al = 2 * s;
    bool ok = true;
    auto chk = [&](const void *q, int64_t bs, int64_t rs) {
        if (q == nullptr) return;
        ok &= (reinterpret_cast<uintptr_t>(q) % al) == 0 && (bs * s) % al == 0 && (rs * s) % al == 0;
    };
    if (bwd) {
        chk(a->du, a->du_bs, a->du_rs);
        chk(a->ddelta, a->ddelta_bs, a->ddelta_rs);
        chk(a->dz, a->dz_bs, a->dz_rs);
    } else {
        chk(a->out, a->out_bs, a->out_rs);
    }
    return ok;
}

template <typename T>
static int launch_fwd_chain_t(const gfe_selscan_args *a, const float *h0, cudaStream_t st) {
    const ChainPlan pl = chain_fwd_plan(a->batch, a->seqlen, a->d_inner);
    const size_t need = chain_bytes(a->batch, a->d_inner, pl);
    if (a->ws == nullptr || a->ws_bytes < need) {
        set_error("selscan_fwd: workspace too small (%zu < %zu)", a->ws ? a->ws_bytes : (size_t)0, need);
        return GFE_ERR_WORKSPACE;
    }
    int rc = chain_check_alignment(a);
    if (rc != GFE_OK) return rc;
    ScanParams p{};
    chain_fill_params(p, a);
    p.out = a->out; p.o_bs = a->out_bs; p.o_rs = a->out_rs; p.last_state = a->last_state; p.h0 = h0;
    ChainSched cs{};
    rc = chain_fill_sched(cs, reinterpret_cast<char *>(a->ws), a->batch, a->d_inner, pl, st);
    if (rc != GFE_OK) return rc;
    const int cpb = (chain_cpb(a, false) == 16 && chain_pair_stores(a, false)) ? 16 : 0;   // 16: cp.async staging AND paired stores
    if (pl.independent && pl.nseg > 1) {
        ScopedKernelTimer tm(K_SELSCAN_FWD_SUMMARY, st);
        rc = seg_launch_carries(p, cs, a->dtype, pl.cpc, false, false, cpb, st);
        if (rc != GFE_OK) return rc;
    }
    {
        ScopedKernelTimer tm(K_SELSCAN_FWD, st);
        v4_launch_fwd_kernel<T>(p, cs, pl.cpc, a->z != nullptr, cpb, st);
    }
    return check_launch("selscan_fwd (chained)");
}

int chain_launch_fwd(const gfe_selscan_args *a, const float *h0, cudaStream_t st) {
    switch (a->dtype) {
        case GFE_F32: return launch_fwd_chain_t<float>(a, h0, st);
        case GFE_BF16: return launch_fwd_chain_t<__nv_bfloat16>(a, h0, st);
        default: return launch_fwd_chain_t<__half>(a, h0, st);
    }
}

// ---- the summary of a whole range (gfe_selscan_summary_fwd / _bwd) ----
// Independent segments for every B * ED, cut as for the forward's summary pass; both directions take the same plan, so one
// workspace query serves both.  Workspace: the unit counter, then nseg slots of local aggregates [nseg][B][ED][16] and of
// sum(delta) [nseg][B][ED].
static ChainPlan chain_summary_plan(int B, int L, int ED) {
    ChainPlan pl{};
    pl.cpc = chain_cpc(ED);
    pl.nblk = ED / pl.cpc;
    pl.independent = 1;
    chain_plan(B, L, pl.nblk, kFwdMinBlocks * (64 / pl.cpc), true, pl.nseg, pl.seg_len);
    return pl;
}

struct SummaryLayout {
    size_t counter, segc, segsd, total;
};
static SummaryLayout chain_summary_layout(int B, int ED, const ChainPlan &pl) {
    SummaryLayout c{};
    size_t off = 256;   // counter
    c.segc = off;
    off += align_up((size_t)pl.nseg * B * ED * kNState * sizeof(float), 256);
    c.segsd = off;
    off += align_up((size_t)pl.nseg * B * ED * sizeof(float), 256);
    c.total = off;
    return c;
}

size_t chain_summary_workspace_bytes(int B, int L, int ED) { return chain_summary_layout(B, ED, chain_summary_plan(B, L, ED)).total; }

int chain_launch_summary(const gfe_selscan_args *a, bool rev, float *out, float *sum_delta, cudaStream_t st) {
    const ChainPlan pl = chain_summary_plan(a->batch, a->seqlen, a->d_inner);
    const SummaryLayout cl = chain_summary_layout(a->batch, a->d_inner, pl);
    const char *who = rev ? "selscan_summary_bwd" : "selscan_summary_fwd";
    if (a->ws == nullptr || a->ws_bytes < cl.total) {
        set_error("%s: workspace too small (%zu < %zu)", who, a->ws ? a->ws_bytes : (size_t)0, cl.total);
        return GFE_ERR_WORKSPACE;
    }
    if (a->dt_bias && (reinterpret_cast<uintptr_t>(a->dt_bias) & 7) != 0) {   // read two channels at a time
        set_error("%s: dt_bias must be 8-byte aligned", who);
        return GFE_ERR_ARG;
    }
    ScanParams p{};
    chain_fill_params(p, a);
    if (rev) { p.dout = a->dout; p.do_bs = a->dout_bs; p.do_rs = a->dout_rs; }
    else p.z = nullptr;   // the forward summary never reads z
    char *ws = reinterpret_cast<char *>(a->ws);
    ChainSched cs{};
    cs.counter = reinterpret_cast<int *>(ws + cl.counter);
    cs.segc = cs.carry = reinterpret_cast<float *>(ws + cl.segc);
    cs.segsd = reinterpret_cast<float *>(ws + cl.segsd);
    cs.nseg = pl.nseg;
    cs.seg_len = pl.seg_len;
    cs.nblk = pl.nblk;
    cs.independent = 1;
    if (cudaMemsetAsync(cs.counter, 0, sizeof(int), st) != cudaSuccess) return check_launch("selscan summary memset");
    gfe_selscan_args b = *a;   // staging checks of the tensors this direction reads
    if (rev) { b.u = nullptr; b.Bm = nullptr; }
    else { b.z = nullptr; b.Cm = nullptr; }
    b.ckpt = nullptr;
    const int cpb = chain_cpb(&b, rev);
    return seg_launch_total(p, cs, a->dtype, pl.cpc, rev, rev && a->z != nullptr, cpb, out, sum_delta, st);
}

}  // namespace gfe
