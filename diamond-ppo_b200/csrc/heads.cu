// Output heads, PPO loss and its gradient (diamond/ppo.py:261-280, continuous_ppo.py:273-292).
//
// One warp owns one minibatch row at a time.  The two head products (actor [A,H], critic [1,H])
// are far too thin for a GEMM tile (A <= 32), so the warp keeps the row's two H-wide activations in
// registers (lane k owns columns k, k+32, ...), forms the A+1 dot products with shuffles, evaluates
// the distribution with lane a <-> action a, and immediately back-propagates into the
// pre-activation gradient of the first head layers (the tanh' factor is applied here).  Weight /
// bias gradients of the heads, the bias gradient of the first head layers and the three loss sums
// are accumulated per CTA and written as one partial per CTA (summed in fixed order later).
#include <math_constants.h>

#include "common.cuh"
#include "heads.cuh"

namespace {

struct RowTerms {
    float policy;      // max(-A r, -A clamp(r))
    float dlogp;       // d(loss)/d(new_log_prob), already scaled by 1/M
};

// ppo.py:266-270 and the gradient torch autograd assigns (see oracle/ppo_oracle.py loss_and_grads)
__device__ __forceinline__ RowTerms policy_terms(float new_lp, float old_lp, float adv, float clip, float inv_m)
{
    const float ratio = expf(new_lp - old_lp);
    const float lo = 1.0f - clip, hi = 1.0f + clip;
    const float s1 = -adv * ratio;
    const float s2 = -adv * fminf(fmaxf(ratio, lo), hi);
    const bool in_range = ratio >= lo && ratio <= hi;
    const float w1 = in_range ? 1.0f : (s1 > s2 ? 1.0f : (s1 == s2 ? 0.5f : 0.0f));
    RowTerms t;
    t.policy = fmaxf(s1, s2);
    t.dlogp = (-adv * w1 * inv_m) * ratio;
    return t;
}

__device__ __forceinline__ void adv_norm_consts(const double* stats, int64_t count, int enabled, float& mean, float& denom)
{
    mean = 0.f; denom = 1.f;
    if (enabled) {
        const double mu = stats[0] / (double)count;
        double var = (stats[1] - stats[0] * mu) / (double)(count - 1);
        var = var > 0.0 ? var : 0.0;
        mean = (float)mu;
        denom = (float)sqrt(var) + 1e-6f;                 // ppo.py:243
    }
}

// Distribution evaluation with lane a <-> action a.  z: this lane's head output (logit / mean).
// Returns new_log_prob and entropy (warp-uniform); dz_scale_* let the caller form d(loss)/dz.
template <bool CONT>
struct Dist {
    float new_lp, entropy;
    float p, lsm;          // discrete: softmax prob / normalised logit of this lane
    float diff, var;       // gaussian: (a - mu), sigma^2 of this lane
};

template <bool CONT>
__device__ __forceinline__ Dist<CONT> eval_dist(float z, int lane, int A, int act_i, float act_f, float log_std)
{
    Dist<CONT> d;
    const bool on = lane < A;
    if (!CONT) {
        // torch/distributions/categorical.py:78 (logits - logsumexp), :151-163 (log_prob, entropy)
        const float zz = on ? z : -CUDART_INF_F;
        const float mx = warp_max(zz);
        const float e = on ? expf(zz - mx) : 0.f;
        const float s = warp_sum(e);
        const float lse = mx + logf(s);
        d.lsm = on ? z - lse : 0.f;
        d.p = on ? expf(d.lsm) : 0.f;
        d.entropy = -warp_sum(on ? d.p * d.lsm : 0.f);
        d.new_lp = __shfl_sync(0xffffffffu, d.lsm, act_i);
        d.diff = d.var = 0.f;
    } else {
        // torch/distributions/normal.py:87-102, :114-115, summed over dims (continuous_ppo.py:40-47)
        const float sigma = expf(log_std);
        const float log_scale = logf(sigma);
        d.var = sigma * sigma;
        d.diff = act_f - z;
        const float lp = on ? (-(d.diff * d.diff) / (2.0f * d.var) - log_scale - 0.91893853320467274178f) : 0.f;
        d.new_lp = warp_sum(lp);
        d.entropy = warp_sum(on ? (0.5f + 0.91893853320467274178f + log_scale) : 0.f);
        d.p = d.lsm = 0.f;
    }
    return d;
}

// Per-CTA partial [dWa A*H | dba A | dWc H | dbc 1 | dlog_std A | db3 2H | losses 4] (head_offsets): sums the per-warp
// accumulators held in s_acc ([HEAD_WARPS][(A+1)][H]) and the per-lane sums in fixed order and writes one partial per CTA.
template <int KPL, int VEC>
__device__ __forceinline__ void head_train_flush(const HeadTrainArgs& a, float* s_acc, const float (&acc_b3)[2 * KPL], float acc_dba,
                                                 float acc_dbc, float acc_dls, float l_pol, float l_val, float l_ent)
{
    const int H = a.H, A = a.A;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    auto kof = [&](int e) { return VEC == 4 ? ((e >> 2) * 128 + 4 * lane + (e & 3)) : lane + 32 * e; };
    __syncthreads();
    float* out = a.partials + (int64_t)blockIdx.x * a.partial_stride;
    for (int i = threadIdx.x; i < (A + 1) * H; i += blockDim.x) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < HEAD_WARPS; ++w) s += s_acc[(size_t)w * (A + 1) * H + i];
        if (i < A * H) out[i] = s; else out[head_offsets(H, A).dwc + (i - A * H)] = s;
    }
    __syncthreads();
    // reuse s_acc as scratch for the small per-warp vectors
    float* scratch = s_acc;                    // [HEAD_WARPS][2H + 3*32 + 4]
    const int sw = 2 * H + 100;
    float* mine = scratch + warp * sw;
#pragma unroll
    for (int i = 0; i < KPL; ++i) {
        const int k = kof(i);
        if (k < H) { mine[k] = acc_b3[i]; mine[H + k] = acc_b3[KPL + i]; }
    }
    mine[2 * H + lane] = acc_dba;
    mine[2 * H + 32 + lane] = acc_dls;
    if (lane == 0) {
        mine[2 * H + 64] = acc_dbc; mine[2 * H + 65] = l_pol; mine[2 * H + 66] = l_val; mine[2 * H + 67] = l_ent;
    }
    __syncthreads();
    const HeadOffsets ho = head_offsets(H, A);
    const int off_dba = ho.dba, off_dbc = ho.dbc, off_dls = ho.dls, off_b3 = ho.b3, off_loss = ho.loss;
    for (int i = threadIdx.x; i < 2 * H + 68; i += blockDim.x) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < HEAD_WARPS; ++w) s += scratch[w * sw + i];
        if (i < 2 * H) out[off_b3 + i] = s;
        else if (i < 2 * H + 32) { if (i - 2 * H < A) out[off_dba + (i - 2 * H)] = s; }
        else if (i < 2 * H + 64) { if (i - 2 * H - 32 < A) out[off_dls + (i - 2 * H - 32)] = s; }
        else if (i == 2 * H + 64) out[off_dbc] = s;
        else out[off_loss + (i - 2 * H - 65)] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// Training kernel: heads forward + loss + backward into the first head layers.
// ---------------------------------------------------------------------------------------------
// VEC == 4 (H a multiple of 128): lane owns columns 128*g + 4*lane + c and moves them as float4; VEC == 1: lane owns
// columns lane + 32*i.  R rows are in flight per warp iteration (their loads are issued together).
template <bool CONT, int KPL, int VEC, int R>
__global__ void __launch_bounds__(HEAD_WARPS * 32, 2)
head_train_kernel(HeadTrainArgs a)
{
    extern __shared__ float smem[];
    const int H = a.H, A = a.A;
    float* s_wa = smem;                         // [A][H]
    float* s_wc = s_wa + A * H;                 // [H]
    float* s_acc = s_wc + H;                    // [HEAD_WARPS][(A+1)][H]  per-warp dWa | dWc
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    DPPO_PDL_ENTER();
    for (int i = threadIdx.x; i < A * H; i += blockDim.x) s_wa[i] = a.wa[i];
    for (int i = threadIdx.x; i < H; i += blockDim.x) s_wc[i] = a.wc[i];
    float* acc = s_acc + (size_t)warp * (A + 1) * H;
    for (int i = lane; i < (A + 1) * H; i += 32) acc[i] = 0.f;
    __syncthreads();

    float mean, denom;
    adv_norm_consts(a.adv_stats, a.adv_count, a.advantage_norm, mean, denom);
    const float bias_a = lane < A ? a.ba[lane] : 0.f;
    const float bias_c = a.bc[0];
    const float log_std = (CONT && lane < A) ? a.log_std[lane] : 0.f;

    // column owned by element e of this lane
    auto kof = [&](int e) { return VEC == 4 ? ((e >> 2) * 128 + 4 * lane + (e & 3)) : lane + 32 * e; };

    float acc_b3[2 * KPL];
#pragma unroll
    for (int i = 0; i < 2 * KPL; ++i) acc_b3[i] = 0.f;
    float acc_dba = 0.f, acc_dbc = 0.f, acc_dls = 0.f;
    float l_pol = 0.f, l_val = 0.f, l_ent = 0.f;

    const int64_t warp_global = (int64_t)blockIdx.x * HEAD_WARPS + warp;
    const int64_t warp_stride = (int64_t)gridDim.x * HEAD_WARPS;
    for (int64_t mb = warp_global * R; mb < a.M; mb += warp_stride * R) {
        float ha[R][KPL], hc[R][KPL], old_lp[R], advv[R], ret[R], act_f[R];
        int act_i[R];
        bool live[R];                                                // false: padding row (idx < 0), contributes nothing
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int64_t m = mb + r;
            const bool ok = m < a.M;
            const int64_t sidx = ok ? (a.idx ? (int64_t)a.idx[m] : m) : 0;
            live[r] = ok && sidx >= 0;
            const int64_t src = live[r] ? sidx : 0;
            const float* h3 = a.h3 + (ok ? m : 0) * (int64_t)(2 * H);
            if (VEC == 4) {
#pragma unroll
                for (int g = 0; g < KPL / 4; ++g) {
                    const float4 va = ok ? __ldg(reinterpret_cast<const float4*>(h3 + g * 128) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 vc = ok ? __ldg(reinterpret_cast<const float4*>(h3 + H + g * 128) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
                    ha[r][4 * g] = va.x; ha[r][4 * g + 1] = va.y; ha[r][4 * g + 2] = va.z; ha[r][4 * g + 3] = va.w;
                    hc[r][4 * g] = vc.x; hc[r][4 * g + 1] = vc.y; hc[r][4 * g + 2] = vc.z; hc[r][4 * g + 3] = vc.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < KPL; ++i) {
                    const int k = lane + 32 * i;
                    ha[r][i] = (ok && k < H) ? __ldg(h3 + k) : 0.f;
                    hc[r][i] = (ok && k < H) ? __ldg(h3 + H + k) : 0.f;
                }
            }
            old_lp[r] = __ldg(a.old_logp + src);
            advv[r] = (__ldg(a.adv + src) - mean) / denom;
            ret[r] = __ldg(a.ret + src);
            act_i[r] = 0; act_f[r] = 0.f;
            if (CONT) act_f[r] = lane < A ? __ldg(a.actions_f + src * A + lane) : 0.f;
            else act_i[r] = __ldg(a.actions_i + src);
        }

#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int64_t m = mb + r;
            if (m >= a.M) break;                                     // warp-uniform
            // head products
            float z = 0.f;
            for (int j = 0; j < A; ++j) {
                float part = 0.f;
                if (VEC == 4) {
#pragma unroll
                    for (int g = 0; g < KPL / 4; ++g) {
                        const float4 w = reinterpret_cast<const float4*>(s_wa + j * H + g * 128)[lane];
                        part = fmaf(ha[r][4 * g], w.x, part); part = fmaf(ha[r][4 * g + 1], w.y, part);
                        part = fmaf(ha[r][4 * g + 2], w.z, part); part = fmaf(ha[r][4 * g + 3], w.w, part);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < KPL; ++e) {
                        const int k = kof(e);
                        if (k < H) part = fmaf(ha[r][e], s_wa[j * H + k], part);
                    }
                }
                part = warp_sum(part);
                if (lane == j) z = part;
            }
            z += bias_a;
            float vpart = 0.f;
            float wcv[KPL];                                          // this lane's critic-head weights
            if (VEC == 4) {
#pragma unroll
                for (int g = 0; g < KPL / 4; ++g) {
                    const float4 w = reinterpret_cast<const float4*>(s_wc + g * 128)[lane];
                    wcv[4 * g] = w.x; wcv[4 * g + 1] = w.y; wcv[4 * g + 2] = w.z; wcv[4 * g + 3] = w.w;
                }
            } else {
#pragma unroll
                for (int e = 0; e < KPL; ++e) wcv[e] = kof(e) < H ? s_wc[kof(e)] : 0.f;
            }
#pragma unroll
            for (int e = 0; e < KPL; ++e) vpart = fmaf(hc[r][e], wcv[e], vpart);
            const float v = warp_sum(vpart) + bias_c;

            const Dist<CONT> d = eval_dist<CONT>(z, lane, A, act_i[r], act_f[r], log_std);
            const RowTerms t = policy_terms(d.new_lp, old_lp[r], advv[r], a.clip, a.inv_m);
            float dz = 0.f;
            if (lane < A && live[r]) {
                if (!CONT) {
                    dz = t.dlogp * ((lane == act_i[r] ? 1.0f : 0.0f) - d.p) + (a.beta * a.inv_m) * d.p * (d.lsm + d.entropy);
                } else {
                    dz = t.dlogp * d.diff / d.var;
                    acc_dls += t.dlogp * (d.diff * d.diff / d.var - 1.0f) - a.beta * a.inv_m;
                }
            }
            const float verr = v - ret[r];
            const float dv = live[r] ? a.vw * verr * a.inv_m : 0.f;
            if (live[r]) { l_pol += t.policy; l_val += verr * verr; l_ent += d.entropy; }
            acc_dba += dz;
            acc_dbc += dv;

            // backward into the first head layers (+ head weight gradients)
            float ga[KPL];
#pragma unroll
            for (int e = 0; e < KPL; ++e) ga[e] = 0.f;
            for (int j = 0; j < A; ++j) {
                const float dzj = __shfl_sync(0xffffffffu, dz, j);
                if (VEC == 4) {
#pragma unroll
                    for (int g = 0; g < KPL / 4; ++g) {
                        const float4 w = reinterpret_cast<const float4*>(s_wa + j * H + g * 128)[lane];
                        ga[4 * g] = fmaf(dzj, w.x, ga[4 * g]); ga[4 * g + 1] = fmaf(dzj, w.y, ga[4 * g + 1]);
                        ga[4 * g + 2] = fmaf(dzj, w.z, ga[4 * g + 2]); ga[4 * g + 3] = fmaf(dzj, w.w, ga[4 * g + 3]);
                        float4* ap = reinterpret_cast<float4*>(acc + j * H + g * 128) + lane;
                        float4 av = *ap;
                        av.x = fmaf(dzj, ha[r][4 * g], av.x); av.y = fmaf(dzj, ha[r][4 * g + 1], av.y);
                        av.z = fmaf(dzj, ha[r][4 * g + 2], av.z); av.w = fmaf(dzj, ha[r][4 * g + 3], av.w);
                        *ap = av;
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < KPL; ++e) {
                        const int k = kof(e);
                        if (k < H) {
                            ga[e] = fmaf(dzj, s_wa[j * H + k], ga[e]);
                            acc[j * H + k] = fmaf(dzj, ha[r][e], acc[j * H + k]);
                        }
                    }
                }
            }
            float* d3 = a.d3 + m * (int64_t)(2 * H);
            float da[KPL], dc[KPL];
#pragma unroll
            for (int e = 0; e < KPL; ++e) {
                const int k = kof(e);
                da[e] = dc[e] = 0.f;
                if (VEC == 4 || k < H) {
                    da[e] = ga[e] * (1.0f - ha[r][e] * ha[r][e]);
                    dc[e] = dv * wcv[e] * (1.0f - hc[r][e] * hc[r][e]);
                    acc_b3[e] += da[e];
                    acc_b3[KPL + e] += dc[e];
                    if (VEC != 4) acc[A * H + k] = fmaf(dv, hc[r][e], acc[A * H + k]);
                }
            }
            if (VEC == 4) {
#pragma unroll
                for (int g = 0; g < KPL / 4; ++g) {
                    float4* ap = reinterpret_cast<float4*>(acc + A * H + g * 128) + lane;
                    float4 av = *ap;
                    av.x = fmaf(dv, hc[r][4 * g], av.x); av.y = fmaf(dv, hc[r][4 * g + 1], av.y);
                    av.z = fmaf(dv, hc[r][4 * g + 2], av.z); av.w = fmaf(dv, hc[r][4 * g + 3], av.w);
                    *ap = av;
                }
#pragma unroll
                for (int g = 0; g < KPL / 4; ++g) {
                    reinterpret_cast<float4*>(d3 + g * 128)[lane] = make_float4(da[4 * g], da[4 * g + 1], da[4 * g + 2], da[4 * g + 3]);
                    reinterpret_cast<float4*>(d3 + H + g * 128)[lane] = make_float4(dc[4 * g], dc[4 * g + 1], dc[4 * g + 2], dc[4 * g + 3]);
                }
            } else {
#pragma unroll
                for (int e = 0; e < KPL; ++e) {
                    const int k = lane + 32 * e;
                    if (k < H) { d3[k] = da[e]; d3[H + k] = dc[e]; }
                }
            }
        }
    }

    head_train_flush<KPL, VEC>(a, s_acc, acc_b3, acc_dba, acc_dbc, acc_dls, l_pol, l_val, l_ent);
}

// ---- packed fp32 arithmetic (sm_100 FFMA2 / FMUL2 / FADD2: two IEEE fp32 operations per instruction) -------------------------
// Element-wise results are identical to the scalar forms nvcc emits (fmaf, *, fma(-h, h, 1)); only dot4 changes the summation order (even and odd
// columns are accumulated separately and added at the end).
__device__ __forceinline__ void axpy4(float4& acc, float s, const float4& x)              // acc += s * x
{
    const float2 ss = make_float2(s, s);
    const float2 lo = __ffma2_rn(ss, make_float2(x.x, x.y), make_float2(acc.x, acc.y));
    const float2 hi = __ffma2_rn(ss, make_float2(x.z, x.w), make_float2(acc.z, acc.w));
    acc = make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ void dot4(float2& acc, const float4& a, const float4& b)       // acc.{x,y} += a.{x,y}*b.{x,y} + a.{z,w}*b.{z,w}
{
    acc = __ffma2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y), acc);
    acc = __ffma2_rn(make_float2(a.z, a.w), make_float2(b.z, b.w), acc);
}
__device__ __forceinline__ float4 mul4(const float4& a, const float4& b)
{
    const float2 lo = __fmul2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
    const float2 hi = __fmul2_rn(make_float2(a.z, a.w), make_float2(b.z, b.w));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ float4 scale4(float s, const float4& a) { return mul4(make_float4(s, s, s, s), a); }
__device__ __forceinline__ float4 one_minus_sq4(const float4& h)                           // fma(-h, h, 1), as nvcc contracts 1 - h*h
{
    const float2 one = make_float2(1.0f, 1.0f);
    const float2 lo = __ffma2_rn(make_float2(-h.x, -h.y), make_float2(h.x, h.y), one);
    const float2 hi = __ffma2_rn(make_float2(-h.z, -h.w), make_float2(h.z, h.w), one);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// ---------------------------------------------------------------------------------------------
// Role-split variant (H a multiple of 128, H <= 256, A <= 4).  The actor half of a row (policy loss, entropy, d3[:, :H], dWa)
// and the critic half (value loss, d3[:, H:], dWc) share nothing but the row index, so they are given to DIFFERENT warps:
// NA actor warps and HEAD_WARPS - NA critic warps per CTA walk the rows independently.  Neither role carries the other's
// accumulators (<= 96 registers, three CTAs per SM, nothing spilled), and the warp-wide reductions become multi-value
// butterflies: the 2 x 4 head products of an actor iteration are reduced with 9 shuffles into the lane layout
// (row = lane bit 4, action = lane bits 3:2) on which the distribution of BOTH rows is evaluated at once (softmax sums are two
// xor steps); a critic iteration reduces the values of 4 rows with 6 shuffles (row = lane bits 4:3).  Per-row scalars are
// loaded by the lanes that use them.  ~300 instructions per row against ~530 for the round-1 kernel that kept both halves of a row in one warp (ncu, config S:
// 76.6 -> 54.1 us per launch, 268 MB = 76 % of the HBM peak).
// Same per-element arithmetic; only the order of the reductions differs.
// ---------------------------------------------------------------------------------------------
constexpr int SPLIT_WARPS = 10;              // warps per CTA (two CTAs per SM at <= 96 registers)
constexpr int SPLIT_NA = 8;                  // actor warps (an actor row costs ~4x a critic row); the other warps take the critic role
template <bool CONT, int G>
__global__ void __launch_bounds__(SPLIT_WARPS * 32, 2)
head_train_split_kernel(HeadTrainArgs a)
{
    constexpr int NA = SPLIT_NA;
    extern __shared__ float smem[];
    constexpr int AM = 4;                       // action slots (rows of s_wa beyond A are zero)
    constexpr int H = 128 * G;
    const int A = a.A;
    constexpr int NC = SPLIT_WARPS - NA;
    float* s_wa = smem;                         // [AM][H]
    float* s_acc = s_wa + AM * H;               // actor warps: [NA][AM][H]; critic warps: [NC][H]; then per-warp tails [SPLIT_WARPS][H + 16]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    DPPO_PDL_ENTER();
    for (int i = threadIdx.x; i < AM * H; i += blockDim.x) s_wa[i] = i < A * H ? a.wa[i] : 0.f;
    __syncthreads();
    float* tails = s_acc + (NA * AM + NC) * H;
    float* tail = tails + warp * (H + 16);
    const uint64_t pol = l2_policy_evict_first();
    const bool h3_first = a.h3_first != 0;

    if (warp < NA) {
        // ------------------------------------------------ actor role: 2 rows per iteration
        const int rl = lane >> 4, jl = (lane >> 2) & 3;          // this lane's (row, action) in the reduced layout
        const bool on = jl < A;
        float mean, denom;
        adv_norm_consts(a.adv_stats, a.adv_count, a.advantage_norm, mean, denom);
        const float bias = on ? a.ba[jl] : 0.f;
        const float log_std = (CONT && on) ? a.log_std[jl] : 0.f;
        float4 gwa[AM][G];
#pragma unroll
        for (int j = 0; j < AM; ++j)
#pragma unroll
            for (int g = 0; g < G; ++g) gwa[j][g] = make_float4(0.f, 0.f, 0.f, 0.f);
        float4* accb = reinterpret_cast<float4*>(tail);         // column sums of d3[:, :H] (db3): this lane's columns, in shared memory
#pragma unroll
        for (int g = 0; g < G; ++g) accb[g * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
        float acc_dba = 0.f, acc_dls = 0.f, l_pol = 0.f, l_ent = 0.f;

        const int Mi = (int)a.M;
        const int nb = (Mi + 1) >> 1;                            // row pairs; a.rev: visited from the last to the first (L2 reuse)
        for (int b = blockIdx.x * NA + warp; b < nb; b += gridDim.x * NA) {
            const int mb = (a.rev ? nb - 1 - b : b) * 2;
            const bool ok1 = mb + 1 < Mi;
            float4 ha[2][G];
            {
                const float4* h0 = reinterpret_cast<const float4*>(a.h3 + (int64_t)mb * (2 * H));
                const float4* h1 = reinterpret_cast<const float4*>(a.h3 + (int64_t)(ok1 ? mb + 1 : mb) * (2 * H));
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    if (h3_first) { ha[0][g] = ldg_l2_hint(h0 + g * 32 + lane, pol); ha[1][g] = ldg_l2_hint(h1 + g * 32 + lane, pol); }
                    else { ha[0][g] = __ldg(h0 + g * 32 + lane); ha[1][g] = __ldg(h1 + g * 32 + lane); }
                }
            }
            // this lane's row scalars
            const int m = mb + rl;
            const bool okl = m < Mi;
            const int sidx = okl ? (a.idx ? __ldg(a.idx + m) : m) : 0;
            const bool live = okl && sidx >= 0;
            const int src = live ? sidx : 0;
            const float old_lp = __ldg(a.old_logp + src);
            const float advv = (__ldg(a.adv + src) - mean) / denom;
            int act_i = 0; float act_f = 0.f;
            if (CONT) act_f = on ? __ldg(a.actions_f + (int64_t)src * A + jl) : 0.f;
            else act_i = __ldg(a.actions_i + src);

            // head products: even / odd column partial sums (packed FFMA2), every weight vector read once for both rows
            float p[2][AM];
#pragma unroll
            for (int j = 0; j < AM; ++j) {
                float2 q0 = make_float2(0.f, 0.f), q1 = make_float2(0.f, 0.f);
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const float4 w = reinterpret_cast<const float4*>(s_wa + j * H + g * 128)[lane];
                    dot4(q0, ha[0][g], w); dot4(q1, ha[1][g], w);
                }
                p[0][j] = q0.x + q0.y; p[1][j] = q1.x + q1.y;
            }
            // butterfly: 8 values -> lane (row = bit 4, action = bits 3:2)
            float s1[AM];
            const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
#pragma unroll
            for (int j = 0; j < AM; ++j) {
                const float keep = b4 ? p[1][j] : p[0][j], send = b4 ? p[0][j] : p[1][j];
                s1[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
            float s2[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float keep = b3 ? s1[2 + j] : s1[j], send = b3 ? s1[j] : s1[2 + j];
                s2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            }
            float z;
            {
                const float keep = b2 ? s2[1] : s2[0], send = b2 ? s2[0] : s2[1];
                z = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
            z += __shfl_xor_sync(0xffffffffu, z, 2);
            z += __shfl_xor_sync(0xffffffffu, z, 1);
            z += bias;

            // distribution of both rows at once (reductions over the action bits: xor 4, xor 8)
            float new_lp, entropy, dz = 0.f, dls = 0.f, pj = 0.f, lsm = 0.f, diff = 0.f, var = 1.f;
            if (!CONT) {
                // torch/distributions/categorical.py:78 (logits - logsumexp), :151-163 (log_prob, entropy)
                const float zz = on ? z : -CUDART_INF_F;
                float mx = fmaxf(zz, __shfl_xor_sync(0xffffffffu, zz, 4));
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
                const float e = on ? expf(zz - mx) : 0.f;
                float s = e + __shfl_xor_sync(0xffffffffu, e, 4);
                s += __shfl_xor_sync(0xffffffffu, s, 8);
                const float lse = mx + logf(s);
                lsm = on ? z - lse : 0.f;
                pj = on ? expf(lsm) : 0.f;
                float en = on ? pj * lsm : 0.f;
                en += __shfl_xor_sync(0xffffffffu, en, 4);
                en += __shfl_xor_sync(0xffffffffu, en, 8);
                entropy = -en;
                new_lp = __shfl_sync(0xffffffffu, lsm, (lane & 16) | ((act_i & 3) << 2));
            } else {
                // torch/distributions/normal.py:87-102, :114-115, summed over dims (continuous_ppo.py:40-47)
                const float sigma = expf(log_std);
                const float log_scale = logf(sigma);
                var = sigma * sigma;
                diff = act_f - z;
                float lp = on ? (-(diff * diff) / (2.0f * var) - log_scale - 0.91893853320467274178f) : 0.f;
                lp += __shfl_xor_sync(0xffffffffu, lp, 4);
                lp += __shfl_xor_sync(0xffffffffu, lp, 8);
                new_lp = lp;
                float en = on ? (0.5f + 0.91893853320467274178f + log_scale) : 0.f;
                en += __shfl_xor_sync(0xffffffffu, en, 4);
                en += __shfl_xor_sync(0xffffffffu, en, 8);
                entropy = en;
            }
            const RowTerms t = policy_terms(new_lp, old_lp, advv, a.clip, a.inv_m);
            if (on && live) {
                if (!CONT) {
                    dz = t.dlogp * ((jl == act_i ? 1.0f : 0.0f) - pj) + (a.beta * a.inv_m) * pj * (lsm + entropy);
                } else {
                    dz = t.dlogp * diff / var;
                    dls = t.dlogp * (diff * diff / var - 1.0f) - a.beta * a.inv_m;
                }
            }
            if (live) { l_pol += t.policy; l_ent += entropy; }
            acc_dba += dz; acc_dls += dls;

            // backward into actor_head.0 + dWa
            float4 ga[2][G];
#pragma unroll
            for (int g = 0; g < G; ++g) { ga[0][g] = make_float4(0.f, 0.f, 0.f, 0.f); ga[1][g] = make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
            for (int j = 0; j < AM; ++j) {
                const float d0 = __shfl_sync(0xffffffffu, dz, j << 2), d1 = __shfl_sync(0xffffffffu, dz, 16 | (j << 2));
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const float4 w = reinterpret_cast<const float4*>(s_wa + j * H + g * 128)[lane];
                    axpy4(ga[0][g], d0, w); axpy4(ga[1][g], d1, w);
                    axpy4(gwa[j][g], d0, ha[0][g]); axpy4(gwa[j][g], d1, ha[1][g]);
                }
            }
            float* d3 = a.d3 + (int64_t)mb * (2 * H);
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const float4 da0 = mul4(ga[0][g], one_minus_sq4(ha[0][g]));
                const float4 da1 = mul4(ga[1][g], one_minus_sq4(ha[1][g]));
                if (a.keep_d3) {
                    reinterpret_cast<float4*>(d3 + g * 128)[lane] = da0;
                    if (ok1) reinterpret_cast<float4*>(d3 + 2 * H + g * 128)[lane] = da1;
                } else {
                    __stcs(reinterpret_cast<float4*>(d3 + g * 128) + lane, da0);
                    if (ok1) __stcs(reinterpret_cast<float4*>(d3 + 2 * H + g * 128) + lane, da1);
                }
                float4 t = accb[g * 32 + lane];
                const float2 lo = __fadd2_rn(make_float2(t.x, t.y), __fadd2_rn(make_float2(da0.x, da0.y), make_float2(da1.x, da1.y)));
                const float2 hi = __fadd2_rn(make_float2(t.z, t.w), __fadd2_rn(make_float2(da0.z, da0.w), make_float2(da1.z, da1.w)));
                accb[g * 32 + lane] = make_float4(lo.x, lo.y, hi.x, hi.y);
            }
        }
        // per-warp accumulators -> shared memory
        float* acc = s_acc + (size_t)warp * AM * H;
#pragma unroll
        for (int j = 0; j < AM; ++j)
#pragma unroll
            for (int g = 0; g < G; ++g) reinterpret_cast<float4*>(acc + j * H + g * 128)[lane] = gwa[j][g];
        acc_dba += __shfl_xor_sync(0xffffffffu, acc_dba, 16);
        acc_dls += __shfl_xor_sync(0xffffffffu, acc_dls, 16);
        l_pol += __shfl_xor_sync(0xffffffffu, l_pol, 16);
        l_ent += __shfl_xor_sync(0xffffffffu, l_ent, 16);
        if (lane < 16 && (lane & 3) == 0) { tail[H + jl] = acc_dba; tail[H + 4 + jl] = acc_dls; }
        if (lane == 0) { tail[H + 8] = l_pol; tail[H + 9] = l_ent; }
    } else {
        // ------------------------------------------------ critic role: 4 rows per iteration
        const int cw = warp - NA;
        const int rl = lane >> 3;
        const float bias_c = a.bc[0];
        float4 wcv[G], gwc[G];
        float2 accb[2 * G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            wcv[g] = __ldg(reinterpret_cast<const float4*>(a.wc + g * 128) + lane);
            gwc[g] = make_float4(0.f, 0.f, 0.f, 0.f);
            accb[2 * g] = make_float2(0.f, 0.f); accb[2 * g + 1] = make_float2(0.f, 0.f);
        }
        float acc_dbc = 0.f, l_val = 0.f;
        const int Mi = (int)a.M;
        const int nb = (Mi + 3) >> 2;                            // blocks of four rows, same sweep direction as the actor warps
        for (int b = blockIdx.x * NC + cw; b < nb; b += gridDim.x * NC) {
            const int mb = (a.rev ? nb - 1 - b : b) * 4;
            float4 hc[4][G];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int mr = mb + r < Mi ? mb + r : mb;
                const float4* h = reinterpret_cast<const float4*>(a.h3 + (int64_t)mr * (2 * H) + H);
#pragma unroll
                for (int g = 0; g < G; ++g) hc[r][g] = h3_first ? ldg_l2_hint(h + g * 32 + lane, pol) : __ldg(h + g * 32 + lane);
            }
            const int m = mb + rl;
            const bool okl = m < Mi;
            const int sidx = okl ? (a.idx ? __ldg(a.idx + m) : m) : 0;
            const bool live = okl && sidx >= 0;
            const float ret = __ldg(a.ret + (live ? sidx : 0));
            float p[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float2 q = make_float2(0.f, 0.f);
#pragma unroll
                for (int g = 0; g < G; ++g) dot4(q, hc[r][g], wcv[g]);
                p[r] = q.x + q.y;
            }
            const bool b4 = lane & 16, b3 = lane & 8;
            float s1[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float keep = b4 ? p[2 + r] : p[r], send = b4 ? p[r] : p[2 + r];
                s1[r] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
            float v;
            {
                const float keep = b3 ? s1[1] : s1[0], send = b3 ? s1[0] : s1[1];
                v = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            }
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += bias_c;
            const float verr = v - ret;
            float dv = 0.f;
            if (live) { dv = a.vw * verr * a.inv_m; l_val += verr * verr; }
            acc_dbc += dv;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float dvr = __shfl_sync(0xffffffffu, dv, r << 3);
                float* d3 = a.d3 + (int64_t)(mb + r) * (2 * H) + H;
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const float4 dc = mul4(scale4(dvr, wcv[g]), one_minus_sq4(hc[r][g]));
                    accb[2 * g] = __fadd2_rn(accb[2 * g], make_float2(dc.x, dc.y));
                    accb[2 * g + 1] = __fadd2_rn(accb[2 * g + 1], make_float2(dc.z, dc.w));
                    axpy4(gwc[g], dvr, hc[r][g]);
                    if (mb + r < Mi) {
                        if (a.keep_d3) reinterpret_cast<float4*>(d3 + g * 128)[lane] = dc;
                        else __stcs(reinterpret_cast<float4*>(d3 + g * 128) + lane, dc);
                    }
                }
            }
        }
        float* acc = s_acc + (size_t)NA * AM * H + (size_t)cw * H;
#pragma unroll
        for (int g = 0; g < G; ++g) {
            reinterpret_cast<float4*>(acc + g * 128)[lane] = gwc[g];
            reinterpret_cast<float4*>(tail + g * 128)[lane] = make_float4(accb[2 * g].x, accb[2 * g].y, accb[2 * g + 1].x, accb[2 * g + 1].y);
        }
        // one lane per row slot holds that slot's sums (lanes 0, 8, 16, 24)
        acc_dbc += __shfl_xor_sync(0xffffffffu, acc_dbc, 16); acc_dbc += __shfl_xor_sync(0xffffffffu, acc_dbc, 8);
        l_val += __shfl_xor_sync(0xffffffffu, l_val, 16); l_val += __shfl_xor_sync(0xffffffffu, l_val, 8);
        if (lane == 0) { tail[H + 10] = acc_dbc; tail[H + 11] = l_val; }
    }
    __syncthreads();

    // one partial per CTA, summed over the warps of a role in fixed order
    const HeadOffsets ho = head_offsets(H, A);
    float* out = a.partials + (int64_t)blockIdx.x * a.partial_stride;
    for (int i = threadIdx.x; i < A * H; i += blockDim.x) {
        float s = 0.f;
        for (int w = 0; w < NA; ++w) s += s_acc[(size_t)w * AM * H + i];
        out[i] = s;
    }
    for (int i = threadIdx.x; i < H; i += blockDim.x) {
        float s = 0.f, ba = 0.f, bc = 0.f;
        for (int w = 0; w < NC; ++w) { s += s_acc[(size_t)NA * AM * H + (size_t)w * H + i]; bc += tails[(NA + w) * (H + 16) + i]; }
        for (int w = 0; w < NA; ++w) ba += tails[w * (H + 16) + i];
        out[ho.dwc + i] = s; out[ho.b3 + i] = ba; out[ho.b3 + H + i] = bc;
    }
    if (threadIdx.x < 12) {
        const int i = threadIdx.x;                // 0..3 dba, 4..7 dls, 8 pol, 9 ent (actor warps); 10 dbc, 11 val (critic warps)
        float s = 0.f;
        if (i < 10) for (int w = 0; w < NA; ++w) s += tails[w * (H + 16) + H + i];
        else for (int w = 0; w < NC; ++w) s += tails[(NA + w) * (H + 16) + H + i];
        if (i < 4) { if (i < A) out[ho.dba + i] = s; }
        else if (i < 8) { if (i - 4 < A) out[ho.dls + (i - 4)] = s; }
        else if (i == 8) out[ho.loss] = s;
        else if (i == 9) out[ho.loss + 2] = s;
        else if (i == 10) out[ho.dbc] = s;
        else out[ho.loss + 1] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// Inference: head outputs (+ log-prob of given actions) for the pre-update pass and get_actions.
// ha/hc point at the first-head-layer activations (row stride ld); either may be null.
// ---------------------------------------------------------------------------------------------
template <int KPL>
__global__ void __launch_bounds__(256)
head_eval_kernel(const float* __restrict__ ha_base, const float* __restrict__ hc_base, int ld, const float* __restrict__ wa,
                 const float* __restrict__ ba, const float* __restrict__ wc, const float* __restrict__ bc,
                 float* __restrict__ head_out, float* __restrict__ values, int64_t rows, int H, int A, const int* __restrict__ rows_dev)
{
    extern __shared__ float smem[];
    if (rows_dev != nullptr && *rows_dev < rows) rows = *rows_dev;
    float* s_wa = smem;
    float* s_wc = smem + A * H;
    if (ha_base) for (int i = threadIdx.x; i < A * H; i += blockDim.x) s_wa[i] = wa[i];
    if (hc_base) for (int i = threadIdx.x; i < H; i += blockDim.x) s_wc[i] = wc[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t ws = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t m = w0; m < rows; m += ws) {
        if (ha_base) {
            float h[KPL];
#pragma unroll
            for (int i = 0; i < KPL; ++i) { const int k = lane + 32 * i; h[i] = k < H ? __ldg(ha_base + m * ld + k) : 0.f; }
            float z = 0.f;
            for (int j = 0; j < A; ++j) {
                float part = 0.f;
#pragma unroll
                for (int i = 0; i < KPL; ++i) { const int k = lane + 32 * i; if (k < H) part = fmaf(h[i], s_wa[j * H + k], part); }
                part = warp_sum(part);
                if (lane == j) z = part;
            }
            if (lane < A) head_out[m * A + lane] = z + ba[lane];
        }
        if (hc_base) {
            float part = 0.f;
#pragma unroll
            for (int i = 0; i < KPL; ++i) { const int k = lane + 32 * i; if (k < H) part = fmaf(__ldg(hc_base + m * ld + k), s_wc[k], part); }
            part = warp_sum(part);
            if (lane == 0) values[m] = part + bc[0];
        }
    }
}

// Vector variant of head_eval_kernel (H a multiple of 128, A <= 4, 16-byte aligned rows): four rows per warp iteration, float4 loads,
// packed FFMA2 dot products, and ONE multi-value butterfly for the 4 x (A + 1) partial sums instead of 5 shuffle trees per row:
// the 16 actor values end in the lane layout (row = lane bits 4:3, action = lane bits 2:1), the 4 critic values in (row = bits 4:3).
// The pre-update pass runs this kernel over every row of the rollout twice (ppo.py:235-238).
template <int G, bool ACTOR, bool CRITIC>
__global__ void __launch_bounds__(256)
head_eval_vec_kernel(const float* __restrict__ ha_base, const float* __restrict__ hc_base, int ld, const float* __restrict__ wa,
                     const float* __restrict__ ba, const float* __restrict__ wc, const float* __restrict__ bc,
                     float* __restrict__ head_out, float* __restrict__ values, int64_t rows, int A, int rev, const int* __restrict__ rows_dev)
{
    constexpr int H = 128 * G, AM = 4;
    __shared__ __align__(16) float s_wa[ACTOR ? AM * H : 4];
    if (rows_dev != nullptr && *rows_dev < rows) rows = *rows_dev;
    if (ACTOR) {
        for (int i = threadIdx.x; i < AM * H; i += blockDim.x) s_wa[i] = i < A * H ? wa[i] : 0.f;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    float4 wcv[G];
    if (CRITIC) {
#pragma unroll
        for (int g = 0; g < G; ++g) wcv[g] = __ldg(reinterpret_cast<const float4*>(wc + g * 128) + lane);
    }
    const int rl = lane >> 3, jl = (lane >> 1) & 3;              // this lane's (row, action) after the reduction
    const float bias_a = (ACTOR && jl < A) ? ba[jl] : 0.f;
    const float bias_c = CRITIC ? bc[0] : 0.f;
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ws = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nb = (rows + 3) >> 2;                          // blocks of four rows; rev: visited from the last to the first (L2 reuse)
    for (int64_t b = w0; b < nb; b += ws) {
        const int64_t mb = (rev ? nb - 1 - b : b) * 4;
        float pa[4][AM], pc[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int64_t m = mb + r < rows ? mb + r : mb;
            if (ACTOR) {
                float4 h[G];
                const float4* hp = reinterpret_cast<const float4*>(ha_base + m * ld);
#pragma unroll
                for (int g = 0; g < G; ++g) h[g] = __ldg(hp + g * 32 + lane);
#pragma unroll
                for (int j = 0; j < AM; ++j) {
                    float2 q = make_float2(0.f, 0.f);
#pragma unroll
                    for (int g = 0; g < G; ++g) dot4(q, h[g], reinterpret_cast<const float4*>(s_wa + j * H + g * 128)[lane]);
                    pa[r][j] = q.x + q.y;
                }
            }
            if (CRITIC) {
                const float4* hp = reinterpret_cast<const float4*>(hc_base + m * ld);
                float2 q = make_float2(0.f, 0.f);
#pragma unroll
                for (int g = 0; g < G; ++g) dot4(q, __ldg(hp + g * 32 + lane), wcv[g]);
                pc[r] = q.x + q.y;
            }
        }
        const int64_t m = mb + rl;
        if (ACTOR) {
            // 16 values: xor 16 keeps rows {0,1} or {2,3}; xor 8 keeps one row; xor 4 keeps two actions; xor 2 keeps one; xor 1 finishes
            float s1[2][AM];
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int j = 0; j < AM; ++j) {
                    const float keep = b4 ? pa[2 + r][j] : pa[r][j], send = b4 ? pa[r][j] : pa[2 + r][j];
                    s1[r][j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                }
            float s2[AM];
#pragma unroll
            for (int j = 0; j < AM; ++j) {
                const float keep = b3 ? s1[1][j] : s1[0][j], send = b3 ? s1[0][j] : s1[1][j];
                s2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            }
            float s3[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float keep = b2 ? s2[2 + j] : s2[j], send = b2 ? s2[j] : s2[2 + j];
                s3[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
            const float keep = b1 ? s3[1] : s3[0], send = b1 ? s3[0] : s3[1];
            float z = keep + __shfl_xor_sync(0xffffffffu, send, 2);
            z += __shfl_xor_sync(0xffffffffu, z, 1);
            if ((lane & 1) == 0 && jl < A && m < rows) head_out[m * A + jl] = z + bias_a;
        }
        if (CRITIC) {
            float s1[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float keep = b4 ? pc[2 + r] : pc[r], send = b4 ? pc[r] : pc[2 + r];
                s1[r] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
            const float keep = b3 ? s1[1] : s1[0], send = b3 ? s1[0] : s1[1];
            float v = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            if ((lane & 7) == 0 && m < rows) values[m] = v + bias_c;
        }
    }
}


__global__ void logprob_categorical_kernel(const float* __restrict__ logits, const int32_t* __restrict__ actions,
                                           float* __restrict__ out, int64_t rows, int A)
{
    for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < rows; m += (int64_t)gridDim.x * blockDim.x) {
        const float* z = logits + m * A;
        float mx = -CUDART_INF_F;
        for (int j = 0; j < A; ++j) mx = fmaxf(mx, z[j]);
        float s = 0.f;
        for (int j = 0; j < A; ++j) s += expf(z[j] - mx);
        out[m] = z[actions[m]] - (mx + logf(s));
    }
}

__global__ void logprob_gaussian_kernel(const float* __restrict__ mean, const float* __restrict__ log_std,
                                        const float* __restrict__ actions, float* __restrict__ out, int64_t rows, int A)
{
    for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < rows; m += (int64_t)gridDim.x * blockDim.x) {
        float lp = 0.f;
        for (int j = 0; j < A; ++j) {
            const float sigma = expf(log_std[j]);
            const float diff = actions[m * A + j] - mean[m * A + j];
            lp += -(diff * diff) / (2.0f * sigma * sigma) - logf(sigma) - 0.91893853320467274178f;
        }
        out[m] = lp;
    }
}

// ---------------------------------------------------------------------------------------------
// Standalone loss forward+backward on already-gathered rows (custom network_cls path).
// One warp per row, lane a <-> action a.  Per-CTA partial: [policy, value, entropy, pad, dlog_std A]
// ---------------------------------------------------------------------------------------------
template <bool CONT>
__global__ void __launch_bounds__(256)
loss_rows_kernel(const float* __restrict__ head, const float* __restrict__ log_std_p, int64_t ls_stride, const float* __restrict__ values,
                 const int32_t* __restrict__ actions_i, const float* __restrict__ actions_f, const float* __restrict__ old_logp,
                 const float* __restrict__ adv_p, const float* __restrict__ ret_p, int64_t M, int A, float clip, float vw,
                 float beta, float inv_m, float* __restrict__ dhead, float* __restrict__ dls_rows, float* __restrict__ dvalues,
                 float* __restrict__ partials)
{
    __shared__ float s_red[8][36];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float log_std = (CONT && lane < A && ls_stride == 0) ? log_std_p[lane] : 0.f;
    float l_pol = 0.f, l_val = 0.f, l_ent = 0.f, acc_dls = 0.f;
    const int64_t w0 = (int64_t)blockIdx.x * 8 + warp, wstride = (int64_t)gridDim.x * 8;
    for (int64_t m = w0; m < M; m += wstride) {
        const float z = lane < A ? head[m * A + lane] : 0.f;
        int act_i = 0; float act_f = 0.f;
        if (CONT) act_f = lane < A ? actions_f[m * A + lane] : 0.f; else act_i = actions_i[m];
        if (CONT && ls_stride != 0) log_std = lane < A ? log_std_p[m * ls_stride + lane] : 0.f;
        const Dist<CONT> d = eval_dist<CONT>(z, lane, A, act_i, act_f, log_std);
        const RowTerms t = policy_terms(d.new_lp, old_logp[m], adv_p[m], clip, inv_m);
        if (lane < A) {
            float dz;
            if (!CONT) dz = t.dlogp * ((lane == act_i ? 1.0f : 0.0f) - d.p) + (beta * inv_m) * d.p * (d.lsm + d.entropy);
            else {
                dz = t.dlogp * d.diff / d.var;
                const float dls = t.dlogp * (d.diff * d.diff / d.var - 1.0f) - beta * inv_m;
                acc_dls += dls;
                if (ls_stride != 0) dls_rows[m * A + lane] = dls;
            }
            dhead[m * A + lane] = dz;
        }
        const float verr = values[m] - ret_p[m];
        if (lane == 0) dvalues[m] = vw * verr * inv_m;
        l_pol += t.policy; l_val += verr * verr; l_ent += d.entropy;
    }
    s_red[warp][lane] = acc_dls;
    if (lane == 0) { s_red[warp][32] = l_pol; s_red[warp][33] = l_val; s_red[warp][34] = l_ent; }
    __syncthreads();
    if (threadIdx.x < 35) {
        float s = 0.f;
        for (int w = 0; w < 8; ++w) s += s_red[w][threadIdx.x];
        float* out = partials + (int64_t)blockIdx.x * 40;
        if (threadIdx.x < 32) out[4 + threadIdx.x] = s; else out[threadIdx.x - 32] = s;
    }
}

__global__ void loss_finalize_kernel(const float* __restrict__ partials, int nparts, int A, float vw, float beta, float inv_m,
                                     float* __restrict__ losses, float* __restrict__ dlog_std)
{
    __shared__ float l[3];
    const int i = threadIdx.x;
    if (i < 35) {
        float s = 0.f;
        for (int p = 0; p < nparts; ++p) s += partials[(int64_t)p * 40 + (i < 3 ? i : i + 1)];
        if (i < 3) l[i] = s;
        if (i >= 3 && dlog_std && i - 3 < A) dlog_std[i - 3] = s;
    }
    __syncthreads();
    if (i == 0) {
        const float pol = l[0] * inv_m, val = 0.5f * l[1] * inv_m, ent = l[2] * inv_m;
        losses[0] = pol; losses[1] = val; losses[2] = ent; losses[3] = pol + vw * val + -beta * ent;
    }
}

// ---------------------------------------------------------------------------------------------
// Wide heads (any A, any H up to the GEMM-head bound).  One warp per row; lane l handles actions l, l+32, ... and critic
// columns l, l+32, ...  The row's logits / means are read in passes (max, sum of exponentials, entropy, gradient), every one a
// lane-strided sum in a fixed order followed by the fixed shuffle tree of warp_sum, so the result does not depend on the launch.
// Same per-element formulas as eval_dist / loss_rows_kernel / head_train_kernel.
// TRAIN: rows are gathered through idx (idx < 0: padding row, contributes nothing), advantages normalised from adv_stats, and
// the critic head of the row is evaluated from h3 (v = h3c.wc + bc, d3c = dv wc (1 - h3c^2)).  Per-warp accumulators
// [dba A | dlog_std A | dWc H | db3 H] live in shared memory (one lane per entry: no atomics) and are summed over the warps in
// fixed order into one partial per CTA.  Standalone (custom network_cls): rows already gathered, values given, accumulator
// [dlog_std A] only.
// ---------------------------------------------------------------------------------------------
template <bool CONT, bool TRAIN>
__global__ void __launch_bounds__(256, 1)
wide_loss_kernel(const WideLossArgs a)
{
    extern __shared__ float smem[];
    const int A = a.A, H = TRAIN ? a.H : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int wf = TRAIN ? 2 * (A + H) : A;
    float* s_wc = smem;                                          // [H]
    float* acc = smem + H + (size_t)warp * wf;
    float* s_small = smem + H + (size_t)nw * wf;                 // [nw][4]: policy, value, entropy, dbc
    float* acc_dba = acc;
    float* acc_dls = TRAIN ? acc + A : acc;
    float* acc_dwc = acc + 2 * A;
    float* acc_db3 = acc + 2 * A + H;
    DPPO_PDL_ENTER();
    for (int i = threadIdx.x; i < H; i += blockDim.x) s_wc[i] = a.wc[i];
    for (int i = lane; i < wf; i += 32) acc[i] = 0.f;
    __syncthreads();

    float mean = 0.f, denom = 1.f;
    if (TRAIN) adv_norm_consts(a.adv_stats, a.adv_count, a.advantage_norm, mean, denom);
    const float bias_c = TRAIN ? a.bc[0] : 0.f;
    const float ent_scale = a.beta * a.inv_m;
    float l_pol = 0.f, l_val = 0.f, l_ent = 0.f, s_dbc = 0.f;
    for (int64_t m = (int64_t)blockIdx.x * nw + warp; m < a.M; m += (int64_t)gridDim.x * nw) {
        int64_t src = m;
        bool live = true;
        if (TRAIN) {
            const int64_t s = a.idx ? (int64_t)__ldg(a.idx + m) : m;
            live = s >= 0;
            src = live ? s : 0;
        }
        const float* z = a.z + m * A;                            // plain loads: dz may alias z
        const float* ls = CONT ? (a.ls_stride ? a.log_std + m * a.ls_stride : a.log_std) : nullptr;
        const float* act_f = CONT ? a.actions_f + src * A : nullptr;
        const float old_lp = __ldg(a.old_logp + src);
        const float advv = (__ldg(a.adv + src) - mean) / denom;
        float new_lp, entropy, lse = 0.f;
        int act = 0;
        if (!CONT) {
            // torch/distributions/categorical.py:78 (logits - logsumexp), :151-163 (log_prob, entropy)
            act = __ldg(a.actions_i + src);
            float mx = -CUDART_INF_F;
            for (int j = lane; j < A; j += 32) mx = fmaxf(mx, z[j]);
            mx = warp_max(mx);
            float s = 0.f;
            for (int j = lane; j < A; j += 32) s += expf(z[j] - mx);
            lse = mx + logf(warp_sum(s));
            float en = 0.f;
            for (int j = lane; j < A; j += 32) { const float lsm = z[j] - lse; en += expf(lsm) * lsm; }
            entropy = -warp_sum(en);
            new_lp = z[act] - lse;
        } else {
            // torch/distributions/normal.py:87-102, :114-115, summed over dims (continuous_ppo.py:40-47)
            float lp = 0.f, en = 0.f;
            for (int j = lane; j < A; j += 32) {
                const float sigma = expf(ls[j]);
                const float log_scale = logf(sigma);
                const float diff = __ldg(act_f + j) - z[j];
                lp += -(diff * diff) / (2.0f * (sigma * sigma)) - log_scale - 0.91893853320467274178f;
                en += 0.5f + 0.91893853320467274178f + log_scale;
            }
            new_lp = warp_sum(lp);
            entropy = warp_sum(en);
        }
        const RowTerms t = policy_terms(new_lp, old_lp, advv, a.clip, a.inv_m);
        float* dz = a.dz + m * A;
        for (int j = lane; j < A; j += 32) {
            float g = 0.f;
            if (!CONT) {
                const float lsm = z[j] - lse, p = expf(lsm);
                if (live) g = t.dlogp * ((j == act ? 1.0f : 0.0f) - p) + ent_scale * p * (lsm + entropy);
            } else if (live) {
                const float sigma = expf(ls[j]);
                const float var = sigma * sigma;
                const float diff = __ldg(act_f + j) - z[j];
                g = t.dlogp * diff / var;
                const float dls = t.dlogp * (diff * diff / var - 1.0f) - ent_scale;
                if (a.ls_stride) a.dls_rows[m * A + j] = dls;
                else acc_dls[j] += dls;
            }
            dz[j] = g;                                           // after this lane's last read of z[j]
            if (TRAIN) acc_dba[j] += g;
        }
        float verr;
        if (TRAIN) {
            const float* hc = a.h3 + m * (2 * (int64_t)H) + H;
            float vp = 0.f;
            for (int k = lane; k < H; k += 32) vp = fmaf(__ldg(hc + k), s_wc[k], vp);
            verr = warp_sum(vp) + bias_c - __ldg(a.ret + src);
            const float dv = live ? a.vw * verr * a.inv_m : 0.f;
            float* dc = a.d3 + m * (2 * (int64_t)H) + H;
            for (int k = lane; k < H; k += 32) {
                const float h = __ldg(hc + k);
                const float g = dv * s_wc[k] * (1.0f - h * h);
                dc[k] = g;
                acc_dwc[k] = fmaf(dv, h, acc_dwc[k]);
                acc_db3[k] += g;
            }
            s_dbc += dv;
        } else {
            verr = __ldg(a.values + m) - __ldg(a.ret + m);
            if (lane == 0) a.dvalues[m] = a.vw * verr * a.inv_m;
        }
        if (live) { l_pol += t.policy; l_val += verr * verr; l_ent += entropy; }
    }
    if (lane == 0) { s_small[warp * 4] = l_pol; s_small[warp * 4 + 1] = l_val; s_small[warp * 4 + 2] = l_ent; s_small[warp * 4 + 3] = s_dbc; }
    __syncthreads();

    const WideOffsets o = wide_offsets(H, A);
    float* out = a.partials + (int64_t)blockIdx.x * a.partial_stride;
    for (int i = threadIdx.x; i < wf; i += blockDim.x) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += smem[H + (size_t)w * wf + i];
        int dst = o.dls + i;
        if (TRAIN) dst = i < A ? o.dba + i : i < 2 * A ? o.dls + (i - A) : i < 2 * A + H ? o.dwc + (i - 2 * A) : o.db3 + (i - 2 * A - H);
        out[dst] = s;
    }
    if (threadIdx.x < 4) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += s_small[w * 4 + threadIdx.x];
        if (threadIdx.x < 3) out[threadIdx.x] = s;
        else { out[3] = 0.f; out[o.dbc] = s; }
    }
}

__global__ void wide_loss_finalize_kernel(const float* __restrict__ partials, int nparts, int stride, int dls_off, int A, float vw,
                                          float beta, float inv_m, float* __restrict__ losses, float* __restrict__ dlog_std)
{
    __shared__ float l[3];
    for (int i = threadIdx.x; i < 3 + A; i += blockDim.x) {
        const int off = i < 3 ? i : dls_off + (i - 3);
        float s = 0.f;
        for (int p = 0; p < nparts; ++p) s += partials[(int64_t)p * stride + off];
        if (i < 3) l[i] = s;
        else if (dlog_std) dlog_std[i - 3] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const float pol = l[0] * inv_m, val = 0.5f * l[1] * inv_m, ent = l[2] * inv_m;
        losses[0] = pol; losses[1] = val; losses[2] = ent; losses[3] = pol + vw * val + -beta * ent;
    }
}

// Critic head of the forward pass at H > 512: one warp per row, wc in shared memory (the actor head is a GEMM there).
__global__ void __launch_bounds__(256)
critic_value_kernel(const float* __restrict__ hc, int ld, const float* __restrict__ wc, const float* __restrict__ bc,
                    float* __restrict__ values, int64_t rows, int H, const int* __restrict__ rows_dev)
{
    extern __shared__ float s_wc[];
    if (rows_dev != nullptr && *rows_dev < rows) rows = *rows_dev;
    for (int i = threadIdx.x; i < H; i += blockDim.x) s_wc[i] = wc[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t ws = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t m = w0; m < rows; m += ws) {
        float part = 0.f;
        for (int k = lane; k < H; k += 32) part = fmaf(__ldg(hc + m * ld + k), s_wc[k], part);
        part = warp_sum(part);
        if (lane == 0) values[m] = part + bc[0];
    }
}

// warps per CTA of the training variant: two CTAs per SM while the per-warp accumulators allow it
int wide_train_warps(int H, int A)
{
    int nw = 8;
    while (nw > 1 && ((size_t)nw * (2 * (A + H) + 4) + H) * sizeof(float) > 110 * 1024) nw >>= 1;
    return nw;
}

template <int KPL, int VEC, int R>
int launch_head_train(dppo_ctx* ctx, const HeadTrainArgs& a, int continuous, int blocks, size_t smem, cudaStream_t st)
{
    if (continuous) {
        cudaFuncSetAttribute(head_train_kernel<true, KPL, VEC, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        dppo_launch_pdl(ctx, head_train_kernel<true, KPL, VEC, R>, dim3(blocks), dim3(HEAD_WARPS * 32), smem, st, a);
    } else {
        cudaFuncSetAttribute(head_train_kernel<false, KPL, VEC, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        dppo_launch_pdl(ctx, head_train_kernel<false, KPL, VEC, R>, dim3(blocks), dim3(HEAD_WARPS * 32), smem, st, a);
    }
    DPPO_CHECK_LAUNCH(ctx, "head_train_kernel");
    return 0;
}

}  // namespace

int head_partial_floats(int H, int A) { return head_offsets(H, A).total; }

static bool head_split_shape(int H, int A) { return (H == 128 || H == 256) && A <= 4; }

int head_train_blocks(dppo_ctx* ctx, int64_t M, int H, int A)
{
    (void)H; (void)A;
    int64_t want = (M + HEAD_WARPS - 1) / HEAD_WARPS;
    int64_t cap = 2 * (int64_t)ctx->sm_count;
    return (int)(want < cap ? want : cap);
}

// dynamic shared memory of head_train_kernel: Wa | wc, then the per-warp accumulators (reused as the flush scratch)
static size_t head_train_smem(int H, int A)
{
    size_t accf = (size_t)HEAD_WARPS * (A + 1) * H;
    const size_t scratchf = (size_t)HEAD_WARPS * (2 * H + 100);
    if (accf < scratchf) accf = scratchf;
    return ((size_t)(A + 1) * H + accf) * sizeof(float);
}

bool head_train_supported(int H, int A)
{
    return A >= 1 && A <= DPPO_MAX_ACT && H >= 1 && H <= 512 && head_train_smem(H, A) <= 200 * 1024;
}

int launch_head_train_kernel(dppo_ctx* ctx, const HeadTrainArgs& a, int continuous, int blocks, cudaStream_t st)
{
    const int H = a.H, A = a.A;
    if (A < 1 || A > DPPO_MAX_ACT) DPPO_FAIL(ctx, "head kernel supports 1..%d actions/action dims, got %d", DPPO_MAX_ACT, A);
    if (H < 1 || H > 512) DPPO_FAIL(ctx, "head kernel supports hidden <= 512, got %d", H);
    const size_t smem = head_train_smem(H, A);
    if (smem > 200 * 1024) DPPO_FAIL(ctx, "head kernel: (A+1)*H = %d too large for shared memory", (A + 1) * H);
    const bool vec = (H % 128 == 0) && ((reinterpret_cast<uintptr_t>(a.h3) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(a.d3) & 15u) == 0);
    if (vec && head_split_shape(H, A)) {
        if (a.M >= (int64_t)1 << 30) DPPO_FAIL(ctx, "head kernel: %lld rows exceed the 32-bit row counter", (long long)a.M);
        const size_t sm = ((size_t)4 * H + (size_t)(SPLIT_NA * 4 + SPLIT_WARPS - SPLIT_NA) * H + (size_t)SPLIT_WARPS * (H + 16)) * sizeof(float);
#define HTS(G)                                                                                                                   \
    do {                                                                                                                         \
        if (continuous) {                                                                                                        \
            cudaFuncSetAttribute(head_train_split_kernel<true, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);         \
            dppo_launch_pdl(ctx, head_train_split_kernel<true, G>, dim3(blocks), dim3(SPLIT_WARPS * 32), sm, st, a);             \
        } else {                                                                                                                 \
            cudaFuncSetAttribute(head_train_split_kernel<false, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);        \
            dppo_launch_pdl(ctx, head_train_split_kernel<false, G>, dim3(blocks), dim3(SPLIT_WARPS * 32), sm, st, a);            \
        }                                                                                                                        \
    } while (0)
        if (H == 128) HTS(1); else HTS(2);
#undef HTS
        DPPO_CHECK_LAUNCH(ctx, "head_train_split_kernel");
        return 0;
    }
    if (H <= 64) return launch_head_train<2, 1, 2>(ctx, a, continuous, blocks, smem, st);
    if (H <= 128) return vec ? launch_head_train<4, 4, 2>(ctx, a, continuous, blocks, smem, st) : launch_head_train<4, 1, 2>(ctx, a, continuous, blocks, smem, st);
    if (H <= 256) return vec ? launch_head_train<8, 4, 2>(ctx, a, continuous, blocks, smem, st) : launch_head_train<8, 1, 2>(ctx, a, continuous, blocks, smem, st);
    return vec ? launch_head_train<16, 4, 1>(ctx, a, continuous, blocks, smem, st) : launch_head_train<16, 1, 1>(ctx, a, continuous, blocks, smem, st);
}

int launch_head_eval(dppo_ctx* ctx, const float* ha, const float* hc, int ld, const float* wa, const float* ba, const float* wc,
                     const float* bc, float* head_out, float* values, int64_t rows, int H, int A, int rev, cudaStream_t st)
{
    if (A < 1 || A > DPPO_MAX_ACT) DPPO_FAIL(ctx, "head kernel supports 1..%d actions/action dims, got %d", DPPO_MAX_ACT, A);
    if (H < 1 || H > 512) DPPO_FAIL(ctx, "head kernel supports hidden <= 512, got %d", H);
    const size_t smem = (size_t)(A + 1) * H * sizeof(float);
    int64_t want = (rows + 7) / 8;
    int blocks = (int)(want < 4 * (int64_t)ctx->sm_count ? want : 4 * (int64_t)ctx->sm_count);
    const bool al = ld % 4 == 0 && (!ha || (reinterpret_cast<uintptr_t>(ha) & 15u) == 0) && (!hc || (reinterpret_cast<uintptr_t>(hc) & 15u) == 0) &&
                    (reinterpret_cast<uintptr_t>(wc) & 15u) == 0;
    if ((H == 128 || H == 256) && A <= 4 && al && (ha || hc)) {
        want = (rows + 31) / 32;                                 // 8 warps x 4 rows per block iteration
        blocks = (int)(want < 4 * (int64_t)ctx->sm_count ? want : 4 * (int64_t)ctx->sm_count);
#define HEV(G, AC, CR) head_eval_vec_kernel<G, AC, CR><<<blocks, 256, 0, st>>>(ha, hc, ld, wa, ba, wc, bc, head_out, values, rows, A, rev, ctx->rows_dev)
        if (H == 128) { if (ha && hc) HEV(1, true, true); else if (ha) HEV(1, true, false); else HEV(1, false, true); }
        else { if (ha && hc) HEV(2, true, true); else if (ha) HEV(2, true, false); else HEV(2, false, true); }
#undef HEV
        DPPO_CHECK_LAUNCH(ctx, "head_eval_vec_kernel");
        return 0;
    }
#define HE(KPL)                                                                                                   \
    do {                                                                                                          \
        cudaFuncSetAttribute(head_eval_kernel<KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
        head_eval_kernel<KPL><<<blocks, 256, smem, st>>>(ha, hc, ld, wa, ba, wc, bc, head_out, values, rows, H, A, ctx->rows_dev); \
    } while (0)
    if (H <= 64) HE(2); else if (H <= 128) HE(4); else if (H <= 256) HE(8); else HE(16);
#undef HE
    DPPO_CHECK_LAUNCH(ctx, "head_eval_kernel");
    return 0;
}

int launch_heads_forward(dppo_ctx* ctx, const float* ha, const float* hc, int ld, const float* wa, const float* ba, const float* wc,
                         const float* bc, float* head_out, float* values, int64_t rows, int H, int A, int rev, cudaStream_t st)
{
    if (A >= 1 && A <= DPPO_MAX_ACT && H >= 1 && H <= 512)
        return launch_head_eval(ctx, ha, hc, ld, wa, ba, wc, bc, head_out, values, rows, H, A, rev, st);
    if (A < 1 || A > DPPO_GEMM_HEADS_MAX_ACT || H < 1 || H > DPPO_GEMM_HEADS_MAX_HIDDEN)
        DPPO_FAIL(ctx, "heads: hidden %d / %d actions outside the GEMM-head bound (hidden <= %d, 1..%d actions)", H, A,
                  DPPO_GEMM_HEADS_MAX_HIDDEN, DPPO_GEMM_HEADS_MAX_ACT);
    // logits / means = h3a Wa^T + ba (ppo.py:63-71)
    if (ha && dppo_gemm_nt(ctx, DPPO_EPI_BIAS, ha, ld, nullptr, wa, H, ba, head_out, A, rows, A, H, st)) return 1;
    if (hc) {
        int64_t want = (rows + 7) / 8;
        const int blocks = (int)(want < 4 * (int64_t)ctx->sm_count ? want : 4 * (int64_t)ctx->sm_count);
        critic_value_kernel<<<blocks, 256, (size_t)H * sizeof(float), st>>>(hc, ld, wc, bc, values, rows, H, ctx->rows_dev);
        DPPO_CHECK_LAUNCH(ctx, "critic_value_kernel");
    }
    return 0;
}

int wide_loss_blocks(dppo_ctx* ctx, int64_t M, int H, int A)
{
    const int nw = wide_train_warps(H, A);
    const int64_t want = (M + nw - 1) / nw;
    const int64_t cap = 2 * (int64_t)ctx->sm_count;
    return (int)(want < cap ? want : cap);
}

int launch_wide_loss_train(dppo_ctx* ctx, const WideLossArgs& a, int continuous, int blocks, cudaStream_t st)
{
    const int nw = wide_train_warps(a.H, a.A);
    const size_t smem = ((size_t)nw * (2 * (a.A + a.H) + 4) + a.H) * sizeof(float);
    auto kern = continuous ? wide_loss_kernel<true, true> : wide_loss_kernel<false, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    dppo_launch_pdl(ctx, kern, dim3(blocks), dim3(nw * 32), smem, st, a);
    DPPO_CHECK_LAUNCH(ctx, "wide_loss_kernel");
    return 0;
}

extern "C" int dppo_logprob_categorical(dppo_ctx* ctx, const float* logits, const int32_t* actions, float* log_probs,
                                        int64_t rows, int A, void* stream)
{
    if (!ctx) return 1;
    if (rows <= 0) return 0;
    int blocks = (int)((rows + 255) / 256);
    if (blocks > 8 * ctx->sm_count) blocks = 8 * ctx->sm_count;
    logprob_categorical_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(logits, actions, log_probs, rows, A);
    DPPO_CHECK_LAUNCH(ctx, "logprob_categorical_kernel");
    return 0;
}

extern "C" int dppo_logprob_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, const float* actions,
                                     float* log_probs, int64_t rows, int A, void* stream)
{
    if (!ctx) return 1;
    if (rows <= 0) return 0;
    int blocks = (int)((rows + 255) / 256);
    if (blocks > 8 * ctx->sm_count) blocks = 8 * ctx->sm_count;
    logprob_gaussian_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(mean, log_std, actions, log_probs, rows, A);
    DPPO_CHECK_LAUNCH(ctx, "logprob_gaussian_kernel");
    return 0;
}

static int loss_blocks(dppo_ctx* ctx, int64_t M)
{
    int64_t want = (M + 7) / 8;
    int64_t cap = 2 * (int64_t)ctx->sm_count;
    return (int)(want < cap ? want : cap);
}

// floats per CTA partial: loss_rows_kernel's 40 up to DPPO_MAX_ACT actions, wide_loss_kernel's above
static int loss_partial_floats(int A) { return A <= DPPO_MAX_ACT ? 40 : wide_offsets(0, A).total; }

extern "C" int64_t dppo_ppo_loss_workspace_bytes(int64_t M, int A)
{
    int64_t blocks = (M + 7) / 8;
    if (blocks > 2 * 256) blocks = 2 * 256;            // upper bound on 2*SMs
    return blocks * loss_partial_floats(A) * (int64_t)sizeof(float);
}

static int ppo_loss_common(dppo_ctx* ctx, bool cont, const float* head, const float* log_std, int64_t ls_stride, const float* values,
                           const int32_t* actions_i, const float* actions_f, const float* old_lp, const float* adv,
                           const float* ret, int64_t M, int A, const dppo_hyper* h, float* losses, float* dhead,
                           float* dlog_std, float* dvalues, void* ws, int64_t ws_bytes, cudaStream_t st)
{
    if (!ctx) return 1;
    if (M <= 0) DPPO_FAIL(ctx, "ppo_loss: empty minibatch");
    if (A < 1 || A > DPPO_GEMM_HEADS_MAX_ACT) DPPO_FAIL(ctx, "ppo_loss supports 1..%d actions/action dims, got %d", DPPO_GEMM_HEADS_MAX_ACT, A);
    const int blocks = loss_blocks(ctx, M);
    if (ws_bytes < (int64_t)blocks * loss_partial_floats(A) * (int64_t)sizeof(float)) DPPO_FAIL(ctx, "ppo_loss: workspace too small");
    const float inv_m = 1.0f / (float)(h->loss_denominator > 0 ? h->loss_denominator : M);
    float* partials = (float*)ws;
    if (A > DPPO_MAX_ACT) {
        // more actions than lanes: lanes stride over the actions (wide_loss_kernel without its critic part)
        WideLossArgs a = {};
        a.z = head; a.dz = dhead; a.log_std = log_std; a.ls_stride = cont ? ls_stride : 0; a.dls_rows = ls_stride ? dlog_std : nullptr;
        a.values = values; a.dvalues = dvalues;
        a.actions_i = actions_i; a.actions_f = actions_f; a.old_logp = old_lp; a.adv = adv; a.ret = ret;
        a.M = M; a.H = 0; a.A = A;
        a.clip = h->ppo_clip; a.vw = h->value_loss_weight; a.beta = h->entropy_beta; a.inv_m = inv_m;
        a.partials = partials; a.partial_stride = loss_partial_floats(A);
        const size_t smem = ((size_t)8 * (A + 4)) * sizeof(float);
        auto kern = cont ? wide_loss_kernel<true, false> : wide_loss_kernel<false, false>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<blocks, 256, smem, st>>>(a);
        DPPO_CHECK_LAUNCH(ctx, "wide_loss_kernel");
        wide_loss_finalize_kernel<<<1, 256, 0, st>>>(partials, blocks, a.partial_stride, wide_offsets(0, A).dls, A, h->value_loss_weight,
                                                    h->entropy_beta, inv_m, losses, (cont && !ls_stride) ? dlog_std : nullptr);
        DPPO_CHECK_LAUNCH(ctx, "wide_loss_finalize_kernel");
        return 0;
    }
    if (cont)
        loss_rows_kernel<true><<<blocks, 256, 0, st>>>(head, log_std, ls_stride, values, actions_i, actions_f, old_lp, adv, ret, M, A,
                                                       h->ppo_clip, h->value_loss_weight, h->entropy_beta, inv_m, dhead,
                                                       ls_stride ? dlog_std : nullptr, dvalues, partials);
    else
        loss_rows_kernel<false><<<blocks, 256, 0, st>>>(head, log_std, 0, values, actions_i, actions_f, old_lp, adv, ret, M, A,
                                                        h->ppo_clip, h->value_loss_weight, h->entropy_beta, inv_m, dhead, nullptr, dvalues, partials);
    DPPO_CHECK_LAUNCH(ctx, "loss_rows_kernel");
    loss_finalize_kernel<<<1, 64, 0, st>>>(partials, blocks, A, h->value_loss_weight, h->entropy_beta, inv_m, losses,
                                           ls_stride ? nullptr : dlog_std);
    DPPO_CHECK_LAUNCH(ctx, "loss_finalize_kernel");
    return 0;
}

extern "C" int dppo_ppo_loss_discrete(dppo_ctx* ctx, const float* logits, const float* values, const int32_t* actions,
                                      const float* old_log_probs, const float* adv, const float* returns, int64_t M, int A,
                                      const dppo_hyper* hyper, float* losses, float* dlogits, float* dvalues, void* ws,
                                      int64_t ws_bytes, void* stream)
{
    return ppo_loss_common(ctx, false, logits, nullptr, 0, values, actions, nullptr, old_log_probs, adv, returns, M, A, hyper,
                           losses, dlogits, nullptr, dvalues, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int dppo_ppo_loss_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, int64_t log_std_row_stride, const float* values,
                                      const float* actions, const float* old_log_probs, const float* adv, const float* returns,
                                      int64_t M, int A, const dppo_hyper* hyper, float* losses, float* dmean, float* dlog_std,
                                      float* dvalues, void* ws, int64_t ws_bytes, void* stream)
{
    return ppo_loss_common(ctx, true, mean, log_std, log_std_row_stride, values, nullptr, actions, old_log_probs, adv, returns, M, A, hyper, losses,
                           dmean, dlog_std, dvalues, ws, ws_bytes, (cudaStream_t)stream);
}
