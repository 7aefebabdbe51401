// Recurrent actor-critic (diamond/recurrent_ppo.py:94-149): Linear-Tanh -> GRU with done-masked hidden resets -> actor / critic
// heads, forward over a whole [T, N] rollout and full-T back-propagation through time for one minibatch (:337-341).
//
// The time loop of the reference is T one-step nn.GRU calls.  Here everything that does not depend on the recurrence is a
// batched product over all T*N rows (input projection, heads, weight gradients), and only the hidden-to-hidden recurrence runs
// in the two scan kernels below: environments are independent sequences, so a scan owns a group of environments for all T
// steps and keeps W_hh and the running hidden state on chip.
//   Hg <= 32 (the default 16): one environment per Hg-lane group of a warp, this lane's three W_hh rows (forward) or columns
//   (backward) in registers, the hidden vector exchanged with shuffles -- no block barrier inside the time loop;
//   Hg <= 128: W_hh in shared memory, hidden vectors double-buffered in shared memory, one barrier per step;
//   128 < Hg <= 512: W_hh split by hidden unit over the CTAs of a thread-block cluster, hidden state exchanged over distributed
//   shared memory, one cluster barrier per step.
// GRU cell (torch nn.GRU, gate order r, z, n): r = s(gi_r + W_hr h + b_hr), z = s(gi_z + W_hz h + b_hz),
// n = tanh(gi_n + r * (W_hn h + b_hn)), h' = (1 - z) * n + z * h, with h <- 0 where prev_dones[t] (recurrent_ppo.py:84).
#include <cooperative_groups.h>

#include "common.cuh"
#include "heads.cuh"
#include "optim.cuh"

namespace cg = cooperative_groups;

namespace {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

struct ScanFwdArgs {
    const float* gi;            // [T, N, 3Hg] input projection incl. b_ih
    const float* whh;           // [3Hg, Hg]
    const float* bhh;           // [3Hg]
    const unsigned char* dones; // [T, N] prev_dones (may be null: no resets)
    const float* hx0;           // [N, Hg] (may be null: zeros)
    float* hs;                  // [T, N, Hg] h_t
    float* hm;                  // [T, N, Hg] masked previous hidden state (training only, else null)
    float* gates;               // [T, N, 3Hg] r, z, n after their activations (training only)
    float* hn;                  // [T, N, Hg]  W_hn hm + b_hn (training only)
    float* hx_out;              // [N, Hg] final hidden state (may be null)
    int T, N, Hg;
};

// ---- forward scan, Hg <= 32: environment = HG-lane group, weights in registers ----------------------------------------------
template <int HG>
__global__ void __launch_bounds__(128)
gru_scan_fwd_warp_kernel(ScanFwdArgs a)
{
    const int lane = threadIdx.x & 31;
    const int j = lane % HG;                                    // hidden unit
    const int base = lane - j;                                  // first lane of this environment's group
    const int64_t env = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / HG;
    const bool on = env < a.N;
    const int64_t e = on ? env : 0;
    float wr[HG], wz[HG], wn[HG];
#pragma unroll
    for (int k = 0; k < HG; ++k) {
        wr[k] = a.whh[(int64_t)j * HG + k];
        wz[k] = a.whh[(int64_t)(HG + j) * HG + k];
        wn[k] = a.whh[(int64_t)(2 * HG + j) * HG + k];
    }
    const float br = a.bhh[j], bz = a.bhh[HG + j], bn = a.bhh[2 * HG + j];
    float h = a.hx0 ? a.hx0[e * HG + j] : 0.f;
    const int64_t rs = (int64_t)a.N;                            // rows per step
    float gr = a.gi[e * 3 * HG + j], gz = a.gi[e * 3 * HG + HG + j], gn = a.gi[e * 3 * HG + 2 * HG + j];
    unsigned char dn = a.dones ? a.dones[e] : 0;
    for (int t = 0; t < a.T; ++t) {
        const int64_t row = (int64_t)t * rs + e;
        // the next step's inputs do not depend on the recurrence: request them before the dependent math
        float gr1 = 0.f, gz1 = 0.f, gn1 = 0.f;
        unsigned char dn1 = 0;
        if (t + 1 < a.T) {
            const float* g1 = a.gi + (row + rs) * 3 * HG;
            gr1 = g1[j]; gz1 = g1[HG + j]; gn1 = g1[2 * HG + j];
            if (a.dones) dn1 = a.dones[row + rs];
        }
        const float m = dn ? 0.f : h;                           // recurrent_ppo.py:84
        float ar = br, az = bz, an = bn;
#pragma unroll
        for (int k = 0; k < HG; ++k) {
            const float hk = __shfl_sync(0xffffffffu, m, base + k);
            ar = fmaf(wr[k], hk, ar); az = fmaf(wz[k], hk, az); an = fmaf(wn[k], hk, an);
        }
        const float r = sigmoidf_(gr + ar), z = sigmoidf_(gz + az);
        const float n = tanhf(gn + r * an);
        h = (1.0f - z) * n + z * m;
        if (on) {
            a.hs[row * HG + j] = h;
            if (a.hm) {
                a.hm[row * HG + j] = m;
                float* g = a.gates + row * 3 * HG;
                g[j] = r; g[HG + j] = z; g[2 * HG + j] = n;
                a.hn[row * HG + j] = an;
            }
        }
        gr = gr1; gz = gz1; gn = gn1; dn = dn1;
    }
    if (on && a.hx_out) a.hx_out[e * HG + j] = h;
}

// ---- forward scan, general Hg: W_hh^T and the hidden vectors in shared memory ------------------------------------------------
__global__ void gru_scan_fwd_smem_kernel(ScanFwdArgs a, int EB)
{
    extern __shared__ float smem[];
    const int Hg = a.Hg;
    float* wt = smem;                                           // [Hg][3Hg]: wt[k][g] = W_hh[g][k]
    float* hb = wt + 3 * Hg * Hg;                               // [2][EB][Hg]
    for (int i = threadIdx.x; i < 3 * Hg * Hg; i += blockDim.x) {
        const int g = i / Hg, k = i % Hg;
        wt[k * 3 * Hg + g] = a.whh[i];
    }
    const int le = threadIdx.x / Hg, j = threadIdx.x % Hg;
    const int64_t env = (int64_t)blockIdx.x * EB + le;
    const bool on = le < EB && env < a.N;
    const int64_t e = on ? env : 0;
    const float br = a.bhh[j], bz = a.bhh[Hg + j], bn = a.bhh[2 * Hg + j];
    float h = (on && a.hx0) ? a.hx0[e * Hg + j] : 0.f;
    const int64_t rs = (int64_t)a.N;
    __syncthreads();
    for (int t = 0; t < a.T; ++t) {
        const int64_t row = (int64_t)t * rs + e;
        const float* g = a.gi + row * 3 * Hg;
        const float gr = g[j], gz = g[Hg + j], gn = g[2 * Hg + j];
        const bool dn = a.dones && a.dones[row];
        const float m = dn ? 0.f : h;
        float* cur = hb + (size_t)(t & 1) * EB * Hg;
        if (le < EB) cur[le * Hg + j] = m;
        __syncthreads();                                        // one barrier per step: the other buffer is written next step
        float ar = br, az = bz, an = bn;
        if (le < EB) {
            const float* hv = cur + le * Hg;
            for (int k = 0; k < Hg; ++k) {
                const float hk = hv[k];
                const float* w = wt + k * 3 * Hg;
                ar = fmaf(w[j], hk, ar); az = fmaf(w[Hg + j], hk, az); an = fmaf(w[2 * Hg + j], hk, an);
            }
        }
        const float r = sigmoidf_(gr + ar), z = sigmoidf_(gz + az);
        const float n = tanhf(gn + r * an);
        h = (1.0f - z) * n + z * m;
        if (on) {
            a.hs[row * Hg + j] = h;
            if (a.hm) {
                a.hm[row * Hg + j] = m;
                float* go = a.gates + row * 3 * Hg;
                go[j] = r; go[Hg + j] = z; go[2 * Hg + j] = n;
                a.hn[row * Hg + j] = an;
            }
        }
    }
    if (on && a.hx_out) a.hx_out[e * Hg + j] = h;
}

// ---- forward scan, Hg a multiple of 4 (beyond the warp kernel's 8 / 16 / 32): E environments per thread -----------------------
// Thread (group, j) owns hidden unit j of E environments.  The one-environment-per-thread kernel above issues four shared-memory
// loads per three FMAs and is bound by the LDS pipe (ncu, round 1: 1.18 ms at N = 4096, Hg = 64); here every W_hh value read
// from shared memory (LDS.128 along k, rows padded by 4 floats so that a quarter warp hits eight different 16-byte bank
// groups) serves E environments and the hidden vectors are read as warp-wide LDS.128 broadcasts: 3 + E loads per 12 E FMAs.
// Same summation order (k ascending, one fused multiply-add chain per gate) as the kernels above: bit-identical results.
template <int E>
__global__ void __launch_bounds__(256)
gru_scan_fwd_tiled_kernel(ScanFwdArgs a, int G)
{
    extern __shared__ float smem[];
    const int Hg = a.Hg, WS = Hg + 4;
    float* w = smem;                                            // [3Hg][WS]  (W_hh rows, padded)
    float* hb = w + 3 * Hg * WS;                                // [2][G * E][Hg] masked hidden vectors, double-buffered over t
    for (int i = threadIdx.x; i < 3 * Hg * Hg; i += blockDim.x) w[(i / Hg) * WS + (i % Hg)] = a.whh[i];
    const int grp = threadIdx.x / Hg, j = threadIdx.x % Hg;
    const int64_t env0 = ((int64_t)blockIdx.x * G + grp) * E;
    const float br = a.bhh[j], bz = a.bhh[Hg + j], bn = a.bhh[2 * Hg + j];
    const int64_t rs = (int64_t)a.N;
    bool on[E];
    int64_t e[E];
    float h[E], gr[E], gz[E], gn[E];
    unsigned char dn[E];
#pragma unroll
    for (int i = 0; i < E; ++i) {
        on[i] = env0 + i < a.N;
        e[i] = on[i] ? env0 + i : 0;
        h[i] = (on[i] && a.hx0) ? a.hx0[e[i] * Hg + j] : 0.f;
        const float* g = a.gi + e[i] * 3 * Hg;
        gr[i] = g[j]; gz[i] = g[Hg + j]; gn[i] = g[2 * Hg + j];
        dn[i] = a.dones ? a.dones[e[i]] : 0;
    }
    const float4* wr4 = reinterpret_cast<const float4*>(w + (size_t)j * WS);
    const float4* wz4 = reinterpret_cast<const float4*>(w + (size_t)(Hg + j) * WS);
    const float4* wn4 = reinterpret_cast<const float4*>(w + (size_t)(2 * Hg + j) * WS);
    __syncthreads();
    for (int t = 0; t < a.T; ++t) {
        // the next step's inputs do not depend on the recurrence: request them before the dependent math
        float gr1[E], gz1[E], gn1[E];
        unsigned char dn1[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            gr1[i] = gz1[i] = gn1[i] = 0.f; dn1[i] = 0;
            if (t + 1 < a.T) {
                const int64_t row1 = (int64_t)(t + 1) * rs + e[i];
                const float* g1 = a.gi + row1 * 3 * Hg;
                gr1[i] = g1[j]; gz1[i] = g1[Hg + j]; gn1[i] = g1[2 * Hg + j];
                if (a.dones) dn1[i] = a.dones[row1];
            }
        }
        float* cur = hb + (size_t)(t & 1) * G * E * Hg + (size_t)grp * E * Hg;
        float m[E], ar[E], az[E], an[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            m[i] = dn[i] ? 0.f : h[i];                          // recurrent_ppo.py:84
            cur[i * Hg + j] = m[i];
            ar[i] = br; az[i] = bz; an[i] = bn;
        }
        __syncthreads();                                        // one barrier per step: the other buffer is written next step
        for (int k4 = 0; k4 < Hg / 4; ++k4) {
            const float4 a_r = wr4[k4], a_z = wz4[k4], a_n = wn4[k4];
#pragma unroll
            for (int i = 0; i < E; ++i) {
                const float4 hv = reinterpret_cast<const float4*>(cur + i * Hg)[k4];
                ar[i] = fmaf(a_r.x, hv.x, ar[i]); az[i] = fmaf(a_z.x, hv.x, az[i]); an[i] = fmaf(a_n.x, hv.x, an[i]);
                ar[i] = fmaf(a_r.y, hv.y, ar[i]); az[i] = fmaf(a_z.y, hv.y, az[i]); an[i] = fmaf(a_n.y, hv.y, an[i]);
                ar[i] = fmaf(a_r.z, hv.z, ar[i]); az[i] = fmaf(a_z.z, hv.z, az[i]); an[i] = fmaf(a_n.z, hv.z, an[i]);
                ar[i] = fmaf(a_r.w, hv.w, ar[i]); az[i] = fmaf(a_z.w, hv.w, az[i]); an[i] = fmaf(a_n.w, hv.w, an[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const float r = sigmoidf_(gr[i] + ar[i]), z = sigmoidf_(gz[i] + az[i]);
            const float n = tanhf(gn[i] + r * an[i]);
            h[i] = (1.0f - z) * n + z * m[i];
            if (on[i]) {
                const int64_t row = (int64_t)t * rs + e[i];
                a.hs[row * Hg + j] = h[i];
                if (a.hm) {
                    a.hm[row * Hg + j] = m[i];
                    float* go = a.gates + row * 3 * Hg;
                    go[j] = r; go[Hg + j] = z; go[2 * Hg + j] = n;
                    a.hn[row * Hg + j] = an[i];
                }
            }
            gr[i] = gr1[i]; gz[i] = gz1[i]; gn[i] = gn1[i]; dn[i] = dn1[i];
        }
    }
#pragma unroll
    for (int i = 0; i < E; ++i)
        if (on[i] && a.hx_out) a.hx_out[e[i] * Hg + j] = h[i];
}

struct ScanBwdArgs {
    const float* dhs;           // [T, N, Hg] d(loss)/d(h_t) from the heads
    const float* whh;           // [3Hg, Hg]
    const unsigned char* dones; // [T, N] (may be null)
    const float* hm;            // [T, N, Hg]
    const float* gates;         // [T, N, 3Hg]
    const float* hn;            // [T, N, Hg]
    float* dgi;                 // [T, N, 3Hg] gradient of the input-side pre-activations
    float* dgh;                 // [T, N, 3Hg] gradient of the hidden-side pre-activations (differs in the n gate)
    float* bias_partials;       // [blocks][6Hg]: column sums of dgi | dgh over this block's environments and all steps
    int T, N, Hg;
};

// Per-element backward of one cell; returns the four pre-activation gradients and the direct path to the previous hidden state.
struct CellGrad { float dr, dz, dn, dghn, dh_direct; };
__device__ __forceinline__ CellGrad gru_cell_grad(float dh, float r, float z, float n, float hn, float m)
{
    CellGrad c;
    const float dn_act = dh * (1.0f - z);
    const float dz_act = dh * (m - n);
    c.dn = dn_act * (1.0f - n * n);
    c.dz = dz_act * z * (1.0f - z);
    c.dr = (c.dn * hn) * r * (1.0f - r);
    c.dghn = c.dn * r;
    c.dh_direct = dh * z;
    return c;
}

// ---- backward scan, Hg <= 32 -------------------------------------------------------------------------------------------------
template <int HG>
__global__ void __launch_bounds__(128)
gru_scan_bwd_warp_kernel(ScanBwdArgs a)
{
    __shared__ float red[128 * 4];
    const int lane = threadIdx.x & 31;
    const int k = lane % HG;
    const int base = lane - k;
    const int64_t env = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / HG;
    const bool on = env < a.N;
    const int64_t e = on ? env : 0;
    float wr[HG], wz[HG], wn[HG];                               // column k of the three gate blocks
#pragma unroll
    for (int g = 0; g < HG; ++g) {
        wr[g] = a.whh[(int64_t)g * HG + k];
        wz[g] = a.whh[(int64_t)(HG + g) * HG + k];
        wn[g] = a.whh[(int64_t)(2 * HG + g) * HG + k];
    }
    const int64_t rs = (int64_t)a.N;
    float carry = 0.f, sr = 0.f, sz = 0.f, sn = 0.f, sgn = 0.f;
    for (int t = a.T - 1; t >= 0; --t) {
        const int64_t row = (int64_t)t * rs + e;
        const float* g = a.gates + row * 3 * HG;
        const float r = g[k], z = g[HG + k], n = g[2 * HG + k];
        const float hn = a.hn[row * HG + k], m = a.hm[row * HG + k];
        const bool dn = a.dones && a.dones[row];
        const float dh = (on ? a.dhs[row * HG + k] : 0.f) + carry;
        const CellGrad c = gru_cell_grad(dh, r, z, n, hn, m);
        if (on) {
            float* o = a.dgi + row * 3 * HG;
            o[k] = c.dr; o[HG + k] = c.dz; o[2 * HG + k] = c.dn;
            float* p = a.dgh + row * 3 * HG;
            p[k] = c.dr; p[HG + k] = c.dz; p[2 * HG + k] = c.dghn;
            sr += c.dr; sz += c.dz; sn += c.dn; sgn += c.dghn;
        }
        float acc = c.dh_direct;
#pragma unroll
        for (int gg = 0; gg < HG; ++gg) {
            acc = fmaf(__shfl_sync(0xffffffffu, c.dr, base + gg), wr[gg], acc);
            acc = fmaf(__shfl_sync(0xffffffffu, c.dz, base + gg), wz[gg], acc);
            acc = fmaf(__shfl_sync(0xffffffffu, c.dghn, base + gg), wn[gg], acc);
        }
        carry = dn ? 0.f : acc;                                 // hm = keep * h_{t-1}
    }
    // bias-gradient partial of this block: sum over its environments in thread order
    red[threadIdx.x * 4 + 0] = sr; red[threadIdx.x * 4 + 1] = sz; red[threadIdx.x * 4 + 2] = sn; red[threadIdx.x * 4 + 3] = sgn;
    __syncthreads();
    if (threadIdx.x < HG) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = threadIdx.x; i < (int)blockDim.x; i += HG)
#pragma unroll
            for (int q = 0; q < 4; ++q) s[q] += red[i * 4 + q];
        float* o = a.bias_partials + (int64_t)blockIdx.x * 6 * HG;
        const int u = threadIdx.x;
        o[u] = s[0]; o[HG + u] = s[1]; o[2 * HG + u] = s[2];
        o[3 * HG + u] = s[0]; o[4 * HG + u] = s[1]; o[5 * HG + u] = s[3];
    }
}

// ---- backward scan, general Hg ------------------------------------------------------------------------------------------------
__global__ void gru_scan_bwd_smem_kernel(ScanBwdArgs a, int EB)
{
    extern __shared__ float smem[];
    const int Hg = a.Hg;
    float* w = smem;                                            // [3Hg][Hg] as in global memory
    float* db = w + 3 * Hg * Hg;                                // [2][EB][3Hg]; reused for the final reduction ([EB*Hg][4])
    for (int i = threadIdx.x; i < 3 * Hg * Hg; i += blockDim.x) w[i] = a.whh[i];
    const int le = threadIdx.x / Hg, k = threadIdx.x % Hg;
    const int64_t env = (int64_t)blockIdx.x * EB + le;
    const bool on = le < EB && env < a.N;
    const int64_t e = on ? env : 0;
    const int64_t rs = (int64_t)a.N;
    float carry = 0.f, sr = 0.f, sz = 0.f, sn = 0.f, sgn = 0.f;
    __syncthreads();
    for (int t = a.T - 1; t >= 0; --t) {
        const int64_t row = (int64_t)t * rs + e;
        const float* g = a.gates + row * 3 * Hg;
        const float r = g[k], z = g[Hg + k], n = g[2 * Hg + k];
        const float hn = a.hn[row * Hg + k], m = a.hm[row * Hg + k];
        const bool dn = a.dones && a.dones[row];
        const float dh = (on ? a.dhs[row * Hg + k] : 0.f) + carry;
        const CellGrad c = gru_cell_grad(dh, r, z, n, hn, m);
        float* cur = db + (size_t)(t & 1) * EB * 3 * Hg;
        if (le < EB) { cur[le * 3 * Hg + k] = c.dr; cur[le * 3 * Hg + Hg + k] = c.dz; cur[le * 3 * Hg + 2 * Hg + k] = c.dghn; }
        if (on) {
            float* o = a.dgi + row * 3 * Hg;
            o[k] = c.dr; o[Hg + k] = c.dz; o[2 * Hg + k] = c.dn;
            float* p = a.dgh + row * 3 * Hg;
            p[k] = c.dr; p[Hg + k] = c.dz; p[2 * Hg + k] = c.dghn;
            sr += c.dr; sz += c.dz; sn += c.dn; sgn += c.dghn;
        }
        __syncthreads();
        float acc = c.dh_direct;
        if (le < EB) {
            const float* dv = cur + le * 3 * Hg;
            for (int gg = 0; gg < 3 * Hg; ++gg) acc = fmaf(dv[gg], w[gg * Hg + k], acc);
        }
        carry = dn ? 0.f : acc;
    }
    __syncthreads();
    float* red = db;                                            // EB*Hg*4 <= 2*EB*3Hg floats
    if (le < EB) { red[threadIdx.x * 4 + 0] = sr; red[threadIdx.x * 4 + 1] = sz; red[threadIdx.x * 4 + 2] = sn; red[threadIdx.x * 4 + 3] = sgn; }
    __syncthreads();
    if (threadIdx.x < Hg) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = threadIdx.x; i < EB * Hg; i += Hg)
#pragma unroll
            for (int q = 0; q < 4; ++q) s[q] += red[i * 4 + q];
        float* o = a.bias_partials + (int64_t)blockIdx.x * 6 * Hg;
        const int u = threadIdx.x;
        o[u] = s[0]; o[Hg + u] = s[1]; o[2 * Hg + u] = s[2];
        o[3 * Hg + u] = s[0]; o[4 * Hg + u] = s[1]; o[5 * Hg + u] = s[3];
    }
}

// ---- backward scan, Hg a multiple of 4: E environments per thread (see gru_scan_fwd_tiled_kernel) ---------------------------------
// Thread (group, k) carries dL/dh[k] of E environments; W_hh is held transposed ([Hg][3Hg], rows padded by 4 floats) so that the
// 3Hg-long products run along LDS.128 loads of the weights (one per 4 E FMAs) against broadcast loads of the gate gradients.
template <int E>
__global__ void __launch_bounds__(256)
gru_scan_bwd_tiled_kernel(ScanBwdArgs a, int G)
{
    extern __shared__ float smem[];
    const int Hg = a.Hg, G3 = 3 * Hg, WS = G3 + 4;
    float* wT = smem;                                           // [Hg][WS]: wT[k][g] = W_hh[g][k]
    float* db = wT + Hg * WS;                                   // [2][G * E][3Hg]; reused for the final reduction ([G * Hg][4])
    for (int i = threadIdx.x; i < G3 * Hg; i += blockDim.x) wT[(i % Hg) * WS + (i / Hg)] = a.whh[i];
    const int grp = threadIdx.x / Hg, k = threadIdx.x % Hg;
    const int64_t env0 = ((int64_t)blockIdx.x * G + grp) * E;
    const int64_t rs = (int64_t)a.N;
    bool on[E];
    int64_t e[E];
    float carry[E];
#pragma unroll
    for (int i = 0; i < E; ++i) { on[i] = env0 + i < a.N; e[i] = on[i] ? env0 + i : 0; carry[i] = 0.f; }
    float sr = 0.f, sz = 0.f, sn = 0.f, sgn = 0.f;
    const float4* w4 = reinterpret_cast<const float4*>(wT + (size_t)k * WS);
    __syncthreads();
    for (int t = a.T - 1; t >= 0; --t) {
        float* cur = db + (size_t)(t & 1) * G * E * G3 + (size_t)grp * E * G3;
        float acc[E];
        bool dn[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int64_t row = (int64_t)t * rs + e[i];
            const float* g = a.gates + row * G3;
            const float r = g[k], z = g[Hg + k], n = g[2 * Hg + k];
            const float hn = a.hn[row * Hg + k], m = a.hm[row * Hg + k];
            dn[i] = a.dones && a.dones[row];
            const float dh = (on[i] ? a.dhs[row * Hg + k] : 0.f) + carry[i];
            const CellGrad c = gru_cell_grad(dh, r, z, n, hn, m);
            cur[i * G3 + k] = c.dr; cur[i * G3 + Hg + k] = c.dz; cur[i * G3 + 2 * Hg + k] = c.dghn;
            if (on[i]) {
                float* o = a.dgi + row * G3;
                o[k] = c.dr; o[Hg + k] = c.dz; o[2 * Hg + k] = c.dn;
                float* p = a.dgh + row * G3;
                p[k] = c.dr; p[Hg + k] = c.dz; p[2 * Hg + k] = c.dghn;
                sr += c.dr; sz += c.dz; sn += c.dn; sgn += c.dghn;
            }
            acc[i] = c.dh_direct;
        }
        __syncthreads();
        for (int g4 = 0; g4 < G3 / 4; ++g4) {
            const float4 wv = w4[g4];
#pragma unroll
            for (int i = 0; i < E; ++i) {
                const float4 dv = reinterpret_cast<const float4*>(cur + i * G3)[g4];
                acc[i] = fmaf(dv.x, wv.x, acc[i]); acc[i] = fmaf(dv.y, wv.y, acc[i]);
                acc[i] = fmaf(dv.z, wv.z, acc[i]); acc[i] = fmaf(dv.w, wv.w, acc[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < E; ++i) carry[i] = dn[i] ? 0.f : acc[i];
    }
    __syncthreads();
    float* red = db;                                            // G * Hg * 4 <= 2 * G * E * 3Hg floats
    red[threadIdx.x * 4 + 0] = sr; red[threadIdx.x * 4 + 1] = sz; red[threadIdx.x * 4 + 2] = sn; red[threadIdx.x * 4 + 3] = sgn;
    __syncthreads();
    if (threadIdx.x < Hg) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = threadIdx.x; i < G * Hg; i += Hg)
#pragma unroll
            for (int q = 0; q < 4; ++q) s[q] += red[i * 4 + q];
        float* o = a.bias_partials + (int64_t)blockIdx.x * 6 * Hg;
        const int u = threadIdx.x;
        o[u] = s[0]; o[Hg + u] = s[1]; o[2 * Hg + u] = s[2];
        o[3 * Hg + u] = s[0]; o[4 * Hg + u] = s[1]; o[5 * Hg + u] = s[3];
    }
}

// ---- cluster scans, 128 < Hg <= 512: W_hh spread over the C CTAs of a thread-block cluster ----------------------------------
// 3 Hg^2 floats of W_hh no longer fit one SM (768 KB at Hg = 256).  CTA c of a cluster owns hidden units [c U, min(Hg, (c+1) U)),
// U = ceil(Hg / C), and keeps the r, z, n rows of those units in shared memory (3U x Hg floats, ~100 KB at Hg = 256 with C = 8,
// ~194 KB at Hg = 512 with C = 16).  Thread (group, j) handles unit j of the CTA for E environments; the cluster owns G * E
// environments for all T steps, and clusters are independent of each other.
//   forward: all-gather.  Each CTA writes the masked hidden values of its units into the hidden-vector buffer of every peer over
//     distributed shared memory, double-buffered by the parity of t, so one cluster barrier per step orders the writes of step t
//     before their reads and the reads of step t before the writes of step t + 2.  The products then run as in the tiled kernel
//     (k ascending, one FMA chain per gate; rows padded to a multiple of 4 with zeros for LDS.128).
//   backward: reduce-scatter over the same row slice (no transposed copy of W_hh).  CTA c forms the gate gradients of its units,
//     the partial P_c[k] = sum over its 3U rows g (ascending) of dg[g] W_hh[g][k] for every k, and sends the slice k in units(c')
//     to CTA c'.  After the barrier each CTA adds the C partials in rank order 0..C-1 (deterministic), then dh_direct, then the
//     done cut.  Each environment moves Hg floats per step in each direction.
// Every per-environment result is independent of E, G and the cluster an environment lands in.
template <int E>
__global__ void __launch_bounds__(256)
gru_scan_fwd_cluster_kernel(ScanFwdArgs a, int G)
{
    extern __shared__ __align__(16) float smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int Hg = a.Hg, U = (Hg + C - 1) / C, HP = (Hg + 3) & ~3, WS = HP + 4;
    const int u0 = rank * U, nu = max(0, min(U, Hg - u0));      // units of this CTA: [u0, u0 + nu)
    float* w = smem;                                            // [3U][WS]: row q U + u = W_hh row q Hg + u0 + u, zero-padded
    float* hb = w + 3 * U * WS;                                 // [2][G * E][HP] gathered masked hidden vectors (zero past Hg)
    for (int i = threadIdx.x; i < 3 * U * WS; i += blockDim.x) {
        const int g = i / WS, k = i % WS, q = g / U, u = g % U;
        w[i] = (u < nu && k < Hg) ? a.whh[(int64_t)(q * Hg + u0 + u) * Hg + k] : 0.f;
    }
    for (int i = threadIdx.x; i < 2 * G * E * HP; i += blockDim.x) hb[i] = 0.f;
    const int grp = threadIdx.x / U, j = threadIdx.x % U;
    const bool unit = j < nu;
    const int ju = u0 + (unit ? j : 0);                         // global hidden unit of this thread
    const int64_t env0 = ((int64_t)(blockIdx.x / C) * G + grp) * E;
    const float br = unit ? a.bhh[ju] : 0.f, bz = unit ? a.bhh[Hg + ju] : 0.f, bn = unit ? a.bhh[2 * Hg + ju] : 0.f;
    const int64_t rs = (int64_t)a.N;
    bool on[E];
    int64_t e[E];
    float h[E], gr[E], gz[E], gn[E];
    unsigned char dn[E];
#pragma unroll
    for (int i = 0; i < E; ++i) {
        on[i] = unit && env0 + i < a.N;
        e[i] = env0 + i < a.N ? env0 + i : 0;
        h[i] = (on[i] && a.hx0) ? a.hx0[e[i] * Hg + ju] : 0.f;
        const float* g = a.gi + e[i] * 3 * Hg;
        gr[i] = g[ju]; gz[i] = g[Hg + ju]; gn[i] = g[2 * Hg + ju];
        dn[i] = a.dones ? a.dones[e[i]] : 0;
    }
    const float4* wr4 = reinterpret_cast<const float4*>(w + (size_t)j * WS);
    const float4* wz4 = reinterpret_cast<const float4*>(w + (size_t)(U + j) * WS);
    const float4* wn4 = reinterpret_cast<const float4*>(w + (size_t)(2 * U + j) * WS);
    cluster.sync();                                             // every peer's buffers are initialised before the first remote write
    for (int t = 0; t < a.T; ++t) {
        float gr1[E], gz1[E], gn1[E];
        unsigned char dn1[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            gr1[i] = gz1[i] = gn1[i] = 0.f; dn1[i] = 0;
            if (t + 1 < a.T) {
                const int64_t row1 = (int64_t)(t + 1) * rs + e[i];
                const float* g1 = a.gi + row1 * 3 * Hg;
                gr1[i] = g1[ju]; gz1[i] = g1[Hg + ju]; gn1[i] = g1[2 * Hg + ju];
                if (a.dones) dn1[i] = a.dones[row1];
            }
        }
        float* cur = hb + (size_t)(t & 1) * G * E * HP + (size_t)grp * E * HP;
        float m[E], ar[E], az[E], an[E];
#pragma unroll
        for (int i = 0; i < E; ++i) { m[i] = dn[i] ? 0.f : h[i]; ar[i] = br; az[i] = bz; an[i] = bn; }   // recurrent_ppo.py:84
        if (unit)
            for (int q = 0; q < C; ++q) {
                float* peer = cluster.map_shared_rank(cur, q);
#pragma unroll
                for (int i = 0; i < E; ++i) peer[i * HP + ju] = m[i];
            }
        cluster.sync();                                         // one barrier per step (arrive.release / wait.acquire)
        for (int k4 = 0; k4 < HP / 4; ++k4) {
            const float4 a_r = wr4[k4], a_z = wz4[k4], a_n = wn4[k4];
#pragma unroll
            for (int i = 0; i < E; ++i) {
                const float4 hv = reinterpret_cast<const float4*>(cur + i * HP)[k4];
                ar[i] = fmaf(a_r.x, hv.x, ar[i]); az[i] = fmaf(a_z.x, hv.x, az[i]); an[i] = fmaf(a_n.x, hv.x, an[i]);
                ar[i] = fmaf(a_r.y, hv.y, ar[i]); az[i] = fmaf(a_z.y, hv.y, az[i]); an[i] = fmaf(a_n.y, hv.y, an[i]);
                ar[i] = fmaf(a_r.z, hv.z, ar[i]); az[i] = fmaf(a_z.z, hv.z, az[i]); an[i] = fmaf(a_n.z, hv.z, an[i]);
                ar[i] = fmaf(a_r.w, hv.w, ar[i]); az[i] = fmaf(a_z.w, hv.w, az[i]); an[i] = fmaf(a_n.w, hv.w, an[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const float r = sigmoidf_(gr[i] + ar[i]), z = sigmoidf_(gz[i] + az[i]);
            const float n = tanhf(gn[i] + r * an[i]);
            h[i] = (1.0f - z) * n + z * m[i];
            if (on[i]) {
                const int64_t row = (int64_t)t * rs + e[i];
                a.hs[row * Hg + ju] = h[i];
                if (a.hm) {
                    a.hm[row * Hg + ju] = m[i];
                    float* go = a.gates + row * 3 * Hg;
                    go[ju] = r; go[Hg + ju] = z; go[2 * Hg + ju] = n;
                    a.hn[row * Hg + ju] = an[i];
                }
            }
            gr[i] = gr1[i]; gz[i] = gz1[i]; gn[i] = gn1[i]; dn[i] = dn1[i];
        }
    }
#pragma unroll
    for (int i = 0; i < E; ++i)
        if (on[i] && a.hx_out) a.hx_out[e[i] * Hg + ju] = h[i];
    cluster.sync();                                             // no CTA exits while a peer may still access its shared memory
}

template <int C, int E>
__global__ void __launch_bounds__(256)
gru_scan_bwd_cluster_kernel(ScanBwdArgs a, int G)
{
    extern __shared__ __align__(16) float smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int Hg = a.Hg, U = (Hg + C - 1) / C, U3 = 3 * U;
    const int u0 = rank * U, nu = max(0, min(U, Hg - u0));
    float* w = smem;                                            // [3U][Hg]: row q U + u = W_hh row q Hg + u0 + u (zero for u >= nu)
    float* dgb = w + (size_t)U3 * Hg;                           // [G * E][3U] this CTA's dr | dz | dghn of the current step
    float* rb = dgb + (size_t)G * E * U3;                       // [2][G * E][C][U] partials received from each rank, by parity of t
    for (int i = threadIdx.x; i < U3 * Hg; i += blockDim.x) {
        const int g = i / Hg, k = i % Hg, q = g / U, u = g % U;
        w[i] = u < nu ? a.whh[(int64_t)(q * Hg + u0 + u) * Hg + k] : 0.f;
    }
    const int grp = threadIdx.x / U, j = threadIdx.x % U;
    const bool unit = j < nu;
    const int ju = u0 + (unit ? j : 0);
    const int64_t env0 = ((int64_t)(blockIdx.x / C) * G + grp) * E;
    const int64_t rs = (int64_t)a.N;
    bool on[E];
    int64_t e[E];
    float carry[E];
#pragma unroll
    for (int i = 0; i < E; ++i) { on[i] = unit && env0 + i < a.N; e[i] = env0 + i < a.N ? env0 + i : 0; carry[i] = 0.f; }
    float sr = 0.f, sz = 0.f, sn = 0.f, sgn = 0.f;
    cluster.sync();
    for (int t = a.T - 1; t >= 0; --t) {
        float direct[E];
        bool dn[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int64_t row = (int64_t)t * rs + e[i];
            dn[i] = a.dones && a.dones[row];
            direct[i] = 0.f;
            if (unit) {
                const float* g = a.gates + row * 3 * Hg;
                const float r = g[ju], z = g[Hg + ju], n = g[2 * Hg + ju];
                const float hn = a.hn[row * Hg + ju], m = a.hm[row * Hg + ju];
                const float dh = (on[i] ? a.dhs[row * Hg + ju] : 0.f) + carry[i];
                const CellGrad c = gru_cell_grad(dh, r, z, n, hn, m);
                float* d = dgb + (size_t)(grp * E + i) * U3;
                d[j] = c.dr; d[U + j] = c.dz; d[2 * U + j] = c.dghn;
                if (on[i]) {
                    float* o = a.dgi + row * 3 * Hg;
                    o[ju] = c.dr; o[Hg + ju] = c.dz; o[2 * Hg + ju] = c.dn;
                    float* p = a.dgh + row * 3 * Hg;
                    p[ju] = c.dr; p[Hg + ju] = c.dz; p[2 * Hg + ju] = c.dghn;
                    sr += c.dr; sz += c.dz; sn += c.dn; sgn += c.dghn;
                }
                direct[i] = c.dh_direct;
            }
        }
        __syncthreads();
        // P_rank[k] for k = q U + j (unit j of rank q), sent to rank q; the C * E chains run side by side, each over g ascending
        float* cur = rb + (size_t)(t & 1) * G * E * C * U;
        float p[C][E];
#pragma unroll
        for (int q = 0; q < C; ++q)
#pragma unroll
            for (int i = 0; i < E; ++i) p[q][i] = 0.f;
        for (int gate = 0; gate < 3; ++gate)
            for (int u = 0; u < nu; ++u) {
                const int g = gate * U + u;
                float dv[E];
#pragma unroll
                for (int i = 0; i < E; ++i) dv[i] = dgb[(size_t)(grp * E + i) * U3 + g];
                const float* wg = w + (size_t)g * Hg;
#pragma unroll
                for (int q = 0; q < C; ++q) {
                    const float wv = wg[min(q * U + j, Hg - 1)];          // k >= Hg (past the last unit): computed, not sent
#pragma unroll
                    for (int i = 0; i < E; ++i) p[q][i] = fmaf(dv[i], wv, p[q][i]);
                }
            }
#pragma unroll
        for (int q = 0; q < C; ++q) {
            if (q * U + j >= Hg) continue;
            float* peer = cluster.map_shared_rank(cur, q);
#pragma unroll
            for (int i = 0; i < E; ++i) peer[((size_t)(grp * E + i) * C + rank) * U + j] = p[q][i];
        }
        cluster.sync();                                         // one barrier per step; also orders dgb's reads before its next writes
#pragma unroll
        for (int i = 0; i < E; ++i) {
            float acc = 0.f;
            if (unit) {
                const float* in = cur + (size_t)(grp * E + i) * C * U + j;
                acc = in[0];
                for (int src = 1; src < C; ++src) acc += in[(size_t)src * U];
                acc += direct[i];
            }
            carry[i] = dn[i] ? 0.f : acc;                       // hm = keep * h_{t-1}
        }
    }
    __syncthreads();
    // bias-gradient partial of this cluster (one part per cluster); this CTA writes the columns of its own units
    float* red = rb;                                            // G * U * 4 <= 2 * G * E * C * U floats
    red[threadIdx.x * 4 + 0] = sr; red[threadIdx.x * 4 + 1] = sz; red[threadIdx.x * 4 + 2] = sn; red[threadIdx.x * 4 + 3] = sgn;
    __syncthreads();
    if (threadIdx.x < nu) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = threadIdx.x; i < G * U; i += U)
#pragma unroll
            for (int q = 0; q < 4; ++q) s[q] += red[i * 4 + q];
        float* o = a.bias_partials + (int64_t)(blockIdx.x / C) * 6 * Hg;
        const int u = u0 + threadIdx.x;
        o[u] = s[0]; o[Hg + u] = s[1]; o[2 * Hg + u] = s[2];
        o[3 * Hg + u] = s[0]; o[4 * Hg + u] = s[1]; o[5 * Hg + u] = s[3];
    }
    cluster.sync();                                             // no CTA exits while a peer may still access its shared memory
}

// dst[idx[m], :] = src[m, :] (rows of a minibatch back to their place in the [T*N, C] sequence tensor; dst is zero elsewhere)
__global__ void scatter_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, float* __restrict__ dst,
                                    int64_t rows, int C)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * C) return;
    const int64_t m = i / C;
    const int c = (int)(i % C);
    dst[(int64_t)idx[m] * C + c] = src[i];
}

bool warp_scan_ok(int Hg) { return Hg == 8 || Hg == 16 || Hg == 32; }
int smem_scan_envs(int Hg) { int eb = 256 / Hg; return eb < 1 ? 1 : eb; }
// tiled kernels: E environments per thread, groups of Hg threads, <= 256 threads per block
bool tiled_scan_ok(int Hg) { return Hg % 4 == 0 && Hg >= 12 && Hg <= 128; }
// The scans are sequential in t: with few environments they are latency-bound and want every (environment, unit) on its own
// thread; E > 1 pays once the problem fills the GPU anyway (>= ~12 warps per SM left after the division; measured on B200 at
// Hg = 64: N = 4096 forward 1.18 -> 0.67 ms, backward 1.67 -> 1.28 ms with E = 4, while N <= 1024 is faster with E = 1).
int tiled_scan_E(int N, int Hg)
{
    const int64_t warps = (int64_t)N * Hg / 32;
    const int64_t want = 12 * 148;
    return warps / 4 >= want ? 4 : warps / 2 >= want ? 2 : 1;
}
int tiled_scan_groups(int N, int Hg, int E)
{
    int g = 256 / Hg;
    if (g < 1) g = 1;
    const int need = (N + E - 1) / E;                           // thread groups the whole problem has
    return g < need ? g : need;
}

// cluster kernels (128 < Hg <= 512): C CTAs per cluster, U units per CTA, G groups of E environments per cluster
constexpr int kScanSmemFloats = 227 * 1024 / 4;                // dynamic shared memory of one B200 block
constexpr int kClusterMaxGroups = 8;                            // <= 8 * 32 = 256 threads per CTA
struct ClusterPlan { int C, U, E, G, clusters; };
bool cluster_scan_ok(int Hg) { return Hg > 128 && Hg <= 512; }
int64_t cluster_fwd_smem_floats(int Hg, int C, int envs)
{
    const int U = (Hg + C - 1) / C, HP = (Hg + 3) & ~3;
    return (int64_t)3 * U * (HP + 4) + (int64_t)2 * envs * HP;
}
int64_t cluster_bwd_smem_floats(int Hg, int C, int envs)
{
    const int U = (Hg + C - 1) / C;
    return (int64_t)3 * U * Hg + (int64_t)envs * (3 * U + 2 * C * U);
}
// Environments per cluster: enough to cover N with one wave of clusters (148 / C of them), spread thinly at small N as the tiled
// kernels do, and at most what the shared memory left after the weight slice holds (8 at Hg = 512).  E > 1 once a cluster
// holds more than kClusterMaxGroups environments: every W_hh value read from shared memory then serves E environments.
ClusterPlan cluster_plan(int N, int Hg)
{
    ClusterPlan p;
    p.C = Hg <= 256 ? 8 : 16;
    p.U = (Hg + p.C - 1) / p.C;
    int cap = 1;
    while (cluster_fwd_smem_floats(Hg, p.C, cap + 1) <= kScanSmemFloats && cluster_bwd_smem_floats(Hg, p.C, cap + 1) <= kScanSmemFloats)
        ++cap;
    const int slots = 148 / p.C;
    const int want = (int)(((int64_t)N + slots - 1) / slots);
    int ec = want < cap ? want : cap;
    if (ec > 4 * kClusterMaxGroups) ec = 4 * kClusterMaxGroups;
    p.E = ec <= kClusterMaxGroups ? 1 : ec <= 2 * kClusterMaxGroups ? 2 : 4;
    p.G = (ec + p.E - 1) / p.E;
    while (p.G > 1 && p.G * p.E > cap) --p.G;
    p.clusters = (int)(((int64_t)N + p.G * p.E - 1) / (p.G * p.E));
    return p;
}

int scan_blocks(int N, int Hg)
{
    if (cluster_scan_ok(Hg)) return cluster_plan(N, Hg).clusters;   // bias partials: one part per cluster
    if (warp_scan_ok(Hg)) return (int)(((int64_t)N * Hg + 127) / 128);
    if (tiled_scan_ok(Hg)) { const int E = tiled_scan_E(N, Hg), per = tiled_scan_groups(N, Hg, E) * E; return (N + per - 1) / per; }
    const int eb = smem_scan_envs(Hg);
    return (N + eb - 1) / eb;
}

// grid of p.clusters clusters of p.C CTAs; refuses (instead of launching) when no such cluster fits on the device
template <typename Args>
int launch_cluster_scan(dppo_ctx* ctx, void (*kern)(Args, int), const Args& a, const ClusterPlan& p, size_t smem, cudaStream_t st,
                        const char* what)
{
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        (p.C > 8 && cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess))
        DPPO_FAIL(ctx, "%s: cudaFuncSetAttribute failed (%s)", what, cudaGetErrorString(cudaGetLastError()));
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)p.clusters * p.C); lc.blockDim = dim3(p.G * p.U); lc.dynamicSmemBytes = smem; lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = p.C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    lc.attrs = attr; lc.numAttrs = 1;
    int active = 0;
    if (cudaOccupancyMaxActiveClusters(&active, kern, &lc) != cudaSuccess || active < 1)
        DPPO_FAIL(ctx, "%s: no %d-CTA cluster with %zu bytes of shared memory per CTA fits on this device (%s)", what, p.C, smem,
                  cudaGetErrorString(cudaGetLastError()));
    cudaLaunchKernelEx(&lc, kern, a, p.G);
    DPPO_CHECK_LAUNCH(ctx, what);
    return 0;
}

int launch_scan_fwd(dppo_ctx* ctx, const ScanFwdArgs& a, cudaStream_t st)
{
    if (cluster_scan_ok(a.Hg)) {
        const ClusterPlan p = cluster_plan(a.N, a.Hg);
        const size_t smem = (size_t)cluster_fwd_smem_floats(a.Hg, p.C, p.G * p.E) * sizeof(float);
        if (p.E == 4) return launch_cluster_scan(ctx, gru_scan_fwd_cluster_kernel<4>, a, p, smem, st, "gru_scan_fwd_cluster_kernel");
        if (p.E == 2) return launch_cluster_scan(ctx, gru_scan_fwd_cluster_kernel<2>, a, p, smem, st, "gru_scan_fwd_cluster_kernel");
        return launch_cluster_scan(ctx, gru_scan_fwd_cluster_kernel<1>, a, p, smem, st, "gru_scan_fwd_cluster_kernel");
    }
    const int blocks = scan_blocks(a.N, a.Hg);
    if (a.Hg == 8) gru_scan_fwd_warp_kernel<8><<<blocks, 128, 0, st>>>(a);
    else if (a.Hg == 16) gru_scan_fwd_warp_kernel<16><<<blocks, 128, 0, st>>>(a);
    else if (a.Hg == 32) gru_scan_fwd_warp_kernel<32><<<blocks, 128, 0, st>>>(a);
    else if (tiled_scan_ok(a.Hg)) {
        const int E = tiled_scan_E(a.N, a.Hg), G = tiled_scan_groups(a.N, a.Hg, E);
        const size_t smem = ((size_t)3 * a.Hg * (a.Hg + 4) + (size_t)2 * G * E * a.Hg) * sizeof(float);
        if (smem > 227 * 1024) DPPO_FAIL(ctx, "gru scan: gru_hidden_dim %d too large for shared memory", a.Hg);
#define SCAN_FWD(E_)                                                                                                  \
    do {                                                                                                              \
        cudaFuncSetAttribute(gru_scan_fwd_tiled_kernel<E_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
        gru_scan_fwd_tiled_kernel<E_><<<blocks, G * a.Hg, smem, st>>>(a, G);                                          \
    } while (0)
        if (E == 4) SCAN_FWD(4); else if (E == 2) SCAN_FWD(2); else SCAN_FWD(1);
#undef SCAN_FWD
    } else {
        const int eb = smem_scan_envs(a.Hg);
        const size_t smem = ((size_t)3 * a.Hg * a.Hg + (size_t)2 * eb * a.Hg) * sizeof(float);
        if (smem > 200 * 1024) DPPO_FAIL(ctx, "gru scan: gru_hidden_dim %d too large for shared memory", a.Hg);
        cudaFuncSetAttribute(gru_scan_fwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gru_scan_fwd_smem_kernel<<<blocks, eb * a.Hg, smem, st>>>(a, eb);
    }
    DPPO_CHECK_LAUNCH(ctx, "gru_scan_fwd_kernel");
    return 0;
}

int launch_scan_bwd(dppo_ctx* ctx, const ScanBwdArgs& a, cudaStream_t st)
{
    if (cluster_scan_ok(a.Hg)) {
        const ClusterPlan p = cluster_plan(a.N, a.Hg);
        const size_t smem = (size_t)cluster_bwd_smem_floats(a.Hg, p.C, p.G * p.E) * sizeof(float);
#define SCAN_BWD(C_, E_) return launch_cluster_scan(ctx, gru_scan_bwd_cluster_kernel<C_, E_>, a, p, smem, st, "gru_scan_bwd_cluster_kernel")
        if (p.C == 8) { if (p.E == 4) SCAN_BWD(8, 4); if (p.E == 2) SCAN_BWD(8, 2); SCAN_BWD(8, 1); }
        if (p.E == 4) SCAN_BWD(16, 4); if (p.E == 2) SCAN_BWD(16, 2); SCAN_BWD(16, 1);
#undef SCAN_BWD
    }
    const int blocks = scan_blocks(a.N, a.Hg);
    if (a.Hg == 8) gru_scan_bwd_warp_kernel<8><<<blocks, 128, 0, st>>>(a);
    else if (a.Hg == 16) gru_scan_bwd_warp_kernel<16><<<blocks, 128, 0, st>>>(a);
    else if (a.Hg == 32) gru_scan_bwd_warp_kernel<32><<<blocks, 128, 0, st>>>(a);
    else if (tiled_scan_ok(a.Hg)) {
        const int E = tiled_scan_E(a.N, a.Hg), G = tiled_scan_groups(a.N, a.Hg, E);
        const size_t smem = ((size_t)a.Hg * (3 * a.Hg + 4) + (size_t)2 * G * E * 3 * a.Hg) * sizeof(float);
        if (smem > 227 * 1024) DPPO_FAIL(ctx, "gru scan: gru_hidden_dim %d too large for shared memory", a.Hg);
#define SCAN_BWD(E_)                                                                                                  \
    do {                                                                                                              \
        cudaFuncSetAttribute(gru_scan_bwd_tiled_kernel<E_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
        gru_scan_bwd_tiled_kernel<E_><<<blocks, G * a.Hg, smem, st>>>(a, G);                                          \
    } while (0)
        if (E == 4) SCAN_BWD(4); else if (E == 2) SCAN_BWD(2); else SCAN_BWD(1);
#undef SCAN_BWD
    } else {
        const int eb = smem_scan_envs(a.Hg);
        const size_t smem = ((size_t)3 * a.Hg * a.Hg + (size_t)2 * eb * 3 * a.Hg) * sizeof(float);
        if (smem > 200 * 1024) DPPO_FAIL(ctx, "gru scan: gru_hidden_dim %d too large for shared memory", a.Hg);
        cudaFuncSetAttribute(gru_scan_bwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gru_scan_bwd_smem_kernel<<<blocks, eb * a.Hg, smem, st>>>(a, eb);
    }
    DPPO_CHECK_LAUNCH(ctx, "gru_scan_bwd_kernel");
    return 0;
}

int check_desc(dppo_ctx* ctx, const dppo_rnn_desc* d)
{
    if (!d || d->obs_dim < 1 || d->hidden < 1 || d->gru_hidden < 1 || d->act_dim < 1 || (d->continuous != 0 && d->continuous != 1))
        DPPO_FAIL(ctx, "rnn: bad descriptor");
    if (d->gru_hidden > 512) DPPO_FAIL(ctx, "rnn: gru_hidden_dim %d > 512 is not supported", d->gru_hidden);
    if (d->hidden > 512) DPPO_FAIL(ctx, "rnn: network_hidden_dim %d > 512 is not supported", d->hidden);
    if (d->act_dim > DPPO_MAX_ACT) DPPO_FAIL(ctx, "rnn: more than %d actions", DPPO_MAX_ACT);
    return 0;
}

struct RnnWs {
    float *x, *gi, *hs, *hm, *gates, *hn, *h3, *d3, *dhm, *dhs, *dgi, *dgh, *d1;
    float *p1, *pih, *phh, *p3, *c1, *bp, *hp;
    int s1, sih, shh, s3, tiles1, scan_parts, head_blocks, head_stride;
    int64_t bytes;
};

RnnWs carve_rnn(const dppo_rnn_desc* d, int64_t B, int64_t N, int64_t M, int training, int sm_count, char* base)
{
    dppo_ctx fake = {}; fake.sm_count = sm_count;
    const int64_t D = d->obs_dim, H = d->hidden, Hg = d->gru_hidden, A = d->act_dim;
    RnnWs w = {};
    int64_t o = 0;
    auto take = [&](int64_t floats) { float* p = reinterpret_cast<float*>(base + o); o += align_up(floats * 4, 256); return p; };
    w.x = take(B * H); w.gi = take(B * 3 * Hg); w.hs = take(B * Hg); w.h3 = take(M * 2 * H);
    if (training) {
        w.hm = take(B * Hg); w.gates = take(B * 3 * Hg); w.hn = take(B * Hg);
        w.d3 = take(M * 2 * H); w.dhm = take(M * Hg); w.dhs = take(B * Hg);
        w.dgi = take(B * 3 * Hg); w.dgh = take(B * 3 * Hg); w.d1 = take(B * H);
        w.s1 = dppo_wgrad_splits(&fake, B, (int)H, (int)D);
        w.sih = dppo_wgrad_splits(&fake, B, (int)(3 * Hg), (int)H);
        w.shh = dppo_wgrad_splits(&fake, B, (int)(3 * Hg), (int)Hg);
        w.s3 = dppo_wgrad_splits(&fake, M, (int)(2 * H), (int)Hg);
        w.p1 = take((int64_t)w.s1 * H * D);
        w.pih = take((int64_t)w.sih * 3 * Hg * H);
        w.phh = take((int64_t)w.shh * 3 * Hg * Hg);
        w.p3 = take((int64_t)w.s3 * 2 * H * Hg);
        w.tiles1 = dppo_gemm_row_tiles(B, (int)H);
        w.c1 = take((int64_t)w.tiles1 * H);
        w.scan_parts = scan_blocks((int)N, (int)Hg);
        w.bp = take((int64_t)w.scan_parts * 6 * Hg);
        w.head_blocks = head_train_blocks(&fake, M, (int)H, (int)A);
        w.head_stride = (int)align_up(head_partial_floats((int)H, (int)A), 4);
        w.hp = take((int64_t)w.head_blocks * w.head_stride);
    }
    w.bytes = o;
    return w;
}

int rnn_sm_count()
{
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms > 148 ? sms : 148;
}

// base Linear+Tanh, input projection and the forward scan over the whole rollout
int rnn_trunk_forward(dppo_ctx* ctx, const dppo_rnn_desc* d, const dppo_rnn_layout& L, const float* params, const float* obs,
                      const unsigned char* dones, const float* hx0, int T, int N, const RnnWs& w, int training, float* hx_out,
                      cudaStream_t st)
{
    const int D = d->obs_dim, H = d->hidden, Hg = d->gru_hidden;
    const int64_t B = (int64_t)T * N;
    if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, obs, D, nullptr, params + L.w1, D, params + L.b1, w.x, H, B, H, D, st)) return 1;
    if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS, w.x, H, nullptr, params + L.wih, H, params + L.bih, w.gi, 3 * Hg, B, 3 * Hg, H, st)) return 1;
    ScanFwdArgs a;
    a.gi = w.gi; a.whh = params + L.whh; a.bhh = params + L.bhh; a.dones = dones; a.hx0 = hx0;
    a.hs = w.hs; a.hm = training ? w.hm : nullptr; a.gates = training ? w.gates : nullptr; a.hn = training ? w.hn : nullptr;
    a.hx_out = hx_out; a.T = T; a.N = N; a.Hg = Hg;
    return launch_scan_fwd(ctx, a, st);
}

}  // namespace

extern "C" int dppo_rnn_layout_compute(const dppo_rnn_desc* d, dppo_rnn_layout* L)
{
    if (!d || !L || d->obs_dim < 1 || d->hidden < 1 || d->gru_hidden < 1 || d->act_dim < 1 || (d->continuous != 0 && d->continuous != 1))
        return 1;
    const int64_t D = d->obs_dim, H = d->hidden, Hg = d->gru_hidden, A = d->act_dim;
    int64_t o = 0;
    auto take = [&](int64_t n) { int64_t p = o; o += (n + 3) / 4 * 4; return p; };
    L->w1 = take(H * D); L->b1 = take(H);
    L->wih = take(3 * Hg * H); L->whh = take(3 * Hg * Hg); L->bih = take(3 * Hg); L->bhh = take(3 * Hg);
    L->w3 = take(2 * H * Hg); L->b3 = take(2 * H);
    L->wa = take(A * H); L->ba = take(A);
    L->wc = take(H); L->bc = take(1);
    L->log_std = d->continuous ? take(A) : -1;
    L->total = o;
    return 0;
}

extern "C" int64_t dppo_rnn_workspace_bytes(const dppo_rnn_desc* d, int T, int N, int64_t M, int training)
{
    if (!d || T < 1 || N < 1 || M < 1) return 0;
    return carve_rnn(d, (int64_t)T * N, N, M, training, rnn_sm_count(), nullptr).bytes + 256;
}

extern "C" int dppo_rnn_forward(dppo_ctx* ctx, const dppo_rnn_desc* d, const float* params, const float* obs,
                                const unsigned char* prev_dones, const float* hx0, int T, int N, int heads, float* logits,
                                float* values, float* hx_out, void* ws, int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (check_desc(ctx, d)) return 1;
    if (!params || !obs || !ws || T < 1 || N < 1) DPPO_FAIL(ctx, "rnn_forward: bad arguments");
    if ((heads & 1) && !logits) DPPO_FAIL(ctx, "rnn_forward: logits is null");
    if ((heads & 2) && !values) DPPO_FAIL(ctx, "rnn_forward: values is null");
    dppo_rnn_layout L;
    dppo_rnn_layout_compute(d, &L);
    const int H = d->hidden, Hg = d->gru_hidden, A = d->act_dim;
    const int64_t B = (int64_t)T * N;
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    RnnWs w = carve_rnn(d, B, N, B, 0, ctx->sm_count, base);
    if ((base - (char*)ws) + w.bytes > ws_bytes) DPPO_FAIL(ctx, "rnn_forward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if (rnn_trunk_forward(ctx, d, L, params, obs, prev_dones, hx0, T, N, w, 0, hx_out, st)) return 1;
    if ((heads & 3) == 0) return 0;
    const bool actor = heads & 1, critic = heads & 2;
    const int64_t w3off = actor ? 0 : (int64_t)H * Hg;
    const int b3off = actor ? 0 : H;
    const int n3 = (actor && critic) ? 2 * H : H;
    if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.hs, Hg, nullptr, params + L.w3 + w3off, Hg, params + L.b3 + b3off, w.h3, n3, B, n3, Hg, st)) return 1;
    const float* ha = actor ? w.h3 : nullptr;
    const float* hc = critic ? (actor ? w.h3 + H : w.h3) : nullptr;
    return launch_head_eval(ctx, ha, hc, n3, params + L.wa, params + L.ba, params + L.wc, params + L.bc, logits, values, B, H, A, 0, st);
}

extern "C" int dppo_rnn_grad_minibatch(dppo_ctx* ctx, const dppo_rnn_desc* d, const float* params, float* grads, const float* obs,
                                       const unsigned char* prev_dones, const float* hx0, int T, int N, const void* actions,
                                       const float* old_log_probs, const float* adv, const float* returns, const double* adv_stats,
                                       const int32_t* idx, int64_t M, const dppo_hyper* hy, float* losses, void* ws,
                                       int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (check_desc(ctx, d)) return 1;
    if (!params || !grads || !obs || !actions || !old_log_probs || !adv || !returns || !hy || !ws || !losses)
        DPPO_FAIL(ctx, "rnn_grad_minibatch: null argument");
    if (T < 1 || N < 1 || M < 1 || M > (int64_t)T * N) DPPO_FAIL(ctx, "rnn_grad_minibatch: bad shape T=%d N=%d M=%lld", T, N, (long long)M);
    if (!idx && M != (int64_t)T * N) DPPO_FAIL(ctx, "rnn_grad_minibatch: a partial minibatch needs row indices");
    if (hy->advantage_norm && (!adv_stats || hy->adv_count < 2)) DPPO_FAIL(ctx, "rnn_grad_minibatch: advantage_norm needs adv_stats and adv_count >= 2");
    if (!head_train_supported(d->hidden, d->act_dim))
        DPPO_FAIL(ctx, "rnn_grad_minibatch: the head kernel's per-warp accumulators, 9 (act_dim + 1) hidden = %d floats, exceed its 200 KB "
                  "of shared memory", 9 * (d->act_dim + 1) * d->hidden);
    dppo_rnn_layout L;
    dppo_rnn_layout_compute(d, &L);
    const int D = d->obs_dim, H = d->hidden, Hg = d->gru_hidden, A = d->act_dim;
    const int64_t B = (int64_t)T * N;
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    RnnWs w = carve_rnn(d, B, N, M, 1, ctx->sm_count, base);
    if ((base - (char*)ws) + w.bytes > ws_bytes) DPPO_FAIL(ctx, "rnn_grad_minibatch: workspace too small (%lld < %lld)", (long long)ws_bytes, (long long)w.bytes + 256);
    cudaStream_t st = (cudaStream_t)stream;
    const float inv_m = 1.0f / (float)(hy->loss_denominator > 0 ? hy->loss_denominator : M);

    // full-sequence forward with the current parameters (recurrent_ppo.py:337), then the minibatch rows (:340-341)
    if (rnn_trunk_forward(ctx, d, L, params, obs, prev_dones, hx0, T, N, w, 1, nullptr, st)) return 1;
    if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.hs, Hg, idx, params + L.w3, Hg, params + L.b3, w.h3, 2 * H, M, 2 * H, Hg, st)) return 1;

    // heads + PPO loss (:343-359) + backward into the first head layers
    HeadTrainArgs ha;
    ha.h3 = w.h3; ha.d3 = w.d3;
    ha.wa = params + L.wa; ha.ba = params + L.ba; ha.wc = params + L.wc; ha.bc = params + L.bc;
    ha.log_std = d->continuous ? params + L.log_std : nullptr;
    ha.idx = idx;
    ha.actions_i = d->continuous ? nullptr : static_cast<const int32_t*>(actions);
    ha.actions_f = d->continuous ? static_cast<const float*>(actions) : nullptr;
    ha.old_logp = old_log_probs; ha.adv = adv; ha.ret = returns;
    ha.adv_stats = adv_stats; ha.adv_count = hy->adv_count; ha.advantage_norm = hy->advantage_norm;
    ha.M = M; ha.H = H; ha.A = A;
    ha.clip = hy->ppo_clip; ha.vw = hy->value_loss_weight; ha.beta = hy->entropy_beta; ha.inv_m = inv_m;
    ha.partials = w.hp; ha.partial_stride = w.head_stride;
    ha.rev = 0; ha.keep_d3 = 0; ha.h3_first = 0;
    if (launch_head_train_kernel(ctx, ha, d->continuous, w.head_blocks, st)) return 1;

    // d(loss)/d(h_t): rows of the minibatch, zero for every other (t, env)
    float* dh_rows = idx ? w.dhm : w.dhs;
    if (dppo_gemm_nn(ctx, w.d3, 2 * H, params + L.w3, Hg, dh_rows, Hg, M, Hg, 2 * H, st)) return 1;
    if (idx) {
        if (cudaMemsetAsync(w.dhs, 0, (size_t)B * Hg * sizeof(float), st) != cudaSuccess) DPPO_FAIL(ctx, "rnn_grad_minibatch: memset failed");
        const int64_t n = M * Hg;
        scatter_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w.dhm, idx, w.dhs, M, Hg);
        DPPO_CHECK_LAUNCH(ctx, "scatter_rows_kernel");
    }

    // back-propagation through time over the whole rollout
    ScanBwdArgs b;
    b.dhs = w.dhs; b.whh = params + L.whh; b.dones = prev_dones; b.hm = w.hm; b.gates = w.gates; b.hn = w.hn;
    b.dgi = w.dgi; b.dgh = w.dgh; b.bias_partials = w.bp; b.T = T; b.N = N; b.Hg = Hg;
    if (launch_scan_bwd(ctx, b, st)) return 1;

    // into the base layer (tanh' and the bias-gradient column sums fused), then the weight gradients as split-K partials
    if (dppo_gemm_nn_tanh_bwd(ctx, w.dgi, 3 * Hg, params + L.wih, H, w.x, H, w.d1, H, w.c1, B, H, 3 * Hg, st)) return 1;
    if (dppo_wgrad(ctx, w.d3, 2 * H, w.hs, Hg, idx, w.p3, w.s3, M, 2 * H, Hg, st)) return 1;
    if (dppo_wgrad(ctx, w.dgi, 3 * Hg, w.x, H, nullptr, w.pih, w.sih, B, 3 * Hg, H, st)) return 1;
    if (dppo_wgrad(ctx, w.dgh, 3 * Hg, w.hm, Hg, nullptr, w.phh, w.shh, B, 3 * Hg, Hg, st)) return 1;
    if (dppo_wgrad(ctx, w.d1, H, obs, D, nullptr, w.p1, w.s1, B, H, D, st)) return 1;

    GradSegTable tab;
    int n = 0;
    auto seg = [&](int64_t dst, int64_t count, const float* src, int64_t stride, int nparts) {
        tab.seg[n].dst = dst; tab.seg[n].count = count; tab.seg[n].src = src; tab.seg[n].stride = stride;
        tab.seg[n].nparts = nparts; tab.seg[n].pad = 0; ++n;
    };
    const HeadOffsets ho = head_offsets(H, A);
    seg(L.w1, (int64_t)H * D, w.p1, (int64_t)H * D, w.s1);
    seg(L.b1, H, w.c1, H, w.tiles1);
    seg(L.wih, (int64_t)3 * Hg * H, w.pih, (int64_t)3 * Hg * H, w.sih);
    seg(L.whh, (int64_t)3 * Hg * Hg, w.phh, (int64_t)3 * Hg * Hg, w.shh);
    seg(L.bih, 3 * Hg, w.bp, 6 * Hg, w.scan_parts);
    seg(L.bhh, 3 * Hg, w.bp + 3 * Hg, 6 * Hg, w.scan_parts);
    seg(L.w3, (int64_t)2 * H * Hg, w.p3, (int64_t)2 * H * Hg, w.s3);
    seg(L.b3, 2 * H, w.hp + ho.b3, w.head_stride, w.head_blocks);
    seg(L.wa, (int64_t)A * H, w.hp, w.head_stride, w.head_blocks);
    seg(L.ba, A, w.hp + ho.dba, w.head_stride, w.head_blocks);
    seg(L.wc, H, w.hp + ho.dwc, w.head_stride, w.head_blocks);
    seg(L.bc, 1, w.hp + ho.dbc, w.head_stride, w.head_blocks);
    if (d->continuous) seg(L.log_std, A, w.hp + ho.dls, w.head_stride, w.head_blocks);
    tab.nseg = n;
    return launch_grad_reduce(ctx, tab, grads, L.total, w.hp + ho.loss, w.head_blocks, w.head_stride, hy->value_loss_weight,
                              hy->entropy_beta, inv_m, losses, hy->grad_sumsq, st);
}
