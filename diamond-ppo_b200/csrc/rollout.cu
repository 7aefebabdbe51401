// Rollout-buffer storage and batched action sampling (diamond/ppo.py:153-186, 73-82;
// continuous_ppo.py:83-93; recurrent_ppo.py:219-221).
#include <math_constants.h>

#include "common.cuh"

namespace {

// Philox4x32-10 (Salmon et al. 2011): counter-based, so a draw is a pure function of
// (seed, env id, draw counter) and never depends on launch geometry or on the number of GPUs.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return ctr;
}
// The top 24 bits of a word -> a uniform in the open interval (0, 1).  For x >> 8 == 0xFFFFFF the sum 16777215.5f rounds (to
// even) up to 2^24, so the top word is clamped to the largest float below 1: a categorical draw's target u*s then stays below
// s (s >= 1) and the walk stops at an action whose probability is not zero.
__device__ __forceinline__ float u01(uint32_t x)
{
    return fminf(((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f), 0x1.fffffep-1f);
}

// Draw-counter tag of Gaussian dimension pair p (dimensions 2p, 2p + 1): t = p + 1, low byte in counter bits 56-63 and the next
// byte in bits 48-55.  Non-zero (0 is the categorical stream) and distinct for every pair up to p = 65534 while the draw counter
// stays below 2^48.  Pairs 0-254 get (p + 1) << 56, so their streams are those of the one-byte tag.
__device__ __forceinline__ uint64_t gaussian_pair_tag(int p)
{
    const uint64_t t = (uint64_t)p + 1;
    return ((t & 0xFF) << 56) | ((t >> 8) << 48);
}

__global__ void sample_categorical_kernel(const float* __restrict__ logits, int N, int A, uint64_t seed, uint64_t counter,
                                          const unsigned long long* __restrict__ counter_base, int64_t env_offset,
                                          int64_t* __restrict__ actions, float* __restrict__ logp)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    if (counter_base) counter += *counter_base;
    const float* z = logits + (int64_t)e * A;
    float mx = -CUDART_INF_F;
    for (int j = 0; j < A; ++j) mx = fmaxf(mx, z[j]);
    float s = 0.f;
    for (int j = 0; j < A; ++j) s += expf(z[j] - mx);
    const uint64_t env = (uint64_t)(env_offset + e);
    const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)counter, (uint32_t)(counter >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float target = u01(r.x) * s;
    float cum = 0.f;
    int a = A - 1;
    for (int j = 0; j < A; ++j) {
        cum += expf(z[j] - mx);
        if (cum > target) { a = j; break; }
    }
    actions[e] = a;
    if (logp) logp[e] = z[a] - (mx + logf(s));
}

// Greedy action of a categorical policy: torch.argmax(logits, -1) -- the first index of the maximum, where a NaN counts as the
// maximum (so the first NaN of a row wins).  The log-prob is sample_categorical_kernel's formula.
__global__ void select_greedy_categorical_kernel(const float* __restrict__ logits, int N, int A, int64_t* __restrict__ actions,
                                                 float* __restrict__ logp)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    const float* z = logits + (int64_t)e * A;
    float best = z[0];
    int a = 0;
    for (int j = 1; j < A && !isnan(best); ++j) {
        const float v = z[j];
        if (isnan(v) || v > best) { best = v; a = j; }
    }
    actions[e] = a;
    if (logp) {
        float mx = -CUDART_INF_F;
        for (int j = 0; j < A; ++j) mx = fmaxf(mx, z[j]);
        float s = 0.f;
        for (int j = 0; j < A; ++j) s += expf(z[j] - mx);
        logp[e] = z[a] - (mx + logf(s));
    }
}

__global__ void sample_gaussian_kernel(const float* __restrict__ mean, const float* __restrict__ log_std, int N, int A,
                                       uint64_t seed, uint64_t counter, const unsigned long long* __restrict__ counter_base,
                                       int64_t env_offset, float* __restrict__ actions, float* __restrict__ logp)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    if (counter_base) counter += *counter_base;
    const uint64_t env = (uint64_t)(env_offset + e);
    float lp = 0.f;
    for (int j0 = 0; j0 < A; j0 += 2) {
        const uint64_t c = counter ^ gaussian_pair_tag(j0 / 2);
        const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)c, (uint32_t)(c >> 32)),
                                      make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const float rad = sqrtf(-2.0f * logf(u01(r.x)));
        float sn, cs;
        sincosf(6.28318530717958647692f * u01(r.y), &sn, &cs);
        const float n[2] = {rad * cs, rad * sn};
        for (int d = 0; d < 2 && j0 + d < A; ++d) {
            const int j = j0 + d;
            const float sigma = expf(log_std[j]);
            const float a = mean[(int64_t)e * A + j] + sigma * n[d];
            actions[(int64_t)e * A + j] = a;
            const float diff = a - mean[(int64_t)e * A + j];
            lp += -(diff * diff) / (2.0f * sigma * sigma) - logf(sigma) - 0.91893853320467274178f;
        }
    }
    if (logp) logp[e] = lp;
}

// One packed host record -> row t of the time-major device buffers (see dppo.h for the record layout).
__global__ void store_step_kernel(const unsigned char* __restrict__ rec, int t, int N, int D, int A, int continuous,
                                  float* __restrict__ obs, float* __restrict__ next_obs, void* __restrict__ actions,
                                  float* __restrict__ rewards, float* __restrict__ terms, float* __restrict__ truncs)
{
    const int64_t nd = (int64_t)N * D;
    const float* r_obs = reinterpret_cast<const float*>(rec);
    const float* r_nobs = r_obs + nd;
    const double* r_rew = reinterpret_cast<const double*>(r_nobs + nd);                  // 8*nd bytes in: 8-byte aligned
    const unsigned char* r_act = reinterpret_cast<const unsigned char*>(r_rew + N);
    const int64_t act_bytes = continuous ? (int64_t)N * A * 4 : (int64_t)N * 8;
    const unsigned char* r_term = r_act + act_bytes;
    const unsigned char* r_trunc = r_term + N;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = tid; i < nd; i += stride) {
        obs[(int64_t)t * nd + i] = r_obs[i];
        next_obs[(int64_t)t * nd + i] = r_nobs[i];
    }
    for (int64_t i = tid; i < N; i += stride) {
        rewards[(int64_t)t * N + i] = (float)r_rew[i];                                   // ppo.py:230
        terms[(int64_t)t * N + i] = r_term[i] ? 1.0f : 0.0f;                             // ppo.py:231
        truncs[(int64_t)t * N + i] = r_trunc[i] ? 1.0f : 0.0f;                           // ppo.py:232
    }
    if (continuous) {
        const float* a = reinterpret_cast<const float*>(r_act);
        float* dst = reinterpret_cast<float*>(actions) + (int64_t)t * N * A;
        for (int64_t i = tid; i < (int64_t)N * A; i += stride) dst[i] = a[i];
    } else {
        const int64_t* a = reinterpret_cast<const int64_t*>(r_act);
        int32_t* dst = reinterpret_cast<int32_t*>(actions) + (int64_t)t * N;
        for (int64_t i = tid; i < N; i += stride) dst[i] = (int32_t)a[i];                // ppo.py:229
    }
}

}  // namespace

extern "C" int64_t dppo_step_record_bytes(int N, int D, int act_dim, int continuous)
{
    const int64_t nd = (int64_t)N * D;
    int64_t b = 2 * nd * 4;                        // obs, next_obs
    b += (int64_t)N * 8;                           // rewards f64
    b += continuous ? (int64_t)N * act_dim * 4 : (int64_t)N * 8;
    b += 2 * (int64_t)N;                           // terminations, truncations (u8)
    return b;
}

extern "C" int dppo_buffer_store_step(dppo_ctx* ctx, const void* record, int t, int N, int D, int act_dim, int continuous,
                                      float* obs, float* next_obs, void* actions, float* rewards, float* terminations,
                                      float* truncations, void* stream)
{
    if (!ctx) return 1;
    if (N <= 0 || D <= 0 || t < 0) DPPO_FAIL(ctx, "buffer_store_step: bad shape N=%d D=%d t=%d", N, D, t);
    if ((reinterpret_cast<uintptr_t>(record) & 7u) != 0) DPPO_FAIL(ctx, "buffer_store_step: record must be 8-byte aligned");
    int64_t work = (int64_t)N * D;
    int blocks = (int)((work + 255) / 256);
    if (blocks > 4 * ctx->sm_count) blocks = 4 * ctx->sm_count;
    store_step_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const unsigned char*)record, t, N, D, act_dim, continuous, obs,
                                                                next_obs, actions, rewards, terminations, truncations);
    DPPO_CHECK_LAUNCH(ctx, "store_step_kernel");
    return 0;
}

extern "C" int dppo_sample_categorical(dppo_ctx* ctx, const float* logits, int N, int A, uint64_t seed, uint64_t counter,
                                       int64_t env_offset, int64_t* actions, float* log_probs, void* stream)
{
    if (!ctx) return 1;
    if (N <= 0 || A <= 0) DPPO_FAIL(ctx, "sample_categorical: bad shape N=%d A=%d", N, A);
    sample_categorical_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(logits, N, A, seed, counter, ctx->draw_base, env_offset, actions, log_probs);
    DPPO_CHECK_LAUNCH(ctx, "sample_categorical_kernel");
    return 0;
}

extern "C" int dppo_select_greedy_categorical(dppo_ctx* ctx, const float* logits, int N, int A, int64_t* actions, float* log_probs,
                                              void* stream)
{
    if (!ctx) return 1;
    if (N <= 0 || A <= 0) DPPO_FAIL(ctx, "select_greedy_categorical: bad shape N=%d A=%d", N, A);
    if (!logits || !actions) DPPO_FAIL(ctx, "select_greedy_categorical: null argument");
    select_greedy_categorical_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(logits, N, A, actions, log_probs);
    DPPO_CHECK_LAUNCH(ctx, "select_greedy_categorical_kernel");
    return 0;
}

extern "C" int dppo_sample_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, int N, int A, uint64_t seed,
                                    uint64_t counter, int64_t env_offset, float* actions, float* log_probs, void* stream)
{
    if (!ctx) return 1;
    if (N <= 0 || A <= 0) DPPO_FAIL(ctx, "sample_gaussian: bad shape N=%d A=%d", N, A);
    sample_gaussian_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(mean, log_std, N, A, seed, counter, ctx->draw_base, env_offset, actions, log_probs);
    DPPO_CHECK_LAUNCH(ctx, "sample_gaussian_kernel");
    return 0;
}

extern "C" int dppo_set_draw_counter_base(dppo_ctx* ctx, const unsigned long long* counter_base_dev)
{
    if (!ctx) return 1;
    ctx->draw_base = counter_base_dev;
    return 0;
}
