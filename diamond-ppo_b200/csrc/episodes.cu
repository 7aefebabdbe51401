// Device-side episode statistics (SURVEY.md 8 f4): replaces the per-step host `Ticker.tick(rewards, dones)` of the rollout loop
// (diamond/utils.py:99-123, call site diamond/ppo.py:181-182) for device-resident rollouts.
//
// The Ticker keeps a running return / length per environment, and on every finished episode appends (return, length) to a
// sliding window of the last `window` episodes, in the order it meets them: step by step, environments in index order.  Here
// the same bookkeeping runs once per rollout over the [T, N] reward / done tensors the rollout already holds on the device:
//   episode_scan_kernel   : one thread per environment walks t = 0..T-1 (coalesced along env), carries the running fp64 return
//                           and length across rollouts in ep_return / ep_len, and drops (return, length) at every done step into
//                           a [T, N] event scratch; counts the finished episodes.
//   episode_window_kernel : one block walks the rows backwards and collects the LAST min(window, finished) events in Ticker
//                           order (t ascending, env ascending) -- typically a handful of rows.
// Nothing is read back per step; the agent copies `window` + 1 numbers to pinned memory asynchronously once per rollout.
#include "common.cuh"

namespace {

__global__ void __launch_bounds__(128)
episode_scan_kernel(const float* __restrict__ rewards, const float* __restrict__ terms, const float* __restrict__ truncs, int T, int N,
                    double* __restrict__ ep_return, int* __restrict__ ep_len, double* __restrict__ ev_ret, int* __restrict__ ev_len,
                    unsigned long long* __restrict__ finished)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long mine = 0;
    if (e < N) {
        double ret = ep_return[e];
        int len = ep_len[e];
        for (int t = 0; t < T; ++t) {
            const int64_t i = (int64_t)t * N + e;
            ret += (double)rewards[i];                                   // Ticker: current_returns += rewards (float64)
            len += 1;
            const bool done = terms[i] != 0.0f || truncs[i] != 0.0f;      // ppo.py: dones = terminations | truncations
            ev_len[i] = done ? len : 0;                                  // 0: no event at (t, e)
            if (done) { ev_ret[i] = ret; ret = 0.0; len = 0; ++mine; }
        }
        ep_return[e] = ret;
        ep_len[e] = len;
    }
    // block total -> one atomic
    __shared__ unsigned long long s[4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(finished, s[0] + s[1] + s[2] + s[3]);
}

// Evaluation bookkeeping: the arithmetic of episode_scan_kernel (f32 rewards summed in fp64, length + 1 per step, done = termination
// | truncation, running values carried across chunks), but environment e keeps only its first quota[e] finished episodes, in
// out[slot_offset[e] + k], and counts itself off `remaining` when it reaches its quota.
__global__ void __launch_bounds__(128)
eval_episodes_kernel(const float* __restrict__ rewards, const float* __restrict__ terms, const float* __restrict__ truncs, int T, int N,
                     const int* __restrict__ quota, const int64_t* __restrict__ slot_offset, double* __restrict__ ep_return,
                     int* __restrict__ ep_len, int* __restrict__ recorded, double* __restrict__ out_ret, int* __restrict__ out_len,
                     int* __restrict__ remaining)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    const int q = quota[e];
    const int64_t base = slot_offset[e];
    double ret = ep_return[e];
    int len = ep_len[e];
    int k = recorded[e];
    for (int t = 0; t < T; ++t) {
        const int64_t i = (int64_t)t * N + e;
        ret += (double)rewards[i];
        len += 1;
        if (terms[i] != 0.0f || truncs[i] != 0.0f) {
            if (k < q) {
                out_ret[base + k] = ret;
                out_len[base + k] = len;
                if (++k == q) atomicSub(remaining, 1);
            }
            ret = 0.0;
            len = 0;
        }
    }
    ep_return[e] = ret;
    ep_len[e] = len;
    recorded[e] = k;
}

constexpr int WIN_THREADS = 1024;

__global__ void __launch_bounds__(WIN_THREADS)
episode_window_kernel(const double* __restrict__ ev_ret, const int* __restrict__ ev_len, int T, int N, int window,
                      const unsigned long long* __restrict__ finished, double* __restrict__ out_ret, int* __restrict__ out_len,
                      int* __restrict__ out_n)
{
    __shared__ int s_warp[WIN_THREADS / 32];
    __shared__ int s_collected;
    const unsigned long long total = *finished;
    const int keep = total < (unsigned long long)window ? (int)total : window;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_collected = 0; *out_n = keep; }
    __syncthreads();
    const int chunks = (N + WIN_THREADS - 1) / WIN_THREADS;
    for (int t = T - 1; t >= 0; --t) {
        for (int c = chunks - 1; c >= 0; --c) {
            if (s_collected >= keep) return;                             // uniform: read after the barrier below
            const int e = c * WIN_THREADS + threadIdx.x;
            const int64_t i = (int64_t)t * N + e;
            const int len = e < N ? ev_len[i] : 0;
            const unsigned ballot = __ballot_sync(0xffffffffu, len > 0);
            if (lane == 0) s_warp[warp] = __popc(ballot);
            __syncthreads();
            int after = s_collected;                                     // events that come later in Ticker order
            for (int w = warp + 1; w < WIN_THREADS / 32; ++w) after += s_warp[w];
            after += __popc(ballot >> lane >> 1);                        // higher lanes of this warp
            if (len > 0 && after < keep) {
                out_ret[keep - 1 - after] = ev_ret[i];
                out_len[keep - 1 - after] = len;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int tot = 0;
                for (int w = 0; w < WIN_THREADS / 32; ++w) tot += s_warp[w];
                s_collected += tot;
            }
            __syncthreads();
        }
    }
}

}  // namespace

extern "C" int64_t dppo_episode_stats_workspace_bytes(int T, int N) { return (int64_t)T * N * 12 + 64; }

extern "C" int dppo_episode_stats(dppo_ctx* ctx, const float* rewards, const float* terminations, const float* truncations, int T, int N,
                                  double* ep_return, int32_t* ep_len, int window, double* out_returns, int32_t* out_lengths,
                                  int32_t* out_n, unsigned long long* finished, void* ws, int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (!rewards || !terminations || !truncations || !ep_return || !ep_len || !out_returns || !out_lengths || !out_n || !finished || !ws)
        DPPO_FAIL(ctx, "episode_stats: null argument");
    if (T < 1 || N < 1 || window < 1) DPPO_FAIL(ctx, "episode_stats: bad shape T=%d N=%d window=%d", T, N, window);
    if (ws_bytes < dppo_episode_stats_workspace_bytes(T, N)) DPPO_FAIL(ctx, "episode_stats: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    double* ev_ret = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(ws) + 7) & ~(uintptr_t)7);
    int* ev_len = reinterpret_cast<int*>(ev_ret + (int64_t)T * N);
    if (cudaMemsetAsync(finished, 0, sizeof(unsigned long long), st) != cudaSuccess) DPPO_FAIL(ctx, "episode_stats: memset failed");
    episode_scan_kernel<<<(N + 127) / 128, 128, 0, st>>>(rewards, terminations, truncations, T, N, ep_return, ep_len, ev_ret, ev_len, finished);
    DPPO_CHECK_LAUNCH(ctx, "episode_scan_kernel");
    episode_window_kernel<<<1, WIN_THREADS, 0, st>>>(ev_ret, ev_len, T, N, window, finished, out_returns, out_lengths, out_n);
    DPPO_CHECK_LAUNCH(ctx, "episode_window_kernel");
    return 0;
}

extern "C" int dppo_eval_episodes(dppo_ctx* ctx, const float* rewards, const float* terminations, const float* truncations, int T, int N,
                                  const int32_t* quota, const int64_t* slot_offset, double* ep_return, int32_t* ep_len, int32_t* recorded,
                                  double* out_returns, int32_t* out_lengths, int32_t* remaining, void* stream)
{
    if (!ctx) return 1;
    if (!rewards || !terminations || !truncations || !quota || !slot_offset || !ep_return || !ep_len || !recorded || !out_returns ||
        !out_lengths || !remaining)
        DPPO_FAIL(ctx, "eval_episodes: null argument");
    if (T < 1 || N < 1) DPPO_FAIL(ctx, "eval_episodes: bad shape T=%d N=%d", T, N);
    eval_episodes_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rewards, terminations, truncations, T, N, quota, slot_offset,
                                                                              ep_return, ep_len, recorded, out_returns, out_lengths, remaining);
    DPPO_CHECK_LAUNCH(ctx, "eval_episodes_kernel");
    return 0;
}
