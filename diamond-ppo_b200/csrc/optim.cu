#include <math.h>
// Gradient assembly, clip_grad_norm_ (diamond/ppo.py:284) and Adam (ppo.py:285) over flat buffers.
#include "optim.cuh"

namespace {

// Block = 32 float4 outputs x 8 partial slices.  Thread (x, y) sums partials y, y+8, y+16, ... of output float4 x in a
// fixed order (four interleaved accumulators, four independent 16-byte loads in flight), the eight slice sums are then
// combined in a fixed order through shared memory: deterministic, and segments with many partials (per-CTA head /
// column-sum partials) no longer serialise on a single thread.  Every segment starts on a multiple of 4 floats
// (dppo_mlp_layout) so a float4 never straddles segments; unaligned sources take the scalar path.
constexpr int RED_X = 32, RED_Y = 8;

__global__ void __launch_bounds__(RED_X * RED_Y)
grad_reduce_kernel(GradSegTable tab, float* __restrict__ grads, int64_t total, const float* __restrict__ loss_partials,
                   int loss_nparts, int64_t loss_stride, float vw, float beta, float inv_m, float* __restrict__ losses,
                   double* __restrict__ sumsq_out)
{
    __shared__ float4 s_part[RED_Y][RED_X];
    DPPO_PDL_ENTER();
    const int x = threadIdx.x, y = threadIdx.y;
    const int64_t total4 = (total + 3) / 4;
    double sq = 0.0;                       // this thread's share of the squared gradient norm (y == 0 threads)
    // blocks walk the flat gradient from its END: the segments with the most partials per output (per-CTA head and column-sum
    // partials: 296 / 148 deep, against ~42 for the weight matrices) sit at the end of the layout and would otherwise start last
    // (22 -> 15.5 us)
    const int64_t nchunks = (total4 + RED_X - 1) / RED_X;
    for (int64_t chunk = nchunks - 1 - (int64_t)blockIdx.x; chunk >= 0; chunk -= (int64_t)gridDim.x) {
        const int64_t base = chunk * RED_X;
        const int64_t i = (base + x) * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
            for (int g = 0; g < tab.nseg; ++g) {
                const GradSeg& sg = tab.seg[g];
                if (i >= sg.dst && i < sg.dst + sg.count) {
                    const float* p = sg.src + (i - sg.dst);
                    const bool vec = (i + 4 <= sg.dst + sg.count) && ((sg.stride & 3) == 0) && ((reinterpret_cast<uintptr_t>(p) & 15u) == 0);
                    if (vec) {
                        float4 a[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) a[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        int q = y;
                        for (; q + 3 * RED_Y < sg.nparts; q += 4 * RED_Y) {
                            float4 v[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) v[u] = __ldcs(reinterpret_cast<const float4*>(p + (int64_t)(q + u * RED_Y) * sg.stride));
#pragma unroll
                            for (int u = 0; u < 4; ++u) { a[u].x += v[u].x; a[u].y += v[u].y; a[u].z += v[u].z; a[u].w += v[u].w; }
                        }
                        for (int u = 0; q < sg.nparts; q += RED_Y, ++u) {
                            const float4 v = __ldcs(reinterpret_cast<const float4*>(p + (int64_t)q * sg.stride));
                            a[u].x += v.x; a[u].y += v.y; a[u].z += v.z; a[u].w += v.w;
                        }
                        acc.x = (a[0].x + a[1].x) + (a[2].x + a[3].x);
                        acc.y = (a[0].y + a[1].y) + (a[2].y + a[3].y);
                        acc.z = (a[0].z + a[1].z) + (a[2].z + a[3].z);
                        acc.w = (a[0].w + a[1].w) + (a[2].w + a[3].w);
                    } else {
                        // element by element; an element past this segment's end may start the next one (a tensor whose
                        // gradient comes from two sources, e.g. the halves of b3 on the GEMM-head path, at an odd split)
                        float o[4] = {0.f, 0.f, 0.f, 0.f};
                        for (int e = 0; e < 4 && i + e < total; ++e) {
                            for (int g2 = g; g2 < tab.nseg; ++g2) {
                                const GradSeg& s2 = tab.seg[g2];
                                if (i + e < s2.dst || i + e >= s2.dst + s2.count) continue;
                                const float* p2 = s2.src + (i + e - s2.dst);
                                float s0 = 0.f;
                                for (int q = y; q < s2.nparts; q += RED_Y) s0 += __ldg(p2 + (int64_t)q * s2.stride);
                                o[e] = s0;
                                break;
                            }
                        }
                        acc = make_float4(o[0], o[1], o[2], o[3]);
                    }
                    break;
                }
            }
        }
        s_part[y][x] = acc;
        __syncthreads();
        if (y == 0 && i < total) {
            float4 r = s_part[0][x];
#pragma unroll
            for (int k = 1; k < RED_Y; ++k) { const float4 v = s_part[k][x]; r.x += v.x; r.y += v.y; r.z += v.z; r.w += v.w; }
            if (i + 4 <= total) {
                *reinterpret_cast<float4*>(grads + i) = r;
                sq += (double)r.x * r.x + (double)r.y * r.y + (double)r.z * r.z + (double)r.w * r.w;
            } else {
                const float rr[4] = {r.x, r.y, r.z, r.w};
                for (int e = 0; i + e < total; ++e) { grads[i + e] = rr[e]; sq += (double)rr[e] * rr[e]; }
            }
        }
        __syncthreads();
    }
    if (sumsq_out != nullptr && y == 0) {          // y == 0 is exactly warp 0 of the block
        sq = warp_sum_d(sq);
        if (x == 0) sumsq_out[blockIdx.x] = sq;
    }
    if (blockIdx.x == 0 && losses != nullptr) {
        // warp w < 3 sums loss term w: lane-strided partial sums in a fixed order, then a fixed shuffle tree
        __shared__ float l[3];
        if (y < 3) {
            float s = 0.f;
            for (int p = x; p < loss_nparts; p += RED_X) s += __ldg(loss_partials + (int64_t)p * loss_stride + y);
            s = warp_sum(s);
            if (x == 0) l[y] = s;
        }
        __syncthreads();
        if (x == 0 && y == 0) {
            const float pol = l[0] * inv_m, val = 0.5f * l[1] * inv_m, ent = l[2] * inv_m;    // ppo.py:270-274
            losses[0] = pol; losses[1] = val; losses[2] = ent;
            losses[3] = pol + vw * val + -beta * ent;                                          // ppo.py:276-280
        }
    }
}

constexpr int SUMSQ_THREADS = 256;

__global__ void __launch_bounds__(SUMSQ_THREADS)
sumsq_kernel(const float* __restrict__ g, int64_t n, double* __restrict__ partials)
{
    __shared__ double red[SUMSQ_THREADS / 32];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float x = g[i];
        s += (double)x * (double)x;
    }
    s = warp_sum_d(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = threadIdx.x < SUMSQ_THREADS / 32 ? red[threadIdx.x] : 0.0;
        s = warp_sum_d(s);
        if (threadIdx.x == 0) partials[blockIdx.x] = s;
    }
}

// torch/nn/utils/clip_grad.py:165-182 then torch/optim/adam.py single-tensor path (:457,:476,:531-547).
__global__ void __launch_bounds__(256)
clip_adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                 const double* __restrict__ norm_partials, int nparts, float max_norm, float w1, float beta2, float w2,
                 float bc2_sqrt, float eps, float neg_step_size, float* __restrict__ grad_norm_out,
                 const float* __restrict__ step_consts)
{
    __shared__ float s_coef;
    DPPO_PDL_ENTER();
    // device-resident step constants (CUDA-graph replay of the update loop): [0] = sqrt(1 - beta2^t), [1] = -lr / (1 - beta1^t)
    if (step_consts != nullptr) { bc2_sqrt = __ldg(step_consts); neg_step_size = __ldg(step_consts + 1); }
    // every block needs the global norm: all 256 threads share the nparts fp64 partials (one warp alone spent ~4 us of this
    // 10 us kernel on 53 dependent-latency loads per lane); fixed order: strided per thread, shuffle tree, then warp 0..7
    __shared__ double s_norm[8];
    {
        double s = 0.0;
        for (int i = threadIdx.x; i < nparts; i += 256) s += norm_partials[i];
        s = warp_sum_d(s);
        if ((threadIdx.x & 31) == 0) s_norm[threadIdx.x >> 5] = s;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        if (threadIdx.x == 0) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) s += s_norm[w];
            const float total = (float)sqrt(s);
            float coef = max_norm / (total + 1e-6f);
            s_coef = coef > 1.0f ? 1.0f : coef;
            if (blockIdx.x == 0 && grad_norm_out) *grad_norm_out = total;
        }
    }
    __syncthreads();
    const float coef = s_coef;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gi = __fmul_rn(g[i], coef);                                   // grads are always scaled
        float mi = m[i], vi = v[i];
        mi = fmaf(w1, gi - mi, mi);                                               // exp_avg.lerp_(grad, 1-beta1)
        vi = __fadd_rn(__fmul_rn(vi, beta2), __fmul_rn(__fmul_rn(w2, gi), gi));   // mul_(beta2).addcmul_(g, g, 1-beta2)
        const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
        p[i] = __fadd_rn(p[i], __fmul_rn(neg_step_size, __fdiv_rn(mi, denom)));   // addcdiv_(m, denom, -step_size)
        g[i] = gi; m[i] = mi; v[i] = vi;
    }
}

__global__ void gather_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, float* __restrict__ dst,
                                   int64_t rows, int row_floats, const int* __restrict__ rows_dev)
{
    if (rows_dev != nullptr && *rows_dev < rows) rows = *rows_dev;
    const int64_t total = rows * row_floats;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / row_floats;
        const int c = (int)(i - r * row_floats);
        dst[i] = __ldg(src + (int64_t)(idx[r] < 0 ? 0 : idx[r]) * row_floats + c);
    }
}

// row_floats % 4 == 0 and 16-byte aligned bases: one float4 per thread, a row is read by row_floats/4 consecutive threads
__global__ void gather_rows4_kernel(const float4* __restrict__ src, const int32_t* __restrict__ idx, float4* __restrict__ dst,
                                    int64_t rows, int row_vec, const int* __restrict__ rows_dev)
{
    if (rows_dev != nullptr && *rows_dev < rows) rows = *rows_dev;
    const int64_t total = rows * row_vec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / row_vec;
        const int c = (int)(i - r * row_vec);
        const int32_t s = __ldg(idx + r);
        dst[i] = __ldg(src + (int64_t)(s < 0 ? 0 : s) * row_vec + c);
    }
}

// 16 independent 3-register FFMA chains per thread (acc = x*y + acc, the form a GEMM inner loop issues):
// the FP32 FMA-pipe ceiling of this GPU at its current clocks.  iters FMAs per thread (multiple of 16).
__global__ void __launch_bounds__(256)
fma_peak_kernel(float* __restrict__ sink, int64_t iters)
{
    float x[4], y[4], acc[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        x[i] = sink[(threadIdx.x + i) & 63] * 1e-6f;
        y[i] = sink[(threadIdx.x + 4 + i) & 63] * 1e-6f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    for (int64_t it = 0; it < iters; it += 16) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i * 4 + j] = fmaf(x[i], y[j], acc[i * 4 + j]);
    }
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) r += acc[i];
    if (r == 123.456f) sink[64] = r;
}

}  // namespace

int grad_reduce_blocks(dppo_ctx* ctx, int64_t total)
{
    int64_t want = ((total + 3) / 4 + RED_X - 1) / RED_X;
    int blocks = (int)(want < 16 * (int64_t)ctx->sm_count ? want : 16 * (int64_t)ctx->sm_count);
    return blocks < 1 ? 1 : blocks;
}

int launch_grad_reduce(dppo_ctx* ctx, const GradSegTable& tab, float* grads, int64_t total, const float* loss_partials,
                       int loss_nparts, int64_t loss_stride, float vw, float beta, float inv_m, float* losses, double* sumsq_out,
                       cudaStream_t st)
{
    if ((reinterpret_cast<uintptr_t>(grads) & 15u) != 0) DPPO_FAIL(ctx, "grad_reduce: gradient buffer must be 16-byte aligned");
    const int blocks = grad_reduce_blocks(ctx, total);
    dppo_launch_pdl(ctx, grad_reduce_kernel, dim3(blocks), dim3(RED_X, RED_Y), 0, st, tab, grads, total, loss_partials, loss_nparts, loss_stride,
                    vw, beta, inv_m, losses, sumsq_out);
    DPPO_CHECK_LAUNCH(ctx, "grad_reduce_kernel");
    return 0;
}

int launch_clip_adam(dppo_ctx* ctx, float* params, float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const double* partials,
                     int nparts, const dppo_hyper* h, float* grad_norm_out, cudaStream_t st)
{
    // bias corrections in double on the host exactly as torch does with python floats (adam.py:531-547)
    const double bc1 = 1.0 - pow(h->beta1, (double)h->step);
    const double bc2 = 1.0 - pow(h->beta2, (double)h->step);
    const double step_size = h->lr / bc1;
    const double bc2_sqrt = sqrt(bc2);
    int blocks = (int)((n + 255) / 256);
    if (blocks > 2 * ctx->sm_count) blocks = 2 * ctx->sm_count;
    dppo_launch_pdl(ctx, clip_adam_kernel, dim3(blocks), dim3(256), 0, st, params, grads, exp_avg, exp_avg_sq, n, partials, nparts,
                    h->grad_norm_clip, (float)(1.0 - h->beta1), (float)h->beta2, (float)(1.0 - h->beta2), (float)bc2_sqrt, h->adam_eps,
                    (float)(-step_size), grad_norm_out, h->step_consts);
    DPPO_CHECK_LAUNCH(ctx, "clip_adam_kernel");
    return 0;
}

static int sumsq_blocks(int64_t n)
{
    int64_t b = (n + SUMSQ_THREADS * 4 - 1) / (SUMSQ_THREADS * 4);
    if (b > 256) b = 256;
    if (b < 1) b = 1;
    return (int)b;
}

extern "C" int64_t dppo_clip_adam_workspace_bytes(int64_t n) { return (int64_t)sumsq_blocks(n) * (int64_t)sizeof(double); }

extern "C" int64_t dppo_grad_sumsq_bytes(dppo_ctx* ctx, int64_t n) { return ctx ? (int64_t)grad_reduce_blocks(ctx, n) * (int64_t)sizeof(double) : 0; }

extern "C" int dppo_clip_adam_step(dppo_ctx* ctx, float* params, float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                   const dppo_hyper* h, float* grad_norm_out, void* ws, int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (n <= 0) DPPO_FAIL(ctx, "clip_adam: empty parameter buffer");
    if (h->step < 1) DPPO_FAIL(ctx, "clip_adam: step must be >= 1 (got %lld)", (long long)h->step);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->grad_sumsq != nullptr)          // dppo_mlp_grad_minibatch already left the partial sums of squares there
        return launch_clip_adam(ctx, params, grads, exp_avg, exp_avg_sq, n, h->grad_sumsq, grad_reduce_blocks(ctx, n), h, grad_norm_out, st);
    const int nb = sumsq_blocks(n);
    if (ws_bytes < (int64_t)nb * (int64_t)sizeof(double)) DPPO_FAIL(ctx, "clip_adam: workspace too small");
    if ((reinterpret_cast<uintptr_t>(ws) & 7u) != 0) DPPO_FAIL(ctx, "clip_adam: workspace must be 8-byte aligned");
    double* partials = (double*)ws;
    sumsq_kernel<<<nb, SUMSQ_THREADS, 0, st>>>(grads, n, partials);
    DPPO_CHECK_LAUNCH(ctx, "sumsq_kernel");
    return launch_clip_adam(ctx, params, grads, exp_avg, exp_avg_sq, n, partials, nb, h, grad_norm_out, st);
}

extern "C" int dppo_gather_rows_f32(dppo_ctx* ctx, const float* src, const int32_t* idx, float* dst, int64_t rows,
                                    int row_floats, void* stream)
{
    if (!ctx) return 1;
    if (rows <= 0 || row_floats <= 0) return 0;
    if (row_floats % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        const int64_t total4 = rows * (row_floats / 4);
        int blocks4 = (int)((total4 + 255) / 256);
        if (blocks4 > 16 * ctx->sm_count) blocks4 = 16 * ctx->sm_count;
        gather_rows4_kernel<<<blocks4, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(src), idx,
                                                                      reinterpret_cast<float4*>(dst), rows, row_floats / 4, ctx->rows_dev);
        DPPO_CHECK_LAUNCH(ctx, "gather_rows4_kernel");
        return 0;
    }
    const int64_t total = rows * row_floats;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 8 * ctx->sm_count) blocks = 8 * ctx->sm_count;
    gather_rows_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(src, idx, dst, rows, row_floats, ctx->rows_dev);
    DPPO_CHECK_LAUNCH(ctx, "gather_rows_kernel");
    return 0;
}

extern "C" int dppo_fma_peak_kernel(dppo_ctx* ctx, float* sink, int64_t iters, int* blocks_out, int* threads_out, void* stream)
{
    if (!ctx) return 1;
    const int blocks = ctx->sm_count * 8, threads = 256;
    fma_peak_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(sink, iters);
    DPPO_CHECK_LAUNCH(ctx, "fma_peak_kernel");
    if (blocks_out) *blocks_out = blocks;
    if (threads_out) *threads_out = threads;
    return 0;
}
