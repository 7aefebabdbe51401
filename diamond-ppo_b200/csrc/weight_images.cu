// Weight images of the 3xTF32 tcgen05 GEMMs (gemm_tc3.cu) for the wide (H >= 128) actor-critic MLP.
//
// fp32 parity needs more than one TF32 pass (single-pass TF32 misses the 1e-4 parameter bar by 70x, SURVEY.md
// 0.6), so every fp32 weight x is split into hi = x rounded to the nearest TF32 number (10 mantissa bits)
// and lo = x - hi (exact in fp32; the tensor core reads its top 19 bits); the GEMMs issue three MMAs per k-step
// into the same fp32 TMEM accumulator:   D += A_hi*B_lo ; D += A_lo*B_hi ; D += A_hi*B_hi.
// The images are laid out in the canonical K-major SWIZZLE_64B shared-memory layout (16 fp32 of K per 64-byte row,
// 8-row atoms of 512 B) so that a GEMM CTA fetches a k-chunk of its weight rows with one bulk async copy.
// One launch per optimiser step rebuilds every image (and gathers the minibatch observations, ppo.py:261).
//
// fp16 images (PrepJob::f16, forward images of the layers whose input is a tanh output): the same three-MMA scheme on fp16
// pairs of W' = W * s_n, hi = fp16_rn(W'), lo = fp16_rn(W' - hi) (22 significant bits).  s_n = 2^e is one power of two per
// output row n with max |W'| in [2^14, 2^15), so that neither half leaves fp16's normal range; the image ends with the column
// factors 2^-14 / s_n the GEMM epilogue applies (dppo_tc_f16_factor_offset).  Layout: K-major SWIZZLE_32B (16 fp16 of K per
// 32-byte row, 8-row atoms of 256 B), [hi | lo] per N tile and 16-wide k chunk as for TF32.
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "gemm_tc.cuh"

namespace {

constexpr int KC = 16;                     // k elements per chunk (one SWIZZLE_64B atom width)

// byte offset of element (row, kk) inside a K-major SWIZZLE_64B image (rows x 16 fp32)
__host__ __device__ __forceinline__ int sw64_offset(int row, int kk)
{
    return (row >> 3) * 512 + (row & 7) * 64 + ((((kk >> 2) ^ ((row & 7) >> 1)) & 3) << 4) + ((kk & 3) << 2);
}

// byte offset of fp16 element (row, kk) inside a K-major SWIZZLE_32B image (rows x 16 fp16)
__device__ __forceinline__ int sw32_offset(int row, int kk)
{
    return row * 32 + ((((kk >> 3) ^ (row >> 2)) & 1) << 4) + ((kk & 7) << 1);
}

__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo)
{
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);   // round to nearest TF32 (|lo| <= 2^-12 |x|)
    lo = x - hi;
}

// ---------------------------------------------------------------------------------------------
// Weight images.  For one Linear weight W [rows_w, cols_w] (row-major) used as the B operand
//   transpose == 0 : B[n, k] = W[n, k]      (forward:  N = rows_w, K = cols_w)
//   transpose == 1 : B[n, k] = W[k, n]      (dgrad:    N = cols_w, K = rows_w)
// Output: for every N tile (n_tile rows) and every 16-wide k chunk, [hi image | lo image], each
// n_tile x 64 B in the SWIZZLE_64B layout, so that the GEMM copies a chunk with one bulk copy.
// ---------------------------------------------------------------------------------------------
__global__ void prep_weights_kernel(const float* __restrict__ W, int rows_w, int cols_w, int transpose, int n_tile,
                                    unsigned char* __restrict__ img)
{
    const int N = transpose ? cols_w : rows_w;
    const int K = transpose ? rows_w : cols_w;
    const int64_t total = (int64_t)N * K;
    const int chunks = K / KC;
    const int img_bytes = n_tile * KC * 4;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        int n, k;
        if (transpose) { k = (int)(e / cols_w); n = (int)(e % cols_w); }      // coalesced read of W[k, n]
        else { n = (int)(e / cols_w); k = (int)(e % cols_w); }
        const float x = W[e];
        float hi, lo;
        split_tf32(x, hi, lo);
        const int tile = n / n_tile, row = n % n_tile, chunk = k / KC, kk = k % KC;
        unsigned char* base = img + ((int64_t)(tile * chunks + chunk) * 2) * img_bytes;
        const int off = sw64_offset(row, kk);
        *reinterpret_cast<float*>(base + off) = hi;
        *reinterpret_cast<float*>(base + img_bytes + off) = lo;
    }
}

// All weight images of one optimiser step in a single launch: blockIdx.y selects the job.
__global__ void prep_weights_multi_kernel(PrepJobs jobs)
{
    DPPO_PDL_ENTER();
    if ((int)blockIdx.y >= jobs.n) {
        // the minibatch observation gather (ppo.py:261 observations[mb]) shares the launch: it is independent of the weights.
        // It takes the remaining gridDim.y - jobs.n slices of the grid (index -> row is a dependent pair of DRAM latencies, so the
        // work is spread over more threads instead of more iterations per thread); two items in flight per thread
        const GatherJob& g = jobs.gather;
        const int64_t total = g.rows * g.row_vec;
        const int64_t nthreads = (int64_t)(gridDim.y - jobs.n) * gridDim.x * blockDim.x;
        const int64_t t0 = ((int64_t)(blockIdx.y - jobs.n) * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        for (int64_t i = t0; i < total; i += 2 * nthreads) {
            const int64_t i2 = i + nthreads;
            const int64_t r = i / g.row_vec, r2 = i2 / g.row_vec;
            int32_t s1 = __ldg(g.idx + r), s2 = i2 < total ? __ldg(g.idx + r2) : 0;
            s1 = s1 < 0 ? 0 : s1; s2 = s2 < 0 ? 0 : s2;            // padding rows (idx < 0) read row 0: finite values, masked in the head kernel
            const float4 v1 = __ldg(g.src + (int64_t)s1 * g.row_vec + (int)(i - r * g.row_vec));
            if (i2 < total) {
                const float4 v2 = __ldg(g.src + (int64_t)s2 * g.row_vec + (int)(i2 - r2 * g.row_vec));
                g.dst[i2] = v2;
            }
            g.dst[i] = v1;
        }
        return;
    }
    const PrepJob& j = jobs.job[blockIdx.y];
    const int N = j.transpose ? j.cols_w : j.rows_w;
    const int K = j.transpose ? j.rows_w : j.cols_w;
    const int64_t total = (int64_t)N * K;
    const int chunks = K / KC;
    if (j.f16) {
        // one warp per weight row n.  The row's largest magnitude is an integer max over the magnitude bits, so Inf and NaN rank
        // above every finite value: such a row keeps s_n = 1 and its Inf / NaN reach the products (lo = Inf - Inf is NaN).  e is
        // clamped so that s_n and the column factor stay normal fp32 numbers (rows whose largest |w| is below 2^-98 keep
        // 2^112 and lose relative, not absolute, accuracy).
        const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
        const int img_bytes = j.n_tile * KC * 2;
        float* factor = reinterpret_cast<float*>(j.img + dppo_tc_f16_factor_offset(N, K));
        for (int n = blockIdx.x * warps + (threadIdx.x >> 5); n < N; n += gridDim.x * warps) {
            const float* w = j.W + (int64_t)n * K;
            unsigned mx = 0;
            for (int k = lane; k < K; k += 32) mx = max(mx, __float_as_uint(w[k]) & 0x7FFFFFFFu);
            mx = __reduce_max_sync(0xffffffffu, mx);
            int e = 0;
            if (mx != 0 && mx < 0x7F800000u) e = min(112, 14 - ((int)(mx >> 23) - 127));
            const float sc = __int_as_float((127 + e) << 23);
            if (lane == 0) factor[n] = __int_as_float((127 - DPPO_F16_A_EXP - e) << 23);
            const int tile = n / j.n_tile, row = n % j.n_tile;
            for (int k = lane; k < K; k += 32) {
                const float x = w[k] * sc;
                const __half hi = __float2half_rn(x);
                const __half lo = __float2half_rn(x - __half2float(hi));
                unsigned char* base = j.img + ((int64_t)(tile * chunks + k / KC) * 2) * img_bytes;
                const int off = sw32_offset(row, k % KC);
                *reinterpret_cast<__half*>(base + off) = hi;
                *reinterpret_cast<__half*>(base + img_bytes + off) = lo;
            }
        }
        return;
    }
    const int img_bytes = j.n_tile * KC * 4;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        int n, k;
        if (j.transpose) { k = (int)(e / j.cols_w); n = (int)(e % j.cols_w); }
        else { n = (int)(e / j.cols_w); k = (int)(e % j.cols_w); }
        const float x = j.W[e];
        float hi, lo;
        split_tf32(x, hi, lo);
        const int tile = n / j.n_tile, row = n % j.n_tile, chunk = k / KC, kk = k % KC;
        unsigned char* base = j.img + ((int64_t)(tile * chunks + chunk) * 2) * img_bytes;
        const int off = sw64_offset(row, kk);
        *reinterpret_cast<float*>(base + off) = hi;
        *reinterpret_cast<float*>(base + img_bytes + off) = lo;
    }
}

}  // namespace

int dppo_tc_n_tile(int N) { return N % 256 == 0 ? 256 : 128; }

// the TF32 images; the fp16 ones (N K 4 bytes + N column factors) fit the same space
int64_t dppo_tc_image_bytes(int N, int K) { return (int64_t)N * K * 4 * 2; }

int dppo_tc_prep_weights(dppo_ctx* ctx, const float* W, int rows_w, int cols_w, int transpose, unsigned char* img, cudaStream_t st)
{
    const int N = transpose ? cols_w : rows_w;
    const int64_t total = (int64_t)rows_w * cols_w;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 4 * ctx->sm_count) blocks = 4 * ctx->sm_count;
    prep_weights_kernel<<<blocks, 256, 0, st>>>(W, rows_w, cols_w, transpose, dppo_tc_n_tile(N), img);
    DPPO_CHECK_LAUNCH(ctx, "prep_weights_kernel");
    return 0;
}

int dppo_tc_prep_weights_multi(dppo_ctx* ctx, PrepJobs jobs, cudaStream_t st)
{
    const bool with_gather = jobs.gather.rows > 0 && jobs.gather.dst != nullptr;
    if (jobs.n < 1 && !with_gather) return 0;
    int64_t most = with_gather ? jobs.gather.rows * jobs.gather.row_vec / 8 : 0;
    for (int i = 0; i < jobs.n; ++i) {
        if (jobs.job[i].f16 && jobs.job[i].transpose) DPPO_FAIL(ctx, "prep_weights_multi: fp16 images are built for forward (untransposed) weights only");
        const int64_t t = (int64_t)jobs.job[i].rows_w * jobs.job[i].cols_w;
        jobs.job[i].n_tile = dppo_tc_n_tile(jobs.job[i].transpose ? jobs.job[i].cols_w : jobs.job[i].rows_w);
        if (t > most) most = t;
    }
    int blocks = (int)((most + 255) / 256);
    if (blocks > 4 * ctx->sm_count) blocks = 4 * ctx->sm_count;
    if (blocks < 1) blocks = 1;
    dppo_launch_pdl(ctx, prep_weights_multi_kernel, dim3(blocks, jobs.n + (with_gather ? 4 : 0)), dim3(256), 0, st, jobs);
    DPPO_CHECK_LAUNCH(ctx, "prep_weights_multi_kernel");
    return 0;
}
