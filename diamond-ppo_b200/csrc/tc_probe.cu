// Measurement helper: issue rate of tcgen05.mma with shared-memory operands on this GPU (the roofline denominator of the
// 3xTF32 GEMMs).  Every CTA issues `iters` back-to-back MMAs on fixed operand tiles and reports the SM cycles they took.
#include <cuda.h>

#include "tc_common.cuh"

using namespace tc;

namespace {

__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate, int two)
{
    if (two)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// fmt: 0 tf32 (K = 8), 1 bf16, 2 fp16 (K = 16; kind::f16 with A/B format 1 or 0); n = MMA N
template <int PAIR>
__global__ void __launch_bounds__(128, 1)
mma_probe_kernel(int fmt, int n, int iters, long long* __restrict__ out)
{
    extern __shared__ unsigned char dyn_raw[];
    __shared__ __align__(8) uint64_t done;
    __shared__ uint32_t s_tmem;
    unsigned char* dyn = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(dyn_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < 48 * 1024 / 4; i += blockDim.x) reinterpret_cast<float*>(dyn)[i] = 0.f;
    if (tid == 0) { mbar_init(&done, 1); fence_mbar_init(); }
    if (warp == 0) { if (PAIR) tmem_alloc2(&s_tmem, 512); else tmem_alloc(&s_tmem, 512); }
    fence_proxy_async();
    fence_before();
    if (PAIR) cluster_sync(); else __syncthreads();
    fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0;
    if (tid == 0 && rank == 0) {
        const uint32_t a = smem_u32(dyn), b = a + 16 * 1024;
        uint32_t idesc = idesc_tf32(PAIR ? 256 : 128, n, 0, 0);
        if (fmt) idesc = (idesc & ~((7u << 7) | (7u << 10))) | (fmt == 1 ? (1u << 7) | (1u << 10) : 0u);
        const uint64_t da = desc_k_sw64(a), db = desc_k_sw64(b);
        const long long t0 = clock64();
        for (int i = 0; i < iters; ++i) {
            if (fmt) umma_f16(tmem, da, db, idesc, 1u, PAIR);
            else if (PAIR) umma_tf32_2cta(tmem, da, db, idesc, 1u);
            else umma_tf32(tmem, da, db, idesc, 1u);
        }
        if (PAIR) umma_commit_2cta(&done, 1); else umma_commit(&done);
        mbar_wait(&done, 0);
        out[blockIdx.x] = clock64() - t0;
    }
    fence_before();
    if (PAIR) cluster_sync(); else __syncthreads();
    if (warp == 0) { fence_after(); if (PAIR) tmem_dealloc2(tmem, 512); else tmem_dealloc(tmem, 512); }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
mma_probe_pair(int fmt, int n, int iters, long long* __restrict__ out)
{
    extern __shared__ unsigned char dyn_raw[];
    __shared__ __align__(8) uint64_t done;
    __shared__ uint32_t s_tmem;
    unsigned char* dyn = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(dyn_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < 48 * 1024 / 4; i += blockDim.x) reinterpret_cast<float*>(dyn)[i] = 0.f;
    if (tid == 0) { mbar_init(&done, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc2(&s_tmem, 512);
    fence_proxy_async();
    fence_before();
    cluster_sync();
    fence_after();
    const uint32_t tmem = s_tmem;
    if (tid == 0 && cluster_ctarank() == 0) {
        const uint32_t a = smem_u32(dyn), b = a + 16 * 1024;
        uint32_t idesc = idesc_tf32(256, n, 0, 0);
        if (fmt) idesc = (idesc & ~((7u << 7) | (7u << 10))) | (fmt == 1 ? (1u << 7) | (1u << 10) : 0u);
        const uint64_t da = desc_k_sw64(a), db = desc_k_sw64(b);
        const long long t0 = clock64();
        for (int i = 0; i < iters; ++i) {
            if (fmt) umma_f16(tmem, da, db, idesc, 1u, 1);
            else umma_tf32_2cta(tmem, da, db, idesc, 1u);
        }
        umma_commit_2cta(&done, 1);
        mbar_wait(&done, 0);
        out[blockIdx.x] = clock64() - t0;
    }
    fence_before();
    cluster_sync();
    if (warp == 0) { fence_after(); tmem_dealloc2(tmem, 512); }
}
}  // namespace

// out: int64 [grid] SM cycles for `iters` MMAs (entries of non-leader CTAs of a pair stay untouched)
extern "C" int dppo_tc_mma_probe(dppo_ctx* ctx, int pair, int fmt, int n, int iters, long long* out, int* grid_out, void* stream)
{
    if (!ctx) return 1;
    if (n % 16 != 0 || n < 16 || n > 256 || iters < 1 || fmt < 0 || fmt > 2) DPPO_FAIL(ctx, "tc_mma_probe: bad arguments");
    const int grid = ctx->sm_count / 2 * 2;
    const size_t smem = 49 * 1024 + 1024;
    cudaStream_t st = (cudaStream_t)stream;
    if (pair) {
        cudaFuncSetAttribute(mma_probe_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        mma_probe_pair<<<grid, 128, smem, st>>>(fmt, n, iters, out);
    } else {
        cudaFuncSetAttribute(mma_probe_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        mma_probe_kernel<0><<<grid, 128, smem, st>>>(fmt, n, iters, out);
    }
    DPPO_CHECK_LAUNCH(ctx, "mma_probe_kernel");
    if (grid_out) *grid_out = grid;
    return 0;
}
