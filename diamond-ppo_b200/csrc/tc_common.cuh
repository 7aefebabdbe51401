// Device-side building blocks of the warp-specialised 3xTF32 tcgen05 kernels (gemm_tc2.cu, wgrad_tc.cu):
// mbarrier / TMA / bulk-copy / tcgen05 PTX wrappers and the shared-memory + instruction descriptors.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "TC_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TC_DONE_%=;\n\t"
        "bra TC_WAIT_%=;\n\t"
        "TC_DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// ---- async copies -----------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, int x, int y, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
// TMA loads / prefetches with an L2 eviction-priority hint (policy: common.cuh l2_policy_evict_first)
__device__ __forceinline__ void tma_load_2d_hint(void* dst, const CUtensorMap* tm, int x, int y, uint64_t* bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_prefetch_2d_hint(const CUtensorMap* tm, int x, int y, uint64_t policy)
{
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.L2::cache_hint [%0, {%1, %2}], %3;"
                 ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "l"(policy) : "memory");
}
// HBM -> L2 prefetch of a box (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* tm, int x, int y)
{
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t saddr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, const float4& v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// shared -> global store of a box (bulk async-group completion); rows/cols outside the tensor are clipped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, int x, int y, uint32_t saddr)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(saddr) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 ----------------------------------------------------------------------------------
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols)       // one full warp
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)     // the same warp
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

// ---- CTA pairs (cta_group::2) ------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync()          // all threads of all CTAs of the cluster
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    // default semantics (release at CTA scope), as CUTLASS's umma_arrive_2x1SM_sm0: the data the leader consumes after this
    // arrival is read by the tensor core from shared memory (async proxy, ordered by fence.proxy.async), never from a cache
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait that also acquires writes released at cluster scope (arrivals from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "TCC_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TCC_DONE_%=;\n\t"
        "bra TCC_WAIT_%=;\n\t"
        "TCC_DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t cols)      // the same warp of both CTAs of the pair
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// one MMA over the CTA pair: D[256 x N] (128 TMEM lanes in each CTA) += A[256 x 8] * B[N x 8]^T, every CTA supplying its
// 128 rows of A and its N/2 rows of B from the same shared-memory offsets.  Issued by one thread of the leader CTA.
__device__ __forceinline__ void umma_tf32_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// the same with 16-bit operands (kind::f16, K = 16, fp32 accumulator)
__device__ __forceinline__ void umma_f16_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the mbarrier at this shared-memory offset in every CTA of `mask` once all MMAs issued so far are complete
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t mask)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}

// Shared-memory matrix descriptors (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14), leading byte
// offset >> 4 in [16,30), stride byte offset >> 4 in [32,46), version 1 (sm_100) in [46,48), layout in [61,64).
// K-major SWIZZLE_64B: rows of 16 fp32 (64 B), 8-row atoms of 512 B; LBO unused (1), SBO = 512 B.
__device__ __forceinline__ uint64_t desc_k_sw64(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// K-major SWIZZLE_32B (layout type 6): rows of 16 fp16 (32 B), 8-row atoms of 256 B; SBO = 256 B.
__device__ __forceinline__ uint64_t desc_k_sw32(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46) | (6ull << 61);
}
// MN-major fp32/tf32 operands have exactly one legal swizzled layout, SWIZZLE_128B_BASE32B (layout type 1; what a
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B box delivers): groups of 32 fp32 along M/N (128 B rows), one row per k, 32-byte
// chunks XOR-swizzled with (row % 4); 4 rows = one 512 B atom.  LBO = bytes between consecutive 32-wide M/N groups,
// SBO = bytes between consecutive 4-row k atoms (512 when the rows of a group are contiguous).
__device__ __forceinline__ uint64_t desc_mn_sw128_32b(uint32_t saddr, uint32_t lbo_bytes)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) |
           (1ull << 61);
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D = f32 (bit 4), A = B = tf32 (2 at bits 7, 10),
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N >> 3 at bit 17, M >> 4 at bit 24.
__device__ __forceinline__ uint32_t idesc_tf32(int m, int n, int a_mn, int b_mn)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}
// kind::f16 instruction descriptor: D = f32, A = B = fp16 (format 0), both K-major
__device__ __forceinline__ uint32_t idesc_f16(int m, int n)
{
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives (count 1) on the mbarrier when every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread l of the warp receives row (lane base + l), columns c..c+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// The same load split in two so that independent work can overlap the TMEM read: issue, then wait (the wait names the
// destination registers as in/out operands so that the compiler cannot move their uses above it).
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// hi = x rounded to the nearest TF32 number (10 mantissa bits), lo = x - hi (exact; |lo| <= 2^-12 |x|)
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo)
{
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
    lo = x - hi;
}
// splits a float4 in place (hi) and returns lo
__device__ __forceinline__ float4 split_tf32x4(float4& x)
{
    float4 lo;
    split_tf32(x.x, x.x, lo.x); split_tf32(x.y, x.y, lo.y); split_tf32(x.z, x.z, lo.z); split_tf32(x.w, x.w, lo.w);
    return lo;
}

// The raw fp32 operand as its own hi image: kind::tf32 reads the upper 19 bits of each fp32 word (the 13 low mantissa bits are
// ignored), i.e. hi = trunc_tf32(x) costs no shared-memory store.  lo = rn_tf32(x - trunc(x)); the difference is exact in fp32
// (13 significant bits) and |lo| < 2^-10 |x|.  Halves the shared-memory write traffic of the split warps (the weight-gradient
// kernel, which splits BOTH operands, is shared-memory-bandwidth bound: 64 KB read + 128 KB written + 64 KB TMA + operand
// fetch per chunk).
__device__ __forceinline__ float lo_of_trunc(float x)
{
    const float r = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
    return __uint_as_float((__float_as_uint(r) + 0x1000u) & 0xFFFFE000u);
}
__device__ __forceinline__ float4 lo_of_trunc_x4(const float4& x)
{
    return make_float4(lo_of_trunc(x.x), lo_of_trunc(x.y), lo_of_trunc(x.z), lo_of_trunc(x.w));
}

// fp16 hi/lo pair of 8 scaled values x' = x * scale (a power of two): hi = fp16_rn(x'), lo = fp16_rn(x' - hi), x' - hi exact in
// fp32.  Each is one 16-byte row segment of a K-major fp16 image (element order = k order).
__device__ __forceinline__ void split_f16x8(const float4& a, const float4& b, float scale, uint4& hi, uint4& lo)
{
    const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float x0 = x[2 * i] * scale, x1 = x[2 * i + 1] * scale;
        uint32_t p;
        asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(p) : "f"(x1), "f"(x0));           // upper half <- x1, lower half <- x0
        h[i] = p;
        const float r0 = x0 - __half2float(__ushort_as_half((unsigned short)(p & 0xFFFFu)));
        const float r1 = x1 - __half2float(__ushort_as_half((unsigned short)(p >> 16)));
        asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(l[i]) : "f"(r1), "f"(r0));
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}
__device__ __forceinline__ void sts128u(uint32_t saddr, const uint4& v)
{
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

}  // namespace tc

// ---- host: tensor maps (gemm_tc2.cu) -------------------------------------------------------------
// 2-D map over a row-major fp32 matrix [rows, cols] with row pitch ld floats; box = box_cols x box_rows;
// swizzle: 0 none, 1 = 32B, 2 = 64B, 3 = 128B, 4 = 128B with 32B atoms.  Returns false if the driver entry point is missing or the
// encode fails (unaligned base / pitch).
bool dppo_make_tensor_map_2d(CUtensorMap* out, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                             int swizzle);

// tanh for the GEMM epilogues: odd 13th-degree over even 6th-degree rational minimax (the coefficients Eigen publishes for its float
// tanh), evaluated as plain FFMA chains with immediate operands + one MUFU.RCP.  |error| <= 2.9e-7 absolute (< 5 ulp, checked over
// [-10, 10] and around 0 in tests/test_tanh_approx.py); libm's tanhf costs two MUFU operations and two divergent code paths
// per element, which made the forward epilogues as expensive as their MMAs (DESIGN section 4).
__device__ __forceinline__ float tanh_rational(float x)
{
    x = fminf(fmaxf(x, -7.90531110763549805f), 7.90531110763549805f);
    const float x2 = x * x;
    float p = fmaf(x2, -2.76076847742355e-16f, 2.00018790482477e-13f);
    p = fmaf(x2, p, -8.60467152213735e-11f);
    p = fmaf(x2, p, 5.12229709037114e-08f);
    p = fmaf(x2, p, 1.48572235717979e-05f);
    p = fmaf(x2, p, 6.37261928875436e-04f);
    p = fmaf(x2, p, 4.89352455891786e-03f);
    float q = fmaf(x2, 1.19825839466702e-06f, 1.18534705686654e-04f);
    q = fmaf(x2, q, 2.26843463243900e-03f);
    q = fmaf(x2, q, 4.89352518554385e-03f);
    return __fdividef(x * p, q);
}
