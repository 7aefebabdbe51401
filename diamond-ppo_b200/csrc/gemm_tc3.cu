// CTA-pair (tcgen05 cta_group::2) 3xTF32 GEMM of the wide actor-critic MLP (diamond/ppo.py:261 forward, :283 dgrad):
//   C[M,N] = epi(A[M,K] * B^T)     A: fp32 activations, B: pre-split weight images (prep_weights_kernel, gemm_tc.cu)
//
// Why pairs: measured on B200, a shared-memory-operand tcgen05.mma of one CTA (M=128, N=256, K=8 tf32) is paced by the
// tensor core's 64 B/clk operand port -- it fetches 4 KB of A and 8 KB of B per instruction, 192 clk instead of the 128 clk
// the math needs -- and 148 CTAs each streaming full weight chunks ask the L2 for more than it delivers.  With
// cta_group::2 the two SMs of a TPC compute one 256 x 256 tile together: each SM feeds its own 128 rows of A and HALF of the
// weight rows (8 KB per instruction per SM = the port rate), keeps 128 x 256 of the accumulator in its own TMEM, and loads
// half of the weight bytes.  A ring stage shrinks to 32 KB, so six stages fit beside the epilogue staging.
//
// One cluster = 2 CTAs x 448 threads (same roles in both CTAs; see gemm_tc2.cu for the 1-CTA variant):
//   warp 0      producer : TMA for this CTA's 128 activation rows + bulk copies of its half of the weight chunk
//   warp 1      MMA      : leader CTA only -- issues tcgen05.mma.cta_group::2, commits (multicast) to both CTAs' barriers
//   warps 2-5   split    : hi/lo split of this CTA's activation chunk, then one arrival per warp on the LEADER's barrier
//   warps 6-13  epilogue : tcgen05.ld of this CTA's 128 x 256 accumulator half, layer epilogue, staged TMA store
// Accumulators are double-buffered in TMEM (2 x 256 columns), so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// FMT = DPPO_TC_FMT_F16 (forward launches whose A is a tanh output, gemm_tc.cuh): the split warps write fp16 hi/lo images of
// A * 2^14 beside the raw fp32 chunk, the weight images are fp16 pairs of W * s_n, and the MMA warp issues three kind::f16
// MMAs (K = 16) per chunk -- the tensor pipe's 16-bit rate, twice the FLOPs per clock of kind::tf32.  The epilogue scales the
// accumulator back by 2^-14 / s_n before the bias.  A stage is 24 KB ([A raw 8 | A hi 4 | A lo 4 | B hi 4 | B lo 4]) and holds
// half the MMA time of a TF32 stage, so the ring is eight stages deep.
#include <cuda.h>

#include "tc_common.cuh"
#include "gemm_tc.cuh"

using namespace tc;

namespace {

constexpr int THREADS = 448;
constexpr int W_PROD = 0, W_MMA = 1, W_SPLIT0 = 2, N_SPLIT = 4, W_EPI0 = 6, N_EPI = 8;
constexpr int SPLIT_THREADS = N_SPLIT * 32;
constexpr int KC = 16;                     // k per chunk (one SWIZZLE_64B atom width)
constexpr int BM = 128;                    // rows per CTA (the pair computes 256)
constexpr int A_IMG = BM * KC * 4;         // 8 KB: one image (hi or lo) of this CTA's activation chunk
constexpr int MAX_STAGES = 8;
// Ring depth: six 32 KB stages for the forward GEMM; the dgrad variant gives one stage to the epilogue warps, which receive their
// 32 x 32 tiles of the layer's activations (tanh' factors) by TMA instead of thread-per-row global loads (32 different 128-byte
// lines per load instruction: 1.27x the algorithmic DRAM traffic and 12 us per launch, profiles/r1f_kernels.csv).
template <int EPI, int FMT> struct RingDepth { static constexpr int v = FMT == DPPO_TC_FMT_F16 ? 8 : EPI == DPPO_EPI_TANH_BWD ? 5 : 6; };
template <int FMT> struct Fmt {
    static constexpr bool f16 = FMT == DPPO_TC_FMT_F16;
    static constexpr int b_row = f16 ? KC * 2 : KC * 4;                // bytes of one weight row of a chunk image
    static constexpr int a_hi = f16 ? A_IMG : 0;                       // stage offsets of the A images (TF32: the raw chunk is hi)
    static constexpr int a_lo = f16 ? A_IMG + A_IMG / 2 : A_IMG;
};
constexpr int STG_BLK = 32 * 128;          // one 32-row x 32-column fp32 staging block (SWIZZLE_128B layout)

template <int EPI, int FMT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
tc3_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmH,
                const unsigned char* __restrict__ Wimg, const float* __restrict__ bias, float* __restrict__ colsum, int64_t M,
                int N, int K, int n_tile, int pair_tiles, int tail_halves, int rev, int dbg, const int* __restrict__ m_dev)
{
    if (m_dev != nullptr) {                              // row count decided on the device (tiles past it are never touched)
        const int64_t md = *m_dev;
        if (md < M) M = md < 0 ? 0 : md;
        pair_tiles = (int)((M + 2 * BM - 1) / (2 * BM));
        if (tail_halves == 1) tail_halves = 0;           // the tail split was planned for the host's row count
    }
    extern __shared__ unsigned char dyn_raw[];
    constexpr int STAGES = RingDepth<EPI, FMT>::v;
    using F = Fmt<FMT>;
    __shared__ __align__(8) uint64_t full[MAX_STAGES], ready[MAX_STAGES], empty[MAX_STAGES], tfull[2], tempty[2], hbar[N_EPI];
    __shared__ uint32_t s_tmem;

    unsigned char* dyn = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(dyn_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const bool in_first = (rev & 2) != 0;                // inputs are read with the L2 evict-first hint (dppo_tc3_gemm)
    const bool no_pf = (rev & 4) != 0;                   // no L2 prefetch of the next tile's activations (the default, see dppo_tc3_gemm)
    rev &= 1;
    const int half_n = n_tile / 2;                       // weight rows held by each CTA
    const int b_half = half_n * F::b_row;                // bytes of one image (hi or lo) of this CTA's weight rows
    const int b_img = n_tile * F::b_row;                 // bytes of one full image in the weight-image buffer
    const int stage_bytes = 2 * A_IMG + 2 * b_half;      // [A_hi | A_lo | B_hi(half) | B_lo(half)], f16: [A | A_hi | A_lo | ...]
    const int n_tiles = N / n_tile;
    const int total = pair_tiles * n_tiles;
    const int chunks = K / KC;
    // Tile schedule of this cluster: `base` full 256 x n_tile tiles (round robin), then the remainder.  When the remainder
    // R satisfies 2R <= clusters (tail_halves), each leftover tile is split into two half-width (n_tile/2 columns) tiles
    // that go to different clusters: the makespan drops from base + 1 to base + ~0.63 tiles.
    // tail_halves == 2 (small problems: fewer full tiles than half of the clusters): EVERY tile is split into its two half-width
    // tiles, so twice as many SM pairs work and each runs the cheaper N = n_tile/2 instruction.
    const bool all_halves = tail_halves == 2;
    const int units = all_halves ? 2 * total : total;
    const int base_tiles = units / n_clusters, rem_tiles = units - base_tiles * n_clusters;
    const int extra = tail_halves == 1 ? (cluster_id < 2 * rem_tiles ? 1 : 0) : (cluster_id < rem_tiles ? 1 : 0);
    const int n_my = base_tiles + extra;
    auto tile_of = [&](int i, int& tile, int& half) {
        if (all_halves) { const int u = i * n_clusters + cluster_id; tile = u >> 1; half = u & 1; }
        else if (i < base_tiles) { tile = i * n_clusters + cluster_id; half = -1; }
        else if (tail_halves) { tile = base_tiles * n_clusters + (cluster_id >> 1); half = cluster_id & 1; }
        else { tile = base_tiles * n_clusters + cluster_id; half = -1; }
        if (rev) tile = total - 1 - tile;                // row sweep from the last rows to the first (see dppo_tc3_gemm)
    };

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&ready[s], 2 * N_SPLIT); mbar_init(&empty[s], 1); }
#pragma unroll
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * N_EPI); }
#pragma unroll
        for (int w = 0; w < N_EPI; ++w) mbar_init(&hbar[w], 1);
        fence_mbar_init();
    }
    if (warp == W_MMA) tmem_alloc2(&s_tmem, 512);
    fence_before();
    cluster_sync();                                      // barriers of both CTAs initialised before any remote arrival
    fence_after();
    const uint32_t tmem = s_tmem;
    DPPO_PDL_ENTER();                                    // set-up done; global memory only after the predecessor grid completed

    if (warp == W_PROD) {
        if (lane == 0) {
            tma_prefetch_desc(&tmA);
            const uint64_t pol = l2_policy_evict_first();
            int s = 0;
            uint32_t ph = 0;
            for (int i = 0; i < n_my; ++i) {
                int tile, half;
                tile_of(i, tile, half);
                const int m_pair = tile / n_tiles, n_blk = tile - m_pair * n_tiles;
                const int m0 = m_pair * 2 * BM + (int)rank * BM;
                const int n_eff = half < 0 ? n_tile : n_tile / 2;                  // columns of this tile
                const int hb = (n_eff / 2) * F::b_row;                             // bytes of this CTA's rows of one image
                const int row_off = (half < 0 ? 0 : half * (n_tile / 2)) + (int)rank * (n_eff / 2);
                const unsigned char* wsrc = Wimg + (int64_t)n_blk * chunks * 2 * b_img + (int64_t)row_off * F::b_row;
                int next_m = -1;
                if (i + 1 < n_my) { int nt, nh; tile_of(i + 1, nt, nh); next_m = nt / n_tiles; }
                for (int c = 0; c < chunks; ++c) {
                    // pull the next tile's activations into L2 while this tile computes
                    if (!no_pf && next_m >= 0 && next_m != m_pair) {
                        if (in_first) tma_prefetch_2d_hint(&tmA, c * KC, next_m * 2 * BM + (int)rank * BM, pol);
                        else tma_prefetch_2d(&tmA, c * KC, next_m * 2 * BM + (int)rank * BM);
                    }
                    mbar_wait(&empty[s], ph ^ 1);
                    const bool skip_b = DPPO_DBG(dbg, 1) && (i != 0 || c >= STAGES);
                    mbar_expect_tx(&full[s], (uint32_t)(A_IMG + (skip_b ? 0 : 2 * hb)));
                    unsigned char* st = dyn + s * stage_bytes;
                    if (in_first) tma_load_2d_hint(st, &tmA, c * KC, m0, &full[s], pol);
                    else tma_load_2d(st, &tmA, c * KC, m0, &full[s]);
                    if (!skip_b) {
                        const unsigned char* w = wsrc + (int64_t)c * 2 * b_img;
                        bulk_copy_g2s(st + 2 * A_IMG, w, (uint32_t)hb, &full[s]);                        // hi rows of this CTA
                        bulk_copy_g2s(st + 2 * A_IMG + b_half, w + b_img, (uint32_t)hb, &full[s]);       // lo rows of this CTA
                    }
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == W_MMA) {
        if (rank == 0 && lane == 0) {
            const uint32_t idesc_full = F::f16 ? idesc_f16(2 * BM, n_tile) : idesc_tf32(2 * BM, n_tile, 0, 0);
            const uint32_t idesc_half = F::f16 ? idesc_f16(2 * BM, n_tile / 2) : idesc_tf32(2 * BM, n_tile / 2, 0, 0);
            int s = 0;
            uint32_t ph = 0;
            for (uint32_t it = 0; it < (uint32_t)n_my; ++it) {
                int tile, half;
                tile_of((int)it, tile, half);
                const uint32_t idesc = half < 0 ? idesc_full : idesc_half;
                const uint32_t set = it & 1;
                mbar_wait(&tempty[set], ((it >> 1) & 1) ^ 1);            // both CTAs' epilogues have drained this accumulator
                fence_after();
                const uint32_t d = tmem + set * 256;
                for (int c = 0; c < chunks; ++c) {
                    mbar_wait(&ready[s], ph);                           // both CTAs: chunk landed and split
                    fence_after();
                    const uint32_t st0 = smem_u32(dyn + s * stage_bytes), a_hi = st0 + F::a_hi, a_lo = st0 + F::a_lo;
                    const uint32_t b_hi = st0 + 2 * A_IMG, b_lo = b_hi + (uint32_t)b_half;
                    if (F::f16) {                                       // one 16-wide k-step: the whole SWIZZLE_32B row
                        if (!DPPO_DBG(dbg, 4)) {
                            umma_f16_2cta(d, desc_k_sw32(a_hi), desc_k_sw32(b_lo), idesc, c != 0);
                            umma_f16_2cta(d, desc_k_sw32(a_lo), desc_k_sw32(b_hi), idesc, 1u);
                            umma_f16_2cta(d, desc_k_sw32(a_hi), desc_k_sw32(b_hi), idesc, 1u);
                        } else {
                            umma_f16_2cta(d, desc_k_sw32(a_hi), desc_k_sw32(b_hi), idesc, c != 0);
                        }
                    } else {
#pragma unroll
                    for (int ks = 0; ks < KC / 8; ++ks) {
                        const uint32_t ko = ks * 32;                    // 8 tf32 = 32 bytes along K inside the swizzle atom
                        if (!DPPO_DBG(dbg, 4)) {
                            umma_tf32_2cta(d, desc_k_sw64(a_hi + ko), desc_k_sw64(b_lo + ko), idesc, (c | ks) != 0);
                            umma_tf32_2cta(d, desc_k_sw64(a_lo + ko), desc_k_sw64(b_hi + ko), idesc, 1u);
                            umma_tf32_2cta(d, desc_k_sw64(a_hi + ko), desc_k_sw64(b_hi + ko), idesc, 1u);
                        } else {
                            umma_tf32_2cta(d, desc_k_sw64(a_hi + ko), desc_k_sw64(b_hi + ko), idesc, (c | ks) != 0);
                        }
                    }
                    }
                    umma_commit_2cta(&empty[s], 3);                     // frees the stage in both CTAs
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
                umma_commit_2cta(&tfull[set], 3);
            }
        }
        __syncwarp();
    } else if (warp < W_EPI0) {
        // hi/lo split of this CTA's activation chunk; one arrival per warp on the leader's ready barrier
        const int ct = tid - W_SPLIT0 * 32;
        constexpr int PER = A_IMG / 16 / SPLIT_THREADS;
        int s = 0;
        uint32_t ph = 0;
        for (int i = 0; i < n_my; ++i) {
            for (int c = 0; c < chunks; ++c) {
                mbar_wait(&full[s], ph);
                if (F::f16) {
                    // thread -> (row, 8-wide k half) pairs: two 16-byte segments of the raw SWIZZLE_64B row in, one 16-byte segment
                    // of each SWIZZLE_32B fp16 image out (both conflict-free per quarter warp)
                    const uint32_t raw = smem_u32(dyn + s * stage_bytes);
                    float4 x[4];
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int p = ct + j * SPLIT_THREADS, row = p >> 1, c2 = (p & 1) * 2, sw = (row >> 1) & 3;
                        x[2 * j] = lds128(raw + row * 64 + ((c2 ^ sw) << 4));
                        x[2 * j + 1] = lds128(raw + row * 64 + (((c2 + 1) ^ sw) << 4));
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int p = ct + j * SPLIT_THREADS, row = p >> 1;
                        const uint32_t o = (uint32_t)(row * 32 + ((((p & 1) ^ (row >> 2)) & 1) << 4));
                        uint4 h, l;
                        split_f16x8(x[2 * j], x[2 * j + 1], (float)(1 << DPPO_F16_A_EXP), h, l);
                        sts128u(raw + F::a_hi + o, h);
                        sts128u(raw + F::a_lo + o, l);
                    }
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&ready[s]), 0));
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                    continue;
                }
                const uint32_t hi = smem_u32(dyn + s * stage_bytes) + ct * 16;
                float4 x[PER];
#pragma unroll
                for (int j = 0; j < PER; ++j) x[j] = lds128(hi + j * SPLIT_THREADS * 16);
                if (DPPO_DBG(dbg, 1024)) {                                       // A/B: round-to-nearest hi image stored in place
#pragma unroll
                    for (int j = 0; j < PER; ++j) {
                        const float4 l = split_tf32x4(x[j]);
                        sts128(hi + j * SPLIT_THREADS * 16, x[j]);
                        sts128(hi + A_IMG + j * SPLIT_THREADS * 16, l);
                    }
                } else {                                                // the raw chunk is the hi image; only lo is written
#pragma unroll
                    for (int j = 0; j < PER; ++j) sts128(hi + A_IMG + j * SPLIT_THREADS * 16, lo_of_trunc_x4(x[j]));
                }
                fence_proxy_async();                                    // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&ready[s]), 0));
                if (++s == STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else {
        // epilogue over this CTA's 128 rows: warp -> TMEM lane quadrant (warp % 4) and column half.  Results leave through a
        // per-warp 32x32 staging block in the SWIZZLE_128B layout and a TMA store (full 128-byte row segments reach HBM).
        const int ew = warp - W_EPI0;
        const int q = warp & 3, grp = ew >> 2;
        const uint32_t stg = smem_u32(dyn + STAGES * stage_bytes) + (uint32_t)ew * STG_BLK;
        // dgrad: this warp's landing block for the 32 x 32 activation tiles (SWIZZLE_128B, as delivered by TMA) + its barrier
        unsigned char* hblk = dyn + STAGES * stage_bytes + N_EPI * STG_BLK + ew * STG_BLK;
        const uint32_t hst = smem_u32(hblk);
        uint32_t hph = 0;
        const uint32_t row_off = (uint32_t)lane * 128, sw = (uint32_t)(lane & 7);
        if (lane == 0) { tma_prefetch_desc(&tmC); if (EPI == DPPO_EPI_TANH_BWD) tma_prefetch_desc(&tmH); }
        for (uint32_t it = 0; it < (uint32_t)n_my; ++it) {
            int tile, half;
            tile_of((int)it, tile, half);
            const int m_pair = tile / n_tiles, n_blk = tile - m_pair * n_tiles;
            const int n_eff = half < 0 ? n_tile : n_tile / 2;
            const int ncols = n_eff / 2;                                 // columns of this warp group
            const int col0 = grp * ncols;                                // first accumulator column of this warp group
            const int nblk = ncols / 32;
            const int n0 = n_blk * n_tile + (half < 0 ? 0 : half * (n_tile / 2)) + col0;
            const int m0 = m_pair * 2 * BM + (int)rank * BM + q * 32;
            const uint32_t set = it & 1;
            if (EPI == DPPO_EPI_TANH_BWD && lane == 0 && !DPPO_DBG(dbg, 8)) {
                // the first activation tile of this output tile travels while the MMAs of the tile are still running
                mbar_expect_tx(&hbar[ew], (uint32_t)STG_BLK);
                tma_load_2d(hblk, &tmH, n0, m0, &hbar[ew]);
            }
            mbar_wait(&tfull[set], (it >> 1) & 1);
            fence_after();
            for (int k = 0; k < (DPPO_DBG(dbg, 8) ? 0 : nblk); ++k) {
                const int n = n0 + k * 32;
                uint32_t r[32];
                tmem_ld32_issue(tmem + set * 256 + ((uint32_t)(q * 32) << 16) + (uint32_t)(col0 + k * 32), r);
                float4 aux[8];                                          // bias (forward) or the layer's activations (dgrad)
                float4 fac[8];                                          // f16: column factors 2^-14 / s_n
                if (EPI == DPPO_EPI_BIAS_TANH) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) aux[j] = __ldg(reinterpret_cast<const float4*>(bias + n) + j);
                    if (F::f16) {
                        const float* f = reinterpret_cast<const float*>(Wimg + dppo_tc_f16_factor_offset(N, K));
#pragma unroll
                        for (int j = 0; j < 8; ++j) fac[j] = __ldg(reinterpret_cast<const float4*>(f + n) + j);
                    }
                } else {
                    mbar_wait(&hbar[ew], hph);
                    hph ^= 1u;
#pragma unroll
                    for (int j = 0; j < 8; ++j) aux[j] = lds128(hst + row_off + ((((uint32_t)j) ^ sw) << 4));    // rows >= M: zero-filled
                    __syncwarp();
                    if (lane == 0 && k + 1 < nblk) {                    // next tile of activations: overlaps this block's epilogue work
                        fence_proxy_async();
                        mbar_expect_tx(&hbar[ew], (uint32_t)STG_BLK);
                        tma_load_2d(hblk, &tmH, n + 32, m0, &hbar[ew]);
                    }
                }
                tmem_ld32_wait(r);
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                if (EPI == DPPO_EPI_BIAS_TANH && F::f16) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {                               // exact: powers of two, no over- or underflow
                        v[4 * j] *= fac[j].x; v[4 * j + 1] *= fac[j].y; v[4 * j + 2] *= fac[j].z; v[4 * j + 3] *= fac[j].w;
                    }
                }
                if (EPI == DPPO_EPI_BIAS_TANH) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (DPPO_DBG(dbg, 32)) {
                            v[4 * j] += aux[j].x; v[4 * j + 1] += aux[j].y; v[4 * j + 2] += aux[j].z; v[4 * j + 3] += aux[j].w;
                        } else {
                            v[4 * j] = tanh_rational(v[4 * j] + aux[j].x); v[4 * j + 1] = tanh_rational(v[4 * j + 1] + aux[j].y);
                            v[4 * j + 2] = tanh_rational(v[4 * j + 2] + aux[j].z); v[4 * j + 3] = tanh_rational(v[4 * j + 3] + aux[j].w);
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        v[4 * j] *= (1.0f - aux[j].x * aux[j].x); v[4 * j + 1] *= (1.0f - aux[j].y * aux[j].y);
                        v[4 * j + 2] *= (1.0f - aux[j].z * aux[j].z); v[4 * j + 3] *= (1.0f - aux[j].w * aux[j].w);
                    }
                }
                if (lane == 0) bulk_wait_read<0>();                     // the previous store has read the staging block
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    sts128(stg + row_off + ((((uint32_t)j) ^ sw) << 4), make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
                fence_proxy_async();
                __syncwarp();
                if (lane == 0 && !DPPO_DBG(dbg, 16)) {
                    tma_store_2d(&tmC, n, m0, stg);                     // rows >= M are clipped by the tensor map
                    bulk_commit();
                }
                if (EPI == DPPO_EPI_TANH_BWD && colsum != nullptr && !DPPO_DBG(dbg, 16384)) {
                    // Bias-gradient partials: one row of column sums per (CTA, lane quadrant), accumulated over all tiles of
                    // this CTA (the row is owned by this warp pair).  With a single column tile every CTA covers all N
                    // columns in its first tile, which then initialises the row; otherwise the launcher zeroes the buffer.
                    // Rows >= M hold exact zeros (TMA zero-fills the out-of-range A rows), so they do not disturb the sums.
                    float* cp = colsum + ((int64_t)gridDim.x + (int64_t)blockIdx.x * 4 + q) * N + n + lane;      // working row of (CTA, quadrant)
                    const float prev = (n_tiles == 1 && it == 0 && half < 0) ? 0.0f : *cp;
                    // warp transpose-reduce: afterwards lane l holds the sum over the warp's 32 rows of column l
#pragma unroll
                    for (int o = 16; o >= 1; o >>= 1) {
#pragma unroll
                        for (int i = 0; i < o; ++i) {
                            const bool up = lane & o;
                            const float send = up ? v[i] : v[i + o];
                            const float keep = up ? v[i + o] : v[i];
                            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                        }
                    }
                    *cp = prev + v[0];
                }
            }
            fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&tempty[set]), 0));
        }
        if (lane == 0) bulk_wait<0>();             // staging memory must outlive the last store's read
        __syncwarp();
        if (EPI == DPPO_EPI_TANH_BWD && colsum != nullptr) {
            // fold the four quadrant rows of this CTA into its one partial row (fixed order): rows [0, grid) are what the
            // gradient reduction reads, rows [grid, 5 grid) the per-quadrant working rows
            __threadfence_block();
            asm volatile("bar.sync 1, 256;" ::: "memory");                       // the eight epilogue warps
            const float* wr = colsum + ((int64_t)gridDim.x + (int64_t)blockIdx.x * 4) * N;
            for (int col = tid - W_EPI0 * 32; col < N; col += N_EPI * 32)
                colsum[(int64_t)blockIdx.x * N + col] = (__ldcg(wr + col) + __ldcg(wr + N + col)) + (__ldcg(wr + 2 * N + col) + __ldcg(wr + 3 * N + col));
        }
    }

    // no CTA may exit (or free TMEM) while its peer can still touch its shared memory, barriers or TMEM
    fence_before();
    cluster_sync();
    if (warp == W_MMA) {
        fence_after();
        tmem_dealloc2(tmem, 512);
    }
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

namespace {
// Tile schedule of a launch: grid (2 CTAs per cluster) and how the tiles are cut.  mode 0: full 256 x n_tile tiles round robin;
// 1: the remainder tiles are split into half-width tiles (one per cluster); 2: every tile is split (small problems).
// Makespans are compared in full-tile units; a half-width tile costs ~0.63 of a full one (the N = 128 instruction is paced by
// operand fetch, dppo_tc_mma_probe).
void tc3_plan(dppo_ctx* ctx, int64_t M, int N, int* grid_out, int* mode_out)
{
    const int n_tile = dppo_tc_n_tile(N);
    const int64_t total = ((M + 2 * BM - 1) / (2 * BM)) * (N / n_tile);
    const int64_t max_clusters = ctx->sm_count / 2;
    if (total < 1 || max_clusters < 1) { *grid_out = 2; *mode_out = 0; return; }      // unsupported shape (sizing calls only)
    int64_t clusters = max_clusters < total ? max_clusters : total;
    const int64_t base = total / clusters, rem = total - base * clusters;
    int mode = (!DPPO_DBG(ctx->tc_debug, 128) && n_tile == 256 && base >= 1 && rem > 0 && 2 * rem <= clusters) ? 1 : 0;
    if (n_tile == 256 && !DPPO_DBG(ctx->tc_debug, 128) && ctx->rows_dev == nullptr) {
        const double full_span = (double)base + (rem > 0 ? (mode == 1 ? 0.63 : 1.0) : 0.0);
        const double half_span = 0.63 * (double)((2 * total + max_clusters - 1) / max_clusters);
        if (half_span < full_span - 0.05) {
            mode = 2;
            clusters = max_clusters < 2 * total ? max_clusters : 2 * total;
        }
    }
    *grid_out = (int)(2 * clusters);
    *mode_out = mode;
}
int tc3_grid(dppo_ctx* ctx, int64_t M, int N)
{
    int grid, mode;
    tc3_plan(ctx, M, N, &grid, &mode);
    return grid;
}
}  // namespace

int dppo_tc3_colsum_parts(dppo_ctx* ctx, int64_t M, int N) { return tc3_grid(ctx, M, N); }      // one partial row per CTA
int dppo_tc3_colsum_rows(dppo_ctx* ctx, int64_t M, int N) { return 5 * tc3_grid(ctx, M, N); }       // + 4 working rows per CTA

bool dppo_tc3_gemm_supported(int64_t M, int N, int K)
{
    return M >= 1024 && M < (int64_t)1 << 31 && K % KC == 0 && (N % 256 == 0 || N == 128);
}

// rev != 0: the tiles are visited from the last rows to the first.  Consecutive launches of a layer chain alternate their sweep
// direction (api.cu), so that a launch starts with the rows its predecessor wrote LAST -- the part of the activations that is still
// in the L2 -- instead of the rows that were evicted first (an ascending sweep over 67-134 MB after an ascending sweep is the
// worst case of an LRU-like cache: nothing is ever hit).  rev & 2: the A operand is read with the L2 evict-first hint.
// The L2 prefetch of the NEXT tile's activations (one box per chunk while the current tile computes; round 1) is off by default
// (tc_prefetch): in-situ DRAM counters showed the prefetched lines being fetched twice -- dgrad3 read 206 MB against 169 MB
// without it (profiles/r4e_prefetch_ab.md) -- and the optimiser step is 1.4 % faster without (2.7 % with the weight-gradient
// kernel's chunk prefetch off as well).
int dppo_tc3_gemm(dppo_ctx* ctx, int epi, const float* A, int lda, const unsigned char* Wimg, const float* bias, const float* Hact,
                  int ldh, float* C, int ldc, float* colsum, int64_t M, int N, int K, int rev, cudaStream_t st, int fmt)
{
    if (!dppo_tc3_gemm_supported(M, N, K)) DPPO_FAIL(ctx, "tc3_gemm: unsupported shape M=%lld N=%d K=%d", (long long)M, N, K);
    const bool f16 = fmt == DPPO_TC_FMT_F16;
    if (fmt != DPPO_TC_FMT_TF32 && !(f16 && epi == DPPO_EPI_BIAS_TANH)) DPPO_FAIL(ctx, "tc3_gemm: operand format %d with epilogue %d", fmt, epi);
    if (lda % 4 != 0 || ldc % 4 != 0 || !al16(A) || !al16(C) || !al16(Wimg) || (Hact && (!al16(Hact) || ldh % 4 != 0)) || (bias && !al16(bias)))
        DPPO_FAIL(ctx, "tc3_gemm: operands must be 16-byte aligned with row pitches multiple of 4 floats");
    CUtensorMap tmA, tmC, tmH;
    if (!dppo_make_tensor_map_2d(&tmA, A, M, K, lda, KC, BM, 2) || !dppo_make_tensor_map_2d(&tmC, C, M, N, ldc, 32, 32, 3))
        DPPO_FAIL(ctx, "tc3_gemm: cuTensorMapEncodeTiled failed");
    tmH = tmC;
    if (epi == DPPO_EPI_TANH_BWD && !dppo_make_tensor_map_2d(&tmH, Hact, M, N, ldh, 32, 32, 3))      // activation tiles of the epilogue
        DPPO_FAIL(ctx, "tc3_gemm: cuTensorMapEncodeTiled(Hact) failed");
    const int n_tile = dppo_tc_n_tile(N);
    const int pair_tiles = (int)((M + 2 * BM - 1) / (2 * BM));
    const int stages = epi == DPPO_EPI_TANH_BWD ? RingDepth<DPPO_EPI_TANH_BWD, DPPO_TC_FMT_TF32>::v
                       : f16 ? RingDepth<DPPO_EPI_BIAS_TANH, DPPO_TC_FMT_F16>::v : RingDepth<DPPO_EPI_BIAS_TANH, DPPO_TC_FMT_TF32>::v;
    const int b_row = f16 ? Fmt<DPPO_TC_FMT_F16>::b_row : Fmt<DPPO_TC_FMT_TF32>::b_row;
    const size_t smem = (size_t)stages * (2 * A_IMG + n_tile * b_row) + (size_t)N_EPI * STG_BLK * (epi == DPPO_EPI_TANH_BWD ? 2 : 1) + 1024;
    int grid, tail_halves;
    tc3_plan(ctx, M, N, &grid, &tail_halves);
    if (!(ctx->tc_prefetch & (epi == DPPO_EPI_TANH_BWD ? 2 : 1))) rev |= 4;
    if (epi == DPPO_EPI_TANH_BWD && colsum != nullptr && (N / n_tile > 1 || tail_halves == 2) &&
        cudaMemsetAsync(colsum + (size_t)grid * N, 0, (size_t)4 * grid * N * sizeof(float), st) != cudaSuccess)
        DPPO_FAIL(ctx, "tc3_gemm: cudaMemsetAsync(colsum) failed");
    if (epi == DPPO_EPI_BIAS_TANH) {
        const auto kern = f16 ? tc3_gemm_kernel<DPPO_EPI_BIAS_TANH, DPPO_TC_FMT_F16> : tc3_gemm_kernel<DPPO_EPI_BIAS_TANH, DPPO_TC_FMT_TF32>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        // forward launches follow each other (and the weight-image kernel) directly: with programmatic stream serialisation the
        // launch latency and the per-CTA set-up (barriers, TMEM allocation, tensor-map fetch) of layer i + 1 hide under the tail of
        // layer i (pre-update pass 3.07 -> 2.93 ms at config S; neutral inside the training step).  The kernel touches global
        // memory only after griddepcontrol.wait.
        dppo_launch_pdl_if(true, kern, dim3(grid), dim3(THREADS), smem, st, tmA, tmC, tmH, Wimg, bias, colsum, M,
                           N, K, n_tile, pair_tiles, tail_halves, rev, ctx->tc_debug, ctx->rows_dev);
    } else if (epi == DPPO_EPI_TANH_BWD) {
        cudaFuncSetAttribute(tc3_gemm_kernel<DPPO_EPI_TANH_BWD, DPPO_TC_FMT_TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        dppo_launch_pdl(ctx, tc3_gemm_kernel<DPPO_EPI_TANH_BWD, DPPO_TC_FMT_TF32>, dim3(grid), dim3(THREADS), smem, st, tmA, tmC, tmH, Wimg, bias, colsum, M,
                        N, K, n_tile, pair_tiles, tail_halves, rev, ctx->tc_debug, ctx->rows_dev);
    } else {
        DPPO_FAIL(ctx, "tc3_gemm: unknown epilogue %d", epi);
    }
    DPPO_CHECK_LAUNCH(ctx, "tc3_gemm_kernel");
    return 0;
}
