#pragma once
#include "common.cuh"

// Operand formats of the forward GEMM (gemm_tc3.cu).  TF32: three kind::tf32 MMAs per k-step on hi/lo TF32 images.
// F16: three kind::f16 MMAs per k-step on fp16 hi/lo pairs of scaled operands, A' = A * 2^DPPO_F16_A_EXP (needs |A| < 4, i.e.
// A is the output of a tanh epilogue) and W' = W * s_n with one power of two s_n per output row n (weight_images.cu).
enum { DPPO_TC_FMT_TF32 = 0, DPPO_TC_FMT_F16 = 1 };
constexpr int DPPO_F16_A_EXP = 14;
// An fp16 image of an [N, K] operand ends with N fp32 column factors 2^-DPPO_F16_A_EXP / s_n at this byte offset: the epilogue's
// accumulator scale (both factors are exact powers of two)
__host__ __device__ __forceinline__ int64_t dppo_tc_f16_factor_offset(int N, int K) { return (int64_t)N * K * 4; }

// weight images of the tcgen05 GEMMs (weight_images.cu)
int dppo_tc_n_tile(int N);
int64_t dppo_tc_image_bytes(int N, int K);        // bytes of the hi/lo weight images of an [N, K] B operand (either format)
int dppo_tc_prep_weights(dppo_ctx* ctx, const float* W, int rows_w, int cols_w, int transpose, unsigned char* img, cudaStream_t st);
// f16: build the fp16 format (transpose 0 only) instead of TF32
struct PrepJob { const float* W; int rows_w, cols_w, transpose, n_tile, f16; unsigned char* img; };
// optional row gather riding in the same launch (blockIdx.y == n): dst[i, :] = src[idx[i], :], row_vec float4 per row
struct GatherJob { const float4* src; const int32_t* idx; float4* dst; int64_t rows; int row_vec; };
struct PrepJobs { PrepJob job[8]; int n; GatherJob gather; };
int dppo_tc_prep_weights_multi(dppo_ctx* ctx, PrepJobs jobs, cudaStream_t st);      // every job in one launch

// tcgen05 weight gradient (wgrad_tc.cu): TMA-fed operand ring, dedicated split / MMA / epilogue warps.
// dW[N1,N2] = sum_m D[m,N1] * H[m,N2] as `splits` deterministic row-range partials [splits][N1][N2]
bool dppo_tc2_wgrad_supported(int64_t M, int N1, int N2);
int dppo_tc2_wgrad_splits(dppo_ctx* ctx, int64_t M, int N1, int N2);
int dppo_tc2_wgrad(dppo_ctx* ctx, const float* Dm, int ldd, const float* Hm, int ldh, float* partials, int splits, int64_t M, int N1,
                   int N2, cudaStream_t st);
// up to three weight gradients over the same M rows in ONE launch, row ranges balanced so that all CTAs carry equal work
void dppo_tc2_wgrad_multi_splits(dppo_ctx* ctx, int64_t M, int n, const int* N1, const int* N2, int* splits_out);
int dppo_tc2_wgrad_multi(dppo_ctx* ctx, int n, const float* const* Dm, const int* ldd, const float* const* Hm, const int* ldh,
                         float* const* partials, const int* splits, int64_t M, const int* N1, const int* N2, cudaStream_t st);

// CTA-pair (cta_group::2) variant of the forward / dgrad GEMM (gemm_tc3.cu)
bool dppo_tc3_gemm_supported(int64_t M, int N, int K);
int dppo_tc3_colsum_parts(dppo_ctx* ctx, int64_t M, int N);   // partial rows of the TANH_BWD epilogue the reduction reads: one per CTA
int dppo_tc3_colsum_rows(dppo_ctx* ctx, int64_t M, int N);    // rows the colsum buffer must hold (partials + per-quadrant working rows)
// fmt (DPPO_TC_FMT_*): the format of Wimg; DPPO_TC_FMT_F16 only with DPPO_EPI_BIAS_TANH
int dppo_tc3_gemm(dppo_ctx* ctx, int epi, const float* A, int lda, const unsigned char* Wimg, const float* bias, const float* Hact,
                  int ldh, float* C, int ldc, float* colsum, int64_t M, int N, int K, int rev, cudaStream_t st, int fmt = DPPO_TC_FMT_TF32);
