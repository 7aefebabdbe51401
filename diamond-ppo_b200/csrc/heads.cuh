#pragma once
#include "common.cuh"

constexpr int HEAD_WARPS = 8;

struct HeadTrainArgs {
    const float* h3;          // [M, 2H] tanh activations of actor_head.0 | critic_head.0
    float* d3;                // [M, 2H] gradient w.r.t. their pre-activations (output)
    const float *wa, *ba, *wc, *bc, *log_std;
    const int32_t* idx;       // minibatch row -> flat sample index (may be null)
    const int32_t* actions_i; // [B]     (discrete)
    const float* actions_f;   // [B, A]  (continuous)
    const float *old_logp, *adv, *ret;
    const double* adv_stats;
    int64_t adv_count;
    int advantage_norm;
    int64_t M;
    int H, A;
    float clip, vw, beta, inv_m;
    float* partials;          // [blocks, partial_stride]
    int partial_stride;
    int rev;                  // role-split kernel: rows are visited from the last to the first (L2 reuse, gemm_tc3.cu dppo_tc3_gemm)
    int h3_first;             // role-split kernel: h3 (never read again) is loaded with the L2 evict-first hint
    int keep_d3;              // role-split kernel: plain instead of streaming (evict-first) stores of d3, which the next launch reads
};

// Layout of one head-kernel partial: [dWa A*H | dba A | dWc H | dbc 1 | dlog_std A | db3 2H | losses 4], every block starting on a
// multiple of 4 floats so that the gradient reduction reads all of them as float4 (an unaligned db3 block took the scalar path
// and was the long pole of grad_reduce_kernel).
struct HeadOffsets { int dba, dwc, dbc, dls, b3, loss, total; };
__host__ __device__ inline HeadOffsets head_offsets(int H, int A)
{
    auto up4 = [](int x) { return (x + 3) / 4 * 4; };
    HeadOffsets o;
    o.dba = up4(A * H);
    o.dwc = up4(o.dba + A);
    o.dbc = up4(o.dwc + H);
    o.dls = up4(o.dbc + 1);
    o.b3 = up4(o.dls + A);
    o.loss = up4(o.b3 + 2 * H);
    o.total = o.loss + 4;
    return o;
}
int head_partial_floats(int H, int A);
int head_train_blocks(dppo_ctx* ctx, int64_t M, int H, int A);
bool head_train_supported(int H, int A);      // the shapes launch_head_train_kernel accepts (dppo_mlp_fused_heads_supported)
int launch_head_train_kernel(dppo_ctx* ctx, const HeadTrainArgs& a, int continuous, int blocks, cudaStream_t st);
int launch_head_eval(dppo_ctx* ctx, const float* ha, const float* hc, int ld, const float* wa, const float* ba, const float* wc,
                     const float* bc, float* head_out, float* values, int64_t rows, int H, int A, int rev, cudaStream_t st);
// launch_head_eval where it accepts the shape (A <= 32, H <= 512), else the actor product as a GEMM and critic_value_kernel
int launch_heads_forward(dppo_ctx* ctx, const float* ha, const float* hc, int ld, const float* wa, const float* ba, const float* wc,
                         const float* bc, float* head_out, float* values, int64_t rows, int H, int A, int rev, cudaStream_t st);

// ---- GEMM-head path (any shape up to DPPO_GEMM_HEADS_MAX_HIDDEN / _ACT) -----------------------------------------------------
// The head products, their backward and the head weight gradients are GEMMs (api.cu); wide_loss_kernel evaluates the distribution,
// the loss and d(loss)/dz of one row per warp (lanes stride over the actions) and, in training, the critic head of the row.
struct WideLossArgs {
    const float* z;           // [M, A] head outputs (logits / means)
    float* dz;                // [M, A] d(loss)/dz; may alias z (each lane reads z[j] before it writes dz[j])
    const float* log_std;     // [A] shared, or [M, ls_stride] per row (standalone loss only)
    int64_t ls_stride;
    float* dls_rows;          // [M, A] per-row d(loss)/d(log_std) when ls_stride != 0
    const float* values;      // standalone: [M] critic outputs
    float* dvalues;           // standalone: [M] d(loss)/d(values)
    const float* h3;          // training: [M, 2H] first-head-layer activations (the critic half is read)
    float* d3;                // training: [M, 2H] the critic half d3[:, H:] is written
    const float *wc, *bc;     // training: critic_head.2
    const int32_t* idx;       // training: minibatch row -> flat sample index (may be null; < 0: padding row)
    const int32_t* actions_i; // discrete: [B]
    const float* actions_f;   // continuous: [B, A]
    const float *old_logp, *adv, *ret;
    const double* adv_stats;  // training: advantage normalisation (adv_norm_consts)
    int64_t adv_count;
    int advantage_norm;
    int64_t M;
    int H, A;
    float clip, vw, beta, inv_m;
    float* partials;          // [blocks, partial_stride], layout wide_offsets(H, A) (standalone: H = 0)
    int partial_stride;
};
// One partial per CTA: [losses 4 (policy, value, entropy, 0) | dbc | dba A | dlog_std A | dWc H | critic db3 H], each block on a
// multiple of 4 floats.  O(A + H) per CTA; dWa is not part of it (a split-K GEMM computes it).
struct WideOffsets { int dbc, dba, dls, dwc, db3, total; };
__host__ __device__ inline WideOffsets wide_offsets(int H, int A)
{
    auto up4 = [](int x) { return (x + 3) / 4 * 4; };
    WideOffsets o;
    o.dbc = 4;
    o.dba = 8;
    o.dls = up4(o.dba + A);
    o.dwc = up4(o.dls + A);
    o.db3 = up4(o.dwc + H);
    o.total = up4(o.db3 + H);
    return o;
}
int wide_loss_blocks(dppo_ctx* ctx, int64_t M, int H, int A);
int launch_wide_loss_train(dppo_ctx* ctx, const WideLossArgs& a, int continuous, int blocks, cudaStream_t st);
