// C-ABI entry points that orchestrate the per-layer kernels: context, parameter layout,
// forward pass (diamond/ppo.py:91-96, 235-238) and one minibatch of the PPO update (ppo.py:258-283).
#include "common.cuh"
#include "heads.cuh"
#include "optim.cuh"
#include "gemm_tc.cuh"

char g_dppo_create_error[512] = "";

extern "C" int dppo_version(void) { return DPPO_VERSION; }

extern "C" const char* dppo_last_error(dppo_ctx* ctx) { return ctx ? ctx->err : g_dppo_create_error; }

extern "C" int dppo_create(dppo_ctx** out, int device)
{
    if (!out) return 1;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        snprintf(g_dppo_create_error, sizeof(g_dppo_create_error),
                 "dppo_create: no CUDA device (%s); libdppo has no CPU fallback", cudaGetErrorString(e));
        return 2;
    }
    if (device < 0 || device >= count) {
        snprintf(g_dppo_create_error, sizeof(g_dppo_create_error), "dppo_create: device %d out of range (%d devices)", device, count);
        return 3;
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        snprintf(g_dppo_create_error, sizeof(g_dppo_create_error), "dppo_create: %s", cudaGetErrorString(e));
        return 4;
    }
    if (prop.major != 10) {
        snprintf(g_dppo_create_error, sizeof(g_dppo_create_error),
                 "dppo_create: device %d is sm_%d%d; libdppo embeds sm_100a code only (B200) and has no fallback", device,
                 prop.major, prop.minor);
        return 5;
    }
    dppo_ctx* c = new dppo_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->err[0] = 0;
    c->use_tensor_cores = 3;
    c->gae_variant = 0;
    c->gae_inputs_settled = 0;
    c->tc_debug = 0;
    c->row_sweep = 31;
    c->tc_prefetch = 0;
    c->draw_base = nullptr;
    c->rows_dev = nullptr;
    c->launch_count = 0;
    c->tm_cache = nullptr;
    c->tm_cache_free = nullptr;
    *out = c;
    return 0;
}

extern "C" int dppo_destroy(dppo_ctx* ctx)
{
    if (ctx && ctx->tm_cache && ctx->tm_cache_free) ctx->tm_cache_free(ctx->tm_cache);
    delete ctx;
    return 0;
}

extern "C" int dppo_set_option(dppo_ctx* ctx, const char* name, int value)
{
    if (!ctx || !name) return 1;
    if (!strcmp(name, "tensor_cores")) { ctx->use_tensor_cores = value != 0 ? 3 : 0; return 0; }
    if (!strcmp(name, "row_sweep")) { ctx->row_sweep = value & 31; return 0; }
    if (!strcmp(name, "tc_prefetch")) { ctx->tc_prefetch = value & 7; return 0; }
    if (!strcmp(name, "gae_variant")) { ctx->gae_variant = value; return 0; }
    if (!strcmp(name, "tc_debug")) {
#ifdef DPPO_TIMING_SWITCHES
        ctx->tc_debug = value;
        return 0;
#else
        DPPO_FAIL(ctx, "dppo_set_option: 'tc_debug' needs a library built with -DDPPO_TIMING_SWITCHES (timing experiments only)");
#endif
    }
    if (!strcmp(name, "gae_inputs_settled")) { ctx->gae_inputs_settled = value < 0 ? 0 : value > 2 ? 2 : value; return 0; }
    DPPO_FAIL(ctx, "dppo_set_option: unknown option '%s'", name);
}

extern "C" int64_t dppo_launch_count(dppo_ctx* ctx) { return ctx ? ctx->launch_count : 0; }

extern "C" int dppo_count_launches(dppo_ctx* ctx, int64_t n)
{
    if (!ctx) return 1;
    ctx->launch_count += n;
    return 0;
}

extern "C" int dppo_device_info(dppo_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor)
{
    if (!ctx) return 1;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    return 0;
}

extern "C" int dppo_mlp_layout_compute(const dppo_mlp_desc* d, dppo_mlp_layout* L)
{
    if (!d || !L || d->obs_dim < 1 || d->hidden < 1 || d->act_dim < 1) return 1;
    const int64_t D = d->obs_dim, H = d->hidden, A = d->act_dim;
    int64_t o = 0;
    auto take = [&](int64_t n) { const int64_t at = o; o += align_up(n, 4); return at; };
    L->w1 = take(H * D); L->b1 = take(H);
    L->w2 = take(H * H); L->b2 = take(H);
    L->w3 = take(2 * H * H); L->b3 = take(2 * H);
    L->wa = take(A * H); L->ba = take(A);
    L->wc = take(H); L->bc = take(1);
    L->log_std = d->continuous ? take(A) : -1;
    L->total = o;
    return 0;
}

namespace {

struct WImages {
    unsigned char *w1f, *w2f, *w3f, *w3b, *w2b;
    int64_t bytes;
};

// hi/lo pre-swizzled weight images for the tensor-core GEMMs (forward: W1, W2, W3; dgrad: W3^T, W2^T)
WImages carve_images(const dppo_mlp_desc* d, char* base)
{
    const int64_t D = d->obs_dim, H = d->hidden;
    WImages w;
    int64_t o = 0;
    auto take = [&](int64_t bytes) { unsigned char* p = reinterpret_cast<unsigned char*>(base + o); o += align_up(bytes, 1024); return p; };
    w.w1f = take(dppo_tc_image_bytes((int)H, (int)D));
    w.w2f = take(dppo_tc_image_bytes((int)H, (int)H));
    w.w3f = take(dppo_tc_image_bytes((int)(2 * H), (int)H));
    w.w3b = take(dppo_tc_image_bytes((int)H, (int)(2 * H)));
    w.w2b = take(dppo_tc_image_bytes((int)H, (int)H));
    w.bytes = o;
    return w;
}

struct TrainWs {
    float *h1, *h2, *h3, *d3, *d2, *d1, *xg;
    float *p3, *p2, *p1, *c2, *c1, *hp;
    int s3, s2, s1, tiles2, tiles1, head_blocks, head_stride;   // head_*: per-CTA partials of the head kernel (GEMM heads: of wide_loss_kernel)
    int t3, t2, t1;          // split counts of the tcgen05 weight-gradient kernels (0: shape unsupported)
    bool multi;              // the three weight gradients run as one balanced launch (t3/t2/t1 then come from the joint plan)
    float *zd, *pa, *ca;     // GEMM heads: head outputs, overwritten by d(loss)/dz [M, A] | dWa split-K partials | actor db3 column sums
    int sa, tiles_a;
    int64_t img_off;
    int64_t bytes;
};

// Carves the training workspace for M rows.  sm_count fixes the split-K / head grid sizes.  gemm_heads: the head stage of
// dppo_mlp_grad_minibatch_gemm_heads (its partials are O(A + H) per CTA instead of the head kernel's O(A * H)).
TrainWs carve_train(const dppo_mlp_desc* d, int64_t M, int sm_count, char* base, bool gemm_heads = false)
{
    dppo_ctx fake = {}; fake.sm_count = sm_count;
    const int64_t D = d->obs_dim, H = d->hidden, A = d->act_dim;
    TrainWs w;
    int64_t o = 0;
    auto take = [&](int64_t floats) { float* p = reinterpret_cast<float*>(base + o); o += align_up(floats * 4, 256); return p; };
    w.h1 = take(M * H); w.h2 = take(M * H); w.h3 = take(M * 2 * H);
    w.d3 = take(M * 2 * H); w.d2 = take(M * H); w.d1 = take(M * H);
    w.xg = take(M * D);
    w.s3 = dppo_wgrad_splits(&fake, M, (int)(2 * H), (int)H);
    w.s2 = dppo_wgrad_splits(&fake, M, (int)H, (int)H);
    w.s1 = dppo_wgrad_splits(&fake, M, (int)H, (int)D);
    w.t3 = dppo_tc2_wgrad_supported(M, (int)(2 * H), (int)H) ? dppo_tc2_wgrad_splits(&fake, M, (int)(2 * H), (int)H) : 0;
    w.t2 = dppo_tc2_wgrad_supported(M, (int)H, (int)H) ? dppo_tc2_wgrad_splits(&fake, M, (int)H, (int)H) : 0;
    w.t1 = dppo_tc2_wgrad_supported(M, (int)H, (int)D) ? dppo_tc2_wgrad_splits(&fake, M, (int)H, (int)D) : 0;
    w.multi = w.t3 > 0 && w.t2 > 0 && w.t1 > 0 && H % 256 == 0;      // all three in one balanced launch
    if (w.multi) {
        const int n1s[3] = {(int)(2 * H), (int)H, (int)H}, n2s[3] = {(int)H, (int)H, (int)D};
        int sp[3];
        dppo_tc2_wgrad_multi_splits(&fake, M, 3, n1s, n2s, sp);
        w.t3 = sp[0]; w.t2 = sp[1]; w.t1 = sp[2];
    }
    auto mx = [](int a, int b) { return a > b ? a : b; };
    w.p3 = take((int64_t)mx(w.s3, w.t3) * 2 * H * H);
    w.p2 = take((int64_t)mx(w.s2, w.t2) * H * H);
    w.p1 = take((int64_t)mx(w.s1, w.t1) * H * D);
    w.tiles2 = dppo_gemm_row_tiles(M, (int)H);
    w.tiles1 = dppo_gemm_row_tiles(M, (int)H);
    const int cparts = mx(dppo_tc3_colsum_rows(&fake, M, (int)H), w.tiles2);
    w.c2 = take((int64_t)cparts * H);
    w.c1 = take((int64_t)cparts * H);
    w.zd = w.pa = w.ca = nullptr;
    w.sa = w.tiles_a = 0;
    if (gemm_heads) {
        w.zd = take(M * A);
        w.sa = dppo_wgrad_splits(&fake, M, (int)A, (int)H);
        w.pa = take((int64_t)w.sa * A * H);
        w.tiles_a = dppo_gemm_row_tiles(M, (int)H);
        w.ca = take((int64_t)w.tiles_a * H);
        w.head_blocks = wide_loss_blocks(&fake, M, (int)H, (int)A);
        w.head_stride = wide_offsets((int)H, (int)A).total;
    } else {
        w.head_blocks = head_train_blocks(&fake, M, (int)H, (int)A);
        w.head_stride = (int)align_up(head_partial_floats((int)H, (int)A), 4);
    }
    w.hp = take((int64_t)w.head_blocks * w.head_stride);
    o = align_up(o, 1024);
    w.img_off = o;
    o += carve_images(d, nullptr).bytes;
    w.bytes = o;
    return w;
}

// Operand format of the forward launches whose A operand is the output of a tanh epilogue (layers 2 and 3): |A| <= 1 + 3e-7 < 4,
// so A * 2^14 cannot leave fp16's range and the fp16-pair GEMM keeps the 3xTF32 accuracy at twice the tensor rate (gemm_tc.cuh).
// Layer 1 (raw observations), the dgrad launches (unbounded loss gradients) and the weight gradients stay on 3xTF32.
// tc_debug bit 2048 forces TF32 here (timing builds only: A/B runs on one box).
int tanh_input_fmt(const dppo_ctx* ctx)
{
    return DPPO_DBG(ctx->tc_debug, 2048) ? DPPO_TC_FMT_TF32 : DPPO_TC_FMT_F16;
}

int current_sm_count()
{
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms > 0 ? sms : 148;
}

}  // namespace

extern "C" int64_t dppo_mlp_workspace_bytes(const dppo_mlp_desc* d, int64_t rows, int training)
{
    if (!d || rows <= 0) return 0;
    const int64_t H = d->hidden;
    if (!training)      // h1 | h2 | h3 | gathered observations (idx != NULL) | weight images
        return align_up(rows * H * 4, 256) * 2 + align_up(rows * 2 * H * 4, 256) + align_up(rows * (int64_t)d->obs_dim * 4, 256) + 1024 +
               carve_images(d, nullptr).bytes;
    // sized for the B200's 148 SMs or the current device, whichever is larger
    int sms = current_sm_count();
    if (sms < 148) sms = 148;
    return carve_train(d, rows, sms, nullptr).bytes;
}

extern "C" int dppo_mlp_fused_heads_supported(const dppo_mlp_desc* d)
{
    return d && head_train_supported(d->hidden, d->act_dim) ? 1 : 0;
}

static bool gemm_heads_in_bound(const dppo_mlp_desc* d)
{
    return d->hidden >= 1 && d->hidden <= DPPO_GEMM_HEADS_MAX_HIDDEN && d->act_dim >= 1 && d->act_dim <= DPPO_GEMM_HEADS_MAX_ACT;
}

extern "C" int64_t dppo_mlp_gemm_heads_workspace_bytes(const dppo_mlp_desc* d, int64_t rows)
{
    if (!d || rows <= 0 || d->obs_dim < 1 || !gemm_heads_in_bound(d)) return 0;
    int sms = current_sm_count();
    if (sms < 148) sms = 148;
    return carve_train(d, rows, sms, nullptr, true).bytes;
}

extern "C" int dppo_mlp_forward(dppo_ctx* ctx, const dppo_mlp_desc* d, const float* params, const float* obs,
                                const int32_t* idx, int64_t rows, int heads, float* head_out, float* values, void* ws,
                                int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (!d || !params || !obs || rows <= 0) DPPO_FAIL(ctx, "mlp_forward: bad arguments");
    if ((heads & 3) == 0) DPPO_FAIL(ctx, "mlp_forward: heads mask selects nothing");
    if ((heads & 1) && !head_out) DPPO_FAIL(ctx, "mlp_forward: head_out is null");
    if ((heads & 2) && !values) DPPO_FAIL(ctx, "mlp_forward: values is null");
    dppo_mlp_layout L;
    if (dppo_mlp_layout_compute(d, &L)) DPPO_FAIL(ctx, "mlp_forward: bad descriptor");
    const int D = d->obs_dim, H = d->hidden, A = d->act_dim;
    cudaStream_t st = (cudaStream_t)stream;
    // weight images (tensor-core path) sit at the front of the workspace; the rest is chunked over rows
    const int64_t img_bytes = align_up(carve_images(d, nullptr).bytes, 1024);
    char* base0 = (char*)ws;
    char* aligned = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(base0) + 1023) & ~(uintptr_t)1023);
    const int64_t head_room = (aligned - base0) + img_bytes;
    const bool tc_on = ctx->use_tensor_cores && ws_bytes > head_room + 3 * 256;
    WImages img = carve_images(d, aligned);
    char* base = tc_on ? aligned + img_bytes : base0;
    const int64_t avail = tc_on ? ws_bytes - head_room : ws_bytes;
    // chunk the rows so that h1 | h2 | h3 (| gathered observations) fit the workspace
    const int64_t per_row = (int64_t)4 * H * 4 + (idx ? (int64_t)D * 4 : 0);
    int64_t chunk = (avail - 4 * 256) / per_row;
    if (chunk > rows) chunk = rows;
    if (chunk < 1) DPPO_FAIL(ctx, "mlp_forward: workspace too small (%lld bytes, need >= %lld per row)", (long long)ws_bytes, (long long)per_row);
    float* h1 = (float*)base;
    float* h2 = (float*)(base + align_up(chunk * H * 4, 256));
    float* h3 = (float*)(base + 2 * align_up(chunk * H * 4, 256));
    float* xg = (float*)(base + 2 * align_up(chunk * H * 4, 256) + align_up(chunk * 2 * H * 4, 256));
    const bool actor = heads & 1, critic = heads & 2;
    const int sweep = ctx->row_sweep;                  // alternating row sweeps along the layer chain (dppo_tc3_gemm)
    const int hint = (sweep & 8) ? 2 : 0;              // inputs read with the L2 evict-first hint
    const int64_t w3off = actor ? 0 : (int64_t)H * H;
    const int b3off = actor ? 0 : H;
    const int n3 = (actor && critic) ? 2 * H : H;
    // the tensor-core path is decided once from the first (largest) chunk; a smaller tail chunk takes the FFMA kernels
    const int64_t first = rows < chunk ? rows : chunk;
    const bool tc1 = tc_on && dppo_tc3_gemm_supported(first, H, D), tc2 = tc_on && dppo_tc3_gemm_supported(first, H, H),
               tc3 = tc_on && dppo_tc3_gemm_supported(first, n3, H);
    const int hfmt = tanh_input_fmt(ctx);              // layers 2 and 3: A = h1, h2 are tanh outputs
    {
        PrepJobs jobs;
        jobs.n = 0;
        jobs.gather = GatherJob{nullptr, nullptr, nullptr, 0, 0};
        auto job = [&](bool on, const float* W, int rows_w, int cols_w, int fmt, unsigned char* im) {
            if (on) { jobs.job[jobs.n].W = W; jobs.job[jobs.n].rows_w = rows_w; jobs.job[jobs.n].cols_w = cols_w;
                      jobs.job[jobs.n].transpose = 0; jobs.job[jobs.n].n_tile = 0; jobs.job[jobs.n].f16 = fmt == DPPO_TC_FMT_F16;
                      jobs.job[jobs.n].img = im; ++jobs.n; }
        };
        job(tc1, params + L.w1, H, D, DPPO_TC_FMT_TF32, img.w1f);
        job(tc2, params + L.w2, H, H, hfmt, img.w2f);
        job(tc3, params + L.w3 + w3off, n3, H, hfmt, img.w3f);
        if (dppo_tc_prep_weights_multi(ctx, jobs, st)) return 1;
    }
    for (int64_t r0 = 0; r0 < rows; r0 += chunk) {
        const int64_t n = rows - r0 < chunk ? rows - r0 : chunk;
        const float* x = idx ? obs : obs + r0 * D;
        const int32_t* rowsel = idx ? idx + r0 : nullptr;
        if (tc1 && dppo_tc3_gemm_supported(n, H, D)) {
            if (rowsel) {       // the TMA-fed GEMM reads contiguous rows: gather this chunk's observations first
                if (dppo_gather_rows_f32(ctx, obs, rowsel, xg, n, D, stream)) return 1;
                x = xg;
            }
            if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, x, D, img.w1f, params + L.b1, nullptr, 0, h1, H, nullptr, n, H, D, hint, st)) return 1;
        } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, x, D, rowsel, params + L.w1, D, params + L.b1, h1, H, n, H, D, st)) return 1;
        if (tc2 && dppo_tc3_gemm_supported(n, H, H)) {
            if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, h1, H, img.w2f, params + L.b2, nullptr, 0, h2, H, nullptr, n, H, H, (sweep & 1) | hint, st, hfmt)) return 1;
        } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, h1, H, nullptr, params + L.w2, H, params + L.b2, h2, H, n, H, H, st)) return 1;
        // first head layers: both (one [2H,H] product) or only the requested half
        if (tc3 && dppo_tc3_gemm_supported(n, n3, H)) {
            if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, h2, H, img.w3f, params + L.b3 + b3off, nullptr, 0, h3, n3, nullptr, n, n3, H, hint, st, hfmt)) return 1;
        } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, h2, H, nullptr, params + L.w3 + w3off, H, params + L.b3 + b3off, h3, n3, n, n3, H, st)) return 1;
        const float* ha = actor ? h3 : nullptr;
        const float* hc = critic ? (actor ? h3 + H : h3) : nullptr;
        if (launch_heads_forward(ctx, ha, hc, n3, params + L.wa, params + L.ba, params + L.wc, params + L.bc,
                                 head_out ? head_out + r0 * A : nullptr, values ? values + r0 : nullptr, n, H, A, (sweep >> 1) & 1, st)) return 1;
    }
    return 0;
}

// One minibatch gradient (ppo.py:258-283).  The trunk (gather, forward GEMMs, dgrad chain, weight gradients, gradient assembly) is
// shared; gemm_heads selects the head stage: the fused head kernel (head_train_kernel, A <= 32 and (A+1) H within its shared
// memory) or GEMM heads (actor products and head weight gradients as GEMMs around wide_loss_kernel).
static int mlp_grad_minibatch_impl(dppo_ctx* ctx, const char* what, bool gemm_heads, const dppo_mlp_desc* d, const float* params,
                                   float* grads, const float* obs, const void* actions, const float* old_log_probs, const float* adv,
                                   const float* returns, const double* adv_stats, const int32_t* idx, int64_t M, const dppo_hyper* hy,
                                   float* losses, void* ws, int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (!d || !params || !grads || !obs || !actions || !old_log_probs || !adv || !returns || !hy || !ws)
        DPPO_FAIL(ctx, "%s: null argument", what);
    if (M <= 0) DPPO_FAIL(ctx, "%s: empty minibatch", what);
    if (hy->advantage_norm && (!adv_stats || hy->adv_count < 2)) DPPO_FAIL(ctx, "%s: advantage_norm needs adv_stats and adv_count >= 2", what);
    dppo_mlp_layout L;
    if (dppo_mlp_layout_compute(d, &L)) DPPO_FAIL(ctx, "%s: bad descriptor", what);
    if (gemm_heads && !gemm_heads_in_bound(d))
        DPPO_FAIL(ctx, "%s: hidden %d / %d actions outside the GEMM-head bound (hidden <= %d, 1..%d actions)", what, d->hidden, d->act_dim,
                  DPPO_GEMM_HEADS_MAX_HIDDEN, DPPO_GEMM_HEADS_MAX_ACT);
    const int D = d->obs_dim, H = d->hidden, A = d->act_dim;
    TrainWs w = carve_train(d, M, ctx->sm_count, (char*)ws, gemm_heads);
    if (w.bytes > ws_bytes) DPPO_FAIL(ctx, "%s: workspace too small (%lld < %lld)", what, (long long)ws_bytes, (long long)w.bytes);
    cudaStream_t st = (cudaStream_t)stream;
    const float inv_m = 1.0f / (float)(hy->loss_denominator > 0 ? hy->loss_denominator : M);

    // tensor-core path: split/swizzle the current weights once per optimiser step
    char* img_base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>((char*)ws + w.img_off) + 1023) & ~(uintptr_t)1023);
    const bool img_fits = (img_base - (char*)ws) + carve_images(d, nullptr).bytes <= ws_bytes;
    const bool tc_on = ctx->use_tensor_cores && img_fits;
    WImages img = carve_images(d, img_base);
    const bool g1 = tc_on && dppo_tc3_gemm_supported(M, H, D), g2 = tc_on && dppo_tc3_gemm_supported(M, H, H),
               g3 = tc_on && dppo_tc3_gemm_supported(M, 2 * H, H), gb3 = tc_on && dppo_tc3_gemm_supported(M, H, 2 * H), gb2 = g2;
    const bool wg3 = tc_on && w.t3 > 0, wg2 = tc_on && w.t2 > 0, wg1 = tc_on && w.t1 > 0;
    const int hfmt = tanh_input_fmt(ctx);              // forward layers 2 and 3: A = h1, h2 are tanh outputs
    // Row sweeps along the chain (dppo_tc3_gemm): L1 up, L2 down, L3 up, head kernel down, dgrad3 up, dgrad2 down -- every launch
    // starts with the rows its predecessor wrote last (still in the L2).
    const int sweep = ctx->row_sweep;
    const int hint = (sweep & 8) ? 2 : 0;              // inputs read with the L2 evict-first hint (not dgrad2: the weight-gradient launch
                                                       // right behind it reads the same d2 / h1 again)
    // the TMA-fed kernels read contiguous rows: gather the minibatch observations once (ppo.py:261 observations[mb])
    const float* x1 = obs;
    const int32_t* x1_idx = idx;
    bool gather_pending = idx && (g1 || wg1);
    if (gather_pending) { x1 = w.xg; x1_idx = nullptr; }
    {
        // one launch: the hi/lo weight images of this step + the observation gather
        PrepJobs jobs;
        jobs.n = 0;
        jobs.gather = GatherJob{nullptr, nullptr, nullptr, 0, 0};
        auto job = [&](bool on, const float* W, int rows_w, int cols_w, int transpose, int fmt, unsigned char* im) {
            if (on) { jobs.job[jobs.n].W = W; jobs.job[jobs.n].rows_w = rows_w; jobs.job[jobs.n].cols_w = cols_w;
                      jobs.job[jobs.n].transpose = transpose; jobs.job[jobs.n].n_tile = 0; jobs.job[jobs.n].f16 = fmt == DPPO_TC_FMT_F16;
                      jobs.job[jobs.n].img = im; ++jobs.n; }
        };
        job(g1, params + L.w1, H, D, 0, DPPO_TC_FMT_TF32, img.w1f);
        job(g2, params + L.w2, H, H, 0, hfmt, img.w2f);
        job(g3, params + L.w3, 2 * H, H, 0, hfmt, img.w3f);
        job(gb3, params + L.w3, 2 * H, H, 1, DPPO_TC_FMT_TF32, img.w3b);
        job(gb2, params + L.w2, H, H, 1, DPPO_TC_FMT_TF32, img.w2b);
        if (gather_pending && D % 4 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15u) == 0 && (reinterpret_cast<uintptr_t>(w.xg) & 15u) == 0) {
            jobs.gather = GatherJob{reinterpret_cast<const float4*>(obs), idx, reinterpret_cast<float4*>(w.xg), M, D / 4};
            gather_pending = false;
        }
        if (dppo_tc_prep_weights_multi(ctx, jobs, st)) return 1;
    }
    if (gather_pending && dppo_gather_rows_f32(ctx, obs, idx, w.xg, M, D, stream)) return 1;

    // forward (ppo.py:261), activations kept for the backward pass
    if (g1) {
        if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, x1, D, img.w1f, params + L.b1, nullptr, 0, w.h1, H, nullptr, M, H, D, hint, st)) return 1;
    } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, x1, D, x1_idx, params + L.w1, D, params + L.b1, w.h1, H, M, H, D, st)) return 1;
    if (g2) {
        if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, w.h1, H, img.w2f, params + L.b2, nullptr, 0, w.h2, H, nullptr, M, H, H, (sweep & 1) | hint, st, hfmt)) return 1;
    } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.h1, H, nullptr, params + L.w2, H, params + L.b2, w.h2, H, M, H, H, st)) return 1;
    if (g3) {
        if (dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, w.h2, H, img.w3f, params + L.b3, nullptr, 0, w.h3, 2 * H, nullptr, M, 2 * H, H, hint, st, hfmt)) return 1;
    } else if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.h2, H, nullptr, params + L.w3, H, params + L.b3, w.h3, 2 * H, M, 2 * H, H, st)) return 1;

    // heads + loss (ppo.py:264-280) + backward into the first head layers
    if (!gemm_heads) {
        HeadTrainArgs ha;
        ha.h3 = w.h3; ha.d3 = w.d3;
        ha.wa = params + L.wa; ha.ba = params + L.ba; ha.wc = params + L.wc; ha.bc = params + L.bc;
        ha.log_std = d->continuous ? params + L.log_std : nullptr;
        ha.idx = idx;
        ha.actions_i = d->continuous ? nullptr : (const int32_t*)actions;
        ha.actions_f = d->continuous ? (const float*)actions : nullptr;
        ha.old_logp = old_log_probs; ha.adv = adv; ha.ret = returns;
        ha.adv_stats = adv_stats; ha.adv_count = hy->adv_count; ha.advantage_norm = hy->advantage_norm;
        ha.M = M; ha.H = H; ha.A = A;
        ha.clip = hy->ppo_clip; ha.vw = hy->value_loss_weight; ha.beta = hy->entropy_beta; ha.inv_m = inv_m;
        ha.partials = w.hp; ha.partial_stride = w.head_stride;
        ha.rev = (sweep >> 1) & 1; ha.keep_d3 = (sweep >> 2) & 1; ha.h3_first = (sweep >> 3) & 1;
        if (launch_head_train_kernel(ctx, ha, d->continuous, w.head_blocks, st)) return 1;
    } else {
        // z = h3a Wa^T + ba (ppo.py:63-71)
        if (dppo_gemm_nt(ctx, DPPO_EPI_BIAS, w.h3, 2 * H, nullptr, params + L.wa, H, params + L.ba, w.zd, A, M, A, H, st)) return 1;
        // distribution + loss -> dz (in place), critic head -> d3[:, H:], small per-CTA partials
        WideLossArgs la = {};
        la.z = w.zd; la.dz = w.zd;
        la.log_std = d->continuous ? params + L.log_std : nullptr;
        la.h3 = w.h3; la.d3 = w.d3; la.wc = params + L.wc; la.bc = params + L.bc;
        la.idx = idx;
        la.actions_i = d->continuous ? nullptr : (const int32_t*)actions;
        la.actions_f = d->continuous ? (const float*)actions : nullptr;
        la.old_logp = old_log_probs; la.adv = adv; la.ret = returns;
        la.adv_stats = adv_stats; la.adv_count = hy->adv_count; la.advantage_norm = hy->advantage_norm;
        la.M = M; la.H = H; la.A = A;
        la.clip = hy->ppo_clip; la.vw = hy->value_loss_weight; la.beta = hy->entropy_beta; la.inv_m = inv_m;
        la.partials = w.hp; la.partial_stride = w.head_stride;
        if (launch_wide_loss_train(ctx, la, d->continuous, w.head_blocks, st)) return 1;
        // d3[:, :H] = (dz Wa) .* (1 - h3a^2) with the actor db3 column sums; dWa = dz^T h3a as split-K partials
        if (dppo_gemm_nn_tanh_bwd(ctx, w.zd, A, params + L.wa, H, w.h3, 2 * H, w.d3, 2 * H, w.ca, M, H, A, st)) return 1;
        if (dppo_wgrad(ctx, w.zd, A, w.h3, 2 * H, nullptr, w.pa, w.sa, M, A, H, st)) return 1;
    }

    // backward (ppo.py:283): dgrad chain with the tanh' factors and bias-gradient column sums fused
    int tiles2 = w.tiles2, tiles1 = w.tiles1;
    if (gb3) {
        tiles2 = dppo_tc3_colsum_parts(ctx, M, H);
        if (dppo_tc3_gemm(ctx, DPPO_EPI_TANH_BWD, w.d3, 2 * H, img.w3b, nullptr, w.h2, H, w.d2, H, w.c2, M, H, 2 * H, hint, st)) return 1;
    } else if (dppo_gemm_nn_tanh_bwd(ctx, w.d3, 2 * H, params + L.w3, H, w.h2, H, w.d2, H, w.c2, M, H, 2 * H, st)) return 1;
    if (gb2) {
        tiles1 = dppo_tc3_colsum_parts(ctx, M, H);
        if (dppo_tc3_gemm(ctx, DPPO_EPI_TANH_BWD, w.d2, H, img.w2b, nullptr, w.h1, H, w.d1, H, w.c1, M, H, H, sweep & 1, st)) return 1;
    } else if (dppo_gemm_nn_tanh_bwd(ctx, w.d2, H, params + L.w2, H, w.h1, H, w.d1, H, w.c1, M, H, H, st)) return 1;
    // weight gradients: deterministic split-K partials
    const int n3p = wg3 ? w.t3 : w.s3, n2p = wg2 ? w.t2 : w.s2, n1p = wg1 ? w.t1 : w.s1;
    if (w.multi && wg3 && wg2 && wg1) {
        const float* Ds[3] = {w.d3, w.d2, w.d1};
        const float* Hs[3] = {w.h2, w.h1, x1};
        float* Ps[3] = {w.p3, w.p2, w.p1};
        const int ldds[3] = {2 * H, H, H}, ldhs[3] = {H, H, D}, sps[3] = {w.t3, w.t2, w.t1}, n1s[3] = {2 * H, H, H}, n2s[3] = {H, H, D};
        if (dppo_tc2_wgrad_multi(ctx, 3, Ds, ldds, Hs, ldhs, Ps, sps, M, n1s, n2s, st)) return 1;
    } else {
    if (wg3) {
        if (dppo_tc2_wgrad(ctx, w.d3, 2 * H, w.h2, H, w.p3, w.t3, M, 2 * H, H, st)) return 1;
    } else if (dppo_wgrad(ctx, w.d3, 2 * H, w.h2, H, nullptr, w.p3, w.s3, M, 2 * H, H, st)) return 1;
    if (wg2) {
        if (dppo_tc2_wgrad(ctx, w.d2, H, w.h1, H, w.p2, w.t2, M, H, H, st)) return 1;
    } else if (dppo_wgrad(ctx, w.d2, H, w.h1, H, nullptr, w.p2, w.s2, M, H, H, st)) return 1;
    if (wg1) {
        if (dppo_tc2_wgrad(ctx, w.d1, H, x1, D, w.p1, w.t1, M, H, D, st)) return 1;
    } else if (dppo_wgrad(ctx, w.d1, H, x1, D, x1_idx, w.p1, w.s1, M, H, D, st)) return 1;
    }

    // assemble the flat gradient
    GradSegTable tab;
    int n = 0;
    auto seg = [&](int64_t dst, int64_t count, const float* src, int64_t stride, int nparts) {
        tab.seg[n].dst = dst; tab.seg[n].count = count; tab.seg[n].src = src; tab.seg[n].stride = stride;
        tab.seg[n].nparts = nparts; tab.seg[n].pad = 0; ++n;
    };
    seg(L.w1, (int64_t)H * D, w.p1, (int64_t)H * D, n1p);
    seg(L.b1, H, w.c1, H, tiles1);
    seg(L.w2, (int64_t)H * H, w.p2, (int64_t)H * H, n2p);
    seg(L.b2, H, w.c2, H, tiles2);
    seg(L.w3, (int64_t)2 * H * H, w.p3, (int64_t)2 * H * H, n3p);
    int off_dba, off_dwc, off_dbc, off_dls, off_loss;
    if (!gemm_heads) {
        const HeadOffsets ho = head_offsets(H, A);
        off_dba = ho.dba; off_dwc = ho.dwc; off_dbc = ho.dbc; off_dls = ho.dls; off_loss = ho.loss;
        seg(L.b3, 2 * H, w.hp + ho.b3, w.head_stride, w.head_blocks);
        seg(L.wa, (int64_t)A * H, w.hp, w.head_stride, w.head_blocks);
    } else {
        const WideOffsets wo = wide_offsets(H, A);
        off_dba = wo.dba; off_dwc = wo.dwc; off_dbc = wo.dbc; off_dls = wo.dls; off_loss = 0;
        seg(L.b3, H, w.ca, H, w.tiles_a);                                   // actor half: column sums of the dgrad GEMM
        seg(L.b3 + H, H, w.hp + wo.db3, w.head_stride, w.head_blocks);      // critic half: wide_loss_kernel
        seg(L.wa, (int64_t)A * H, w.pa, (int64_t)A * H, w.sa);
    }
    seg(L.ba, A, w.hp + off_dba, w.head_stride, w.head_blocks);
    seg(L.wc, H, w.hp + off_dwc, w.head_stride, w.head_blocks);
    seg(L.bc, 1, w.hp + off_dbc, w.head_stride, w.head_blocks);
    if (d->continuous) seg(L.log_std, A, w.hp + off_dls, w.head_stride, w.head_blocks);
    tab.nseg = n;
    return launch_grad_reduce(ctx, tab, grads, L.total, w.hp + off_loss, w.head_blocks, w.head_stride, hy->value_loss_weight,
                              hy->entropy_beta, inv_m, losses, hy->grad_sumsq, st);
}

extern "C" int dppo_mlp_grad_minibatch(dppo_ctx* ctx, const dppo_mlp_desc* d, const float* params, float* grads,
                                       const float* obs, const void* actions, const float* old_log_probs, const float* adv,
                                       const float* returns, const double* adv_stats, const int32_t* idx, int64_t M,
                                       const dppo_hyper* hy, float* losses, void* ws, int64_t ws_bytes, void* stream)
{
    return mlp_grad_minibatch_impl(ctx, "mlp_grad_minibatch", false, d, params, grads, obs, actions, old_log_probs, adv, returns,
                                   adv_stats, idx, M, hy, losses, ws, ws_bytes, stream);
}

extern "C" int dppo_mlp_grad_minibatch_gemm_heads(dppo_ctx* ctx, const dppo_mlp_desc* d, const float* params, float* grads,
                                                  const float* obs, const void* actions, const float* old_log_probs, const float* adv,
                                                  const float* returns, const double* adv_stats, const int32_t* idx, int64_t M,
                                                  const dppo_hyper* hy, float* losses, void* ws, int64_t ws_bytes, void* stream)
{
    return mlp_grad_minibatch_impl(ctx, "mlp_grad_minibatch_gemm_heads", true, d, params, grads, obs, actions, old_log_probs, adv,
                                   returns, adv_stats, idx, M, hy, losses, ws, ws_bytes, stream);
}

// ---- V(final observation) only where it is needed (SURVEY.md 8f-2), shapes decided on the device --------------------
namespace {

// next_values[t] = values[t+1] wherever the environment did not finish at step t (then next_obs[t] IS obs[t+1] and the rollout
// already recorded its value); the flat indices of all other (t, env) -- finished steps and the last row -- are appended to idx
// (order irrelevant: every entry is scattered back to its own index) and counted in *count.
__global__ void __launch_bounds__(256)
next_value_plan_kernel(const float* __restrict__ terms, const float* __restrict__ truncs, const float* __restrict__ values, int T, int N,
                       float* __restrict__ next_values, int32_t* __restrict__ idx, int* __restrict__ count)
{
    const int64_t B = (int64_t)T * N;
    const int lane = threadIdx.x & 31;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < B; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + threadIdx.x;
        bool need = false;
        if (i < B) {
            need = i >= B - N || terms[i] != 0.0f || truncs[i] != 0.0f;
            if (!need) next_values[i] = values[i + N];
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, need);
        int start = 0;
        if (lane == 0 && ballot) start = atomicAdd(count, __popc(ballot));
        start = __shfl_sync(0xffffffffu, start, 0);
        if (need) idx[start + __popc(ballot & ((1u << lane) - 1u))] = (int32_t)i;
    }
}

__global__ void __launch_bounds__(256)
scatter_values_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, const int* __restrict__ count, float* __restrict__ dst)
{
    const int n = *count;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[idx[i]] = src[i];
}

struct NextWs { int* count; int32_t* idx; float *xg, *h1, *h2, *h3, *tmp; int64_t img_off, bytes; };

NextWs carve_next(const dppo_mlp_desc* d, int64_t B, char* base)
{
    NextWs w;
    int64_t o = 0;
    auto take = [&](int64_t bytes) { char* p = base + o; o += align_up(bytes, 256); return p; };
    w.count = reinterpret_cast<int*>(take(256));
    w.idx = reinterpret_cast<int32_t*>(take(B * 4));
    w.xg = reinterpret_cast<float*>(take(B * d->obs_dim * 4));
    w.h1 = reinterpret_cast<float*>(take(B * d->hidden * 4));
    w.h2 = reinterpret_cast<float*>(take(B * d->hidden * 4));
    w.h3 = reinterpret_cast<float*>(take(B * d->hidden * 4));
    w.tmp = reinterpret_cast<float*>(take(B * 4));
    o = align_up(o, 1024);
    w.img_off = o;
    o += carve_images(d, nullptr).bytes + 1024;
    w.bytes = o;
    return w;
}

}  // namespace

extern "C" int64_t dppo_mlp_next_values_workspace_bytes(const dppo_mlp_desc* d, int T, int N)
{
    if (!d || T < 1 || N < 1) return 0;
    return carve_next(d, (int64_t)T * N, nullptr).bytes + 256;
}

extern "C" int dppo_mlp_next_values(dppo_ctx* ctx, const dppo_mlp_desc* d, const float* params, const float* next_obs,
                                    const float* terminations, const float* truncations, const float* values, int T, int N,
                                    float* next_values, void* ws, int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (!d || !params || !next_obs || !terminations || !truncations || !values || !next_values || !ws || T < 1 || N < 1)
        DPPO_FAIL(ctx, "mlp_next_values: bad arguments");
    dppo_mlp_layout L;
    if (dppo_mlp_layout_compute(d, &L)) DPPO_FAIL(ctx, "mlp_next_values: bad descriptor");
    const int D = d->obs_dim, H = d->hidden;
    const int64_t B = (int64_t)T * N;
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    NextWs w = carve_next(d, B, base);
    if ((base - (char*)ws) + w.bytes > ws_bytes) DPPO_FAIL(ctx, "mlp_next_values: workspace too small (%lld < %lld)", (long long)ws_bytes, (long long)w.bytes);
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(w.count, 0, sizeof(int), st) != cudaSuccess) DPPO_FAIL(ctx, "mlp_next_values: memset failed");
    int blocks = (int)((B + 255) / 256);
    if (blocks > 8 * ctx->sm_count) blocks = 8 * ctx->sm_count;
    next_value_plan_kernel<<<blocks, 256, 0, st>>>(terminations, truncations, values, T, N, next_values, w.idx, w.count);
    DPPO_CHECK_LAUNCH(ctx, "next_value_plan_kernel");

    // critic of the listed rows: every launch below has the fixed shape of B rows and reads the true row count on the device
    char* img_base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(base + w.img_off) + 1023) & ~(uintptr_t)1023);
    WImages img = carve_images(d, img_base);
    const bool tc_on = ctx->use_tensor_cores != 0;
    const bool tc1 = tc_on && dppo_tc3_gemm_supported(B, H, D), tc2 = tc_on && dppo_tc3_gemm_supported(B, H, H);
    const int hfmt = tanh_input_fmt(ctx);              // layer 2 and the critic layer 3: A = h1, h2 are tanh outputs
    {
        PrepJobs jobs;
        jobs.n = 0;
        jobs.gather = GatherJob{nullptr, nullptr, nullptr, 0, 0};
        auto job = [&](bool on, const float* W, int rows_w, int cols_w, int fmt, unsigned char* im) {
            if (on) { jobs.job[jobs.n].W = W; jobs.job[jobs.n].rows_w = rows_w; jobs.job[jobs.n].cols_w = cols_w;
                      jobs.job[jobs.n].transpose = 0; jobs.job[jobs.n].n_tile = 0; jobs.job[jobs.n].f16 = fmt == DPPO_TC_FMT_F16;
                      jobs.job[jobs.n].img = im; ++jobs.n; }
        };
        job(tc1, params + L.w1, H, D, DPPO_TC_FMT_TF32, img.w1f);
        job(tc2, params + L.w2, H, H, hfmt, img.w2f);
        job(tc2, params + L.w3 + (int64_t)H * H, H, H, hfmt, img.w3f);          // critic_head.0
        if (dppo_tc_prep_weights_multi(ctx, jobs, st)) return 1;
    }
    ctx->rows_dev = w.count;
    int rc = dppo_gather_rows_f32(ctx, next_obs, w.idx, w.xg, B, D, stream);
    if (!rc) rc = tc1 ? dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, w.xg, D, img.w1f, params + L.b1, nullptr, 0, w.h1, H, nullptr, B, H, D, 0, st)
                      : dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.xg, D, nullptr, params + L.w1, D, params + L.b1, w.h1, H, B, H, D, st);
    if (!rc) rc = tc2 ? dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, w.h1, H, img.w2f, params + L.b2, nullptr, 0, w.h2, H, nullptr, B, H, H, 0, st, hfmt)
                      : dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.h1, H, nullptr, params + L.w2, H, params + L.b2, w.h2, H, B, H, H, st);
    if (!rc) rc = tc2 ? dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, w.h2, H, img.w3f, params + L.b3 + H, nullptr, 0, w.h3, H, nullptr, B, H, H, 0, st, hfmt)
                      : dppo_gemm_nt(ctx, DPPO_EPI_BIAS_TANH, w.h2, H, nullptr, params + L.w3 + (int64_t)H * H, H, params + L.b3 + H, w.h3, H, B, H, H, st);
    if (!rc) rc = launch_heads_forward(ctx, nullptr, w.h3, H, params + L.wa, params + L.ba, params + L.wc, params + L.bc, nullptr, w.tmp, B, H,
                                       d->act_dim, 0, st);
    ctx->rows_dev = nullptr;
    if (rc) return 1;
    scatter_values_kernel<<<blocks, 256, 0, st>>>(w.tmp, w.idx, w.count, next_values);
    DPPO_CHECK_LAUNCH(ctx, "scatter_values_kernel");
    return 0;
}

// ---- tensor-core building blocks exposed for unit tests and A/B measurements ----------------------
extern "C" int64_t dppo_tc_linear_workspace_bytes(int N, int K) { return dppo_tc_image_bytes(N, K) + 1024; }

extern "C" int dppo_tc_colsum_parts(dppo_ctx* ctx, int64_t M, int N)
{
    return ctx ? dppo_tc3_colsum_rows(ctx, M, N) : 0;
}

extern "C" int dppo_tc_linear_f32(dppo_ctx* ctx, int epi, const float* A, int64_t M, int K, const float* W, int N, int transpose,
                                  const float* bias, const float* Hact, float* C, float* colsum, void* ws, int64_t ws_bytes,
                                  int prepared, void* stream)
{
    if (!ctx) return 1;
    if (!A || !W || !C || !ws) DPPO_FAIL(ctx, "tc_linear: null argument");
    if (epi == DPPO_EPI_BIAS_TANH && !bias) DPPO_FAIL(ctx, "tc_linear: bias is null");
    if (epi == DPPO_EPI_TANH_BWD && !Hact) DPPO_FAIL(ctx, "tc_linear: Hact is null");
    unsigned char* img = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~(uintptr_t)1023);
    if ((img - (unsigned char*)ws) + dppo_tc_image_bytes(N, K) > ws_bytes) DPPO_FAIL(ctx, "tc_linear: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int rows_w = transpose ? K : N, cols_w = transpose ? N : K;
    if (!dppo_tc3_gemm_supported(M, N, K)) DPPO_FAIL(ctx, "tc_linear: unsupported shape M=%lld N=%d K=%d", (long long)M, N, K);
    // prepared != 0: the images an earlier call with the same weights left in ws are re-used (kernel-only timing)
    if (!prepared && dppo_tc_prep_weights(ctx, W, rows_w, cols_w, transpose, img, st)) return 1;
    return dppo_tc3_gemm(ctx, epi, A, K, img, bias, Hact, N, C, N, colsum, M, N, K, 0, st);
}

extern "C" int dppo_tc_linear_forward(dppo_ctx* ctx, int fmt, const float* A, int64_t M, int K, const float* W, int N, const float* bias,
                                      float* C, const int* rows_dev, void* ws, int64_t ws_bytes, int prepared, void* stream)
{
    if (!ctx) return 1;
    if (!A || !W || !bias || !C || !ws) DPPO_FAIL(ctx, "tc_linear_forward: null argument");
    if (fmt != DPPO_TC_FMT_TF32 && fmt != DPPO_TC_FMT_F16) DPPO_FAIL(ctx, "tc_linear_forward: unknown operand format %d", fmt);
    if (!dppo_tc3_gemm_supported(M, N, K)) DPPO_FAIL(ctx, "tc_linear_forward: unsupported shape M=%lld N=%d K=%d", (long long)M, N, K);
    unsigned char* img = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~(uintptr_t)1023);
    if ((img - (unsigned char*)ws) + dppo_tc_image_bytes(N, K) > ws_bytes) DPPO_FAIL(ctx, "tc_linear_forward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if (!prepared) {
        PrepJobs jobs;
        jobs.n = 1;
        jobs.job[0] = PrepJob{W, N, K, 0, 0, fmt == DPPO_TC_FMT_F16, img};
        jobs.gather = GatherJob{nullptr, nullptr, nullptr, 0, 0};
        if (dppo_tc_prep_weights_multi(ctx, jobs, st)) return 1;
    }
    ctx->rows_dev = rows_dev;
    const int rc = dppo_tc3_gemm(ctx, DPPO_EPI_BIAS_TANH, A, K, img, bias, nullptr, 0, C, N, nullptr, M, N, K, 0, st, fmt);
    ctx->rows_dev = nullptr;
    return rc;
}

extern "C" int64_t dppo_tc_wgrad_workspace_bytes(dppo_ctx* ctx, int64_t M, int N1, int N2)
{
    if (!ctx || !dppo_tc2_wgrad_supported(M, N1, N2)) return 0;
    return (int64_t)dppo_tc2_wgrad_splits(ctx, M, N1, N2) * N1 * N2 * 4 + 256;
}

extern "C" int dppo_tc_wgrad_f32(dppo_ctx* ctx, const float* Dm, const float* Hm, int64_t M, int N1, int N2, float* dW, void* ws,
                                 int64_t ws_bytes, void* stream)
{
    if (!ctx) return 1;
    if (!Dm || !Hm || !dW || !ws) DPPO_FAIL(ctx, "tc_wgrad: null argument");
    if (!dppo_tc2_wgrad_supported(M, N1, N2)) DPPO_FAIL(ctx, "tc_wgrad: unsupported shape M=%lld N1=%d N2=%d", (long long)M, N1, N2);
    float* parts = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    const int splits = dppo_tc2_wgrad_splits(ctx, M, N1, N2);
    if (((char*)parts - (char*)ws) + (int64_t)splits * N1 * N2 * 4 > ws_bytes) DPPO_FAIL(ctx, "tc_wgrad: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    if (dppo_tc2_wgrad(ctx, Dm, N1, Hm, N2, parts, splits, M, N1, N2, st)) return 1;
    GradSegTable tab;
    tab.seg[0].dst = 0; tab.seg[0].count = (int64_t)N1 * N2; tab.seg[0].src = parts; tab.seg[0].stride = (int64_t)N1 * N2;
    tab.seg[0].nparts = splits; tab.seg[0].pad = 0;
    tab.nseg = 1;
    return launch_grad_reduce(ctx, tab, dW, (int64_t)N1 * N2, nullptr, 0, 0, 0.f, 0.f, 0.f, nullptr, nullptr, st);
}
