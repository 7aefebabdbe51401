// Device-resident vectorised environments (SURVEY.md 8f-1): one kernel per vector step replaces the reference's host
// `envs.step` + masked `envs.reset` + list append (diamond/ppo.py:160-182) and both PCIe crossings of a rollout step.
// The kernel steps every environment, writes the step straight into row t of the rollout buffer with the casts of
// ppo.py:229-232, keeps Gymnasium's autoreset-DISABLED contract (next_obs is the TRUE final observation; environments
// that finished are then reset, and the post-reset observation is what the next sampling step sees, ppo.py:174-179), and
// maintains per-environment episode return / length.
//
// Dynamics follow Gymnasium's classic-control environments (third-party, not in the reference tree; gymnasium >= 1.0.0,
// `classic_control/cartpole.py` CartPole-v1: Euler integrator, tau 0.02, termination |x| > 2.4 or |theta| > 12 deg, 500-step
// time limit; `classic_control/pendulum.py` Pendulum-v1: dt 0.05, g 10, torque clipped to [-2, 2], speed clipped to [-8, 8],
// 200-step time limit, never terminates; `classic_control/acrobot.py` Acrobot-v1: "book" dynamics, one RK4 step of dt 0.2,
// angles wrapped into [-pi, pi], speeds bounded to 4 pi / 9 pi, torque a - 1, 500-step time limit;
// `classic_control/mountain_car.py` MountainCar-v0: force (a - 1) * 0.001, 200-step time limit;
// `classic_control/continuous_mountain_car.py` MountainCarContinuous-v0: 999-step time limit) with the state held in float64
// as Gymnasium does, observations cast to float32.  MountainCarContinuous keeps Gymnasium's float32 state: under NumPy 2's
// promotion rules (NEP 50) its step runs in float32 except cos(3 p) and, for an action outside [-1, 1], the force term,
// which are double; the explicitly rounded intrinsics below keep the compiler from contracting those operations into FMAs.
// The time limit is the repository's convention: truncated = steps >= limit && !terminated.
// The checkers are oracle/env_oracle.py (CartPole, Pendulum) and tests/classic_env_oracle.py (Acrobot, MountainCar,
// MountainCarContinuous); reset draws come from Philox4x32-10 keyed by (seed, global env id, episode index),
// so a run does not depend on launch geometry or GPU count.
#include "common.cuh"

namespace {

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
__device__ __forceinline__ double u01d(uint32_t x) { return ((double)x + 0.5) * (1.0 / 4294967296.0); }      // (0,1)

struct EnvArgs {
    int kind, N, D, A, t, auto_reset;
    double* state;              // [N, 4]  CartPole: x, x_dot, theta, theta_dot; Pendulum: theta, theta_dot; Acrobot: theta1,
                                //         theta2, theta1_dot, theta2_dot; MountainCar(Continuous): position, velocity; synthetic: unused
    int32_t* steps;             // [N] steps taken in the current episode
    int64_t* episode;           // [N] episodes started so far (reset draw index)
    double* ep_return;          // [N] running return
    const void* actions;        // int64 [N] (discrete) or f32 [N, A]
    float *obs_t, *next_obs_t;  // row t of the rollout buffer: [N, D] each (obs_t may be null)
    void* act_t;                // row t: int32 [N] or f32 [N, A] (may be null)
    float *rew_t, *term_t, *trunc_t;
    float* cur_obs;             // [N, D] observation the next sampling step reads
    float* done_return;         // [N] return of the episode that ended at this step (else untouched), optional
    unsigned long long seed;
    long long env_offset;
    float p_term, p_trunc;      // synthetic env
    // per-environment normalisation (NORM instantiations only; dppo.h dppo_env_desc / dppo_env_state)
    int norm_obs, norm_rew;
    double gamma, eps, clip_obs, clip_rew;
    double *obs_mean, *obs_var;  // [N, D]
    double* obs_count;          // [N]
    double* ret_stats;          // [N, 4]: discounted return accumulator, its running mean, variance, count
    const int32_t* update;      // [1] nonzero: update the statistics (read at run time, so replayed graphs follow it)
    float* raw_rew_t;           // row t of the raw reward buffer (may be null)
};

template <int KIND>
__device__ __forceinline__ void reset_state(const EnvArgs& a, int e, double* s)
{
    const unsigned long long env = (unsigned long long)(a.env_offset + e);
    const unsigned long long ep = (unsigned long long)a.episode[e];
    const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)ep, (uint32_t)(ep >> 32) ^ 0x52534554u),
                                  make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
    if constexpr (KIND == 0) {    // uniform(-0.05, 0.05) x 4
        s[0] = -0.05 + 0.1 * u01d(r.x); s[1] = -0.05 + 0.1 * u01d(r.y); s[2] = -0.05 + 0.1 * u01d(r.z); s[3] = -0.05 + 0.1 * u01d(r.w);
    } else if constexpr (KIND == 1) {   // theta ~ U(-pi, pi), theta_dot ~ U(-1, 1)
        s[0] = -3.14159265358979323846 + 6.28318530717958647692 * u01d(r.x); s[1] = -1.0 + 2.0 * u01d(r.y); s[2] = 0.0; s[3] = 0.0;
    } else if constexpr (KIND == 4) {   // uniform(-0.1, 0.1) x 4 rounded to float32, as Gymnasium's .astype(np.float32)
        s[0] = (float)(-0.1 + 0.2 * u01d(r.x)); s[1] = (float)(-0.1 + 0.2 * u01d(r.y));
        s[2] = (float)(-0.1 + 0.2 * u01d(r.z)); s[3] = (float)(-0.1 + 0.2 * u01d(r.w));
    } else {                            // position ~ U(-0.6, -0.4) (float32 state for the continuous car), velocity 0
        const double p = -0.6 + 0.2 * u01d(r.x);
        s[0] = KIND == 6 ? (double)(float)p : p; s[1] = 0.0; s[2] = 0.0; s[3] = 0.0;
    }
    a.episode[e] += 1;
    a.steps[e] = 0;
}

template <int KIND> constexpr int kObsDim = KIND == 0 ? 4 : KIND == 1 ? 3 : KIND == 4 ? 6 : 2;

template <int KIND>
__device__ __forceinline__ void write_obs(const double* s, float* o)
{
    if constexpr (KIND == 0) { o[0] = (float)s[0]; o[1] = (float)s[1]; o[2] = (float)s[2]; o[3] = (float)s[3]; }
    else if constexpr (KIND == 1) { o[0] = (float)cos(s[0]); o[1] = (float)sin(s[0]); o[2] = (float)s[1]; }
    else if constexpr (KIND == 4) {
        o[0] = (float)cos(s[0]); o[1] = (float)sin(s[0]); o[2] = (float)cos(s[1]); o[3] = (float)sin(s[1]); o[4] = (float)s[2]; o[5] = (float)s[3];
    } else { o[0] = (float)s[0]; o[1] = (float)s[1]; }
}

// Gymnasium's RunningMeanStd.update on a batch of one value x (batch mean x, batch variance 0, batch count 1), in NumPy's operation
// order with every rounding explicit (no contraction):  delta = x - mean;  tot = count + 1;  mean += delta * 1 / tot;
// M2 = var * count + 0 + delta^2 * count * 1 / tot;  var = M2 / tot;  count = tot.  The caller stores count = tot.
__device__ __forceinline__ void rms_update(double& mean, double& var, double count, double x)
{
    const double delta = __dsub_rn(x, mean), tot = __dadd_rn(count, 1.0);
    mean = __dadd_rn(mean, __ddiv_rn(delta, tot));
    var = __ddiv_rn(__dadd_rn(__dmul_rn(var, count), __ddiv_rn(__dmul_rn(__dmul_rn(delta, delta), count), tot)), tot);
}

// NormalizeObservation of one feature: update (unless frozen), then float32((x - mean) / sqrt(var + eps)), clipped in float32
__device__ __forceinline__ float norm_feature(const EnvArgs& a, int64_t i, double count, bool upd, float xf)
{
    double mean = a.obs_mean[i], var = a.obs_var[i];
    if (upd) {
        rms_update(mean, var, count, (double)xf);
        a.obs_mean[i] = mean; a.obs_var[i] = var;
    }
    float y = (float)__ddiv_rn(__dsub_rn((double)xf, mean), __dsqrt_rn(__dadd_rn(var, a.eps)));
    if (a.clip_obs > 0.0) {
        const float c = (float)a.clip_obs;
        y = fminf(fmaxf(y, -c), c);
    }
    return y;
}

// One classic environment's observation of D features through NormalizeObservation (or copied when only rewards are normalised)
template <int D>
__device__ __forceinline__ void norm_obs(const EnvArgs& a, int e, const float* x, float* dst)
{
    if (!a.norm_obs) {
#pragma unroll
        for (int j = 0; j < D; ++j) dst[j] = x[j];
        return;
    }
    const bool upd = *a.update != 0;
    const double count = a.obs_count[e];
#pragma unroll
    for (int j = 0; j < D; ++j) dst[j] = norm_feature(a, (int64_t)e * D + j, count, upd, x[j]);
    if (upd) a.obs_count[e] = __dadd_rn(count, 1.0);
}

// NormalizeReward: acc = acc * gamma * (1 - terminated) + r; update the return statistics with acc (unless frozen);
// emit r / sqrt(var + eps), clipped in double.  The accumulator is cut by termination only, as in Gymnasium.
__device__ __forceinline__ float norm_reward(const EnvArgs& a, int e, double r, bool term)
{
    if (!a.norm_rew) return (float)r;
    double* st = a.ret_stats + (int64_t)e * 4;
    const double acc = __dadd_rn(__dmul_rn(__dmul_rn(st[0], a.gamma), term ? 0.0 : 1.0), r);
    double mean = st[1], var = st[2];
    st[0] = acc;
    if (*a.update != 0) {
        const double count = st[3];
        rms_update(mean, var, count, acc);
        st[1] = mean; st[2] = var; st[3] = __dadd_rn(count, 1.0);
    }
    double y = __ddiv_rn(r, __dsqrt_rn(__dadd_rn(var, a.eps)));
    if (a.clip_rew > 0.0) y = fmin(fmax(y, -a.clip_rew), a.clip_rew);
    return (float)y;
}

// Acrobot-v1 `_dsdt` ("book" dynamics; m1 = m2 = l1 = 1, lc1 = lc2 = 0.5, I1 = I2 = 1, g = 9.8) in Gymnasium's operation order
__device__ __forceinline__ void acrobot_dsdt(const double* y, double torque, double* dy)
{
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8, pi = 3.14159265358979323846;
    const double th1 = y[0], th2 = y[1], dth1 = y[2], dth2 = y[3];
    const double c2 = cos(th2), s2 = sin(th2);
    const double d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2.0 * l1 * lc2 * c2) + I1 + I2;
    const double d2 = m2 * (lc2 * lc2 + l1 * lc2 * c2) + I2;
    const double phi2 = m2 * lc2 * g * cos(th1 + th2 - pi / 2.0);
    const double phi1 = -m2 * l1 * lc2 * (dth2 * dth2) * s2 - 2.0 * m2 * l1 * lc2 * dth2 * dth1 * s2 + (m1 * lc1 + m2 * l1) * g * cos(th1 - pi / 2.0)
                        + phi2;
    const double ddth2 = (torque + d2 / d1 * phi1 - m2 * l1 * lc2 * (dth1 * dth1) * s2 - phi2) / (m2 * (lc2 * lc2) + I2 - d2 * d2 / d1);
    dy[0] = dth1; dy[1] = dth2; dy[2] = -(d2 * ddth2 + phi1) / d1; dy[3] = ddth2;
}

// mode 0: step (t, actions); mode 1: reset the environments with mask[e] != 0 (mask null: all).  NORM: the environment's
// observations and rewards pass through its NormalizeObservation / NormalizeReward statistics (a.norm_obs, a.norm_rew) in this thread;
// the NORM = false instantiations are the kernels without normalisation, unchanged.
template <int KIND, bool NORM>
__global__ void classic_env_kernel(EnvArgs a, int mode, const unsigned char* __restrict__ mask)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.N) return;
    double s[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) s[i] = a.state[(int64_t)e * 4 + i];
    if (mode == 1) {
        if (mask == nullptr || mask[e]) {
            reset_state<KIND>(a, e, s);
            a.ep_return[e] = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) a.state[(int64_t)e * 4 + i] = s[i];
            if constexpr (NORM) {
                float o[6];
                write_obs<KIND>(s, o);
                norm_obs<kObsDim<KIND>>(a, e, o, a.cur_obs + (int64_t)e * a.D);
            } else {
                write_obs<KIND>(s, a.cur_obs + (int64_t)e * a.D);
            }
        }
        return;
    }
    if constexpr (NORM) {                                               // the (normalised) observation the action was sampled from
        if (a.obs_t)
#pragma unroll
            for (int j = 0; j < kObsDim<KIND>; ++j) a.obs_t[(int64_t)e * a.D + j] = a.cur_obs[(int64_t)e * a.D + j];
    } else {
        if (a.obs_t) write_obs<KIND>(s, a.obs_t + (int64_t)e * a.D);
    }
    double reward;
    bool term = false;
    int limit;                                                          // TimeLimit of the registered id
    if constexpr (KIND == 0) {
        const long long act = reinterpret_cast<const long long*>(a.actions)[e];
        if (a.act_t) reinterpret_cast<int32_t*>(a.act_t)[e] = (int32_t)act;
        const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
        const double total_mass = masspole + masscart, pml = masspole * length;
        const double force = act == 1 ? force_mag : -force_mag;
        const double ct = cos(s[2]), st = sin(s[2]);
        const double temp = (force + pml * s[3] * s[3] * st) / total_mass;
        const double th_acc = (gravity * st - ct * temp) / (length * (4.0 / 3.0 - masspole * ct * ct / total_mass));
        const double x_acc = temp - pml * th_acc * ct / total_mass;
        const double x = s[0] + tau * s[1], xd = s[1] + tau * x_acc, th = s[2] + tau * s[3], thd = s[3] + tau * th_acc;
        s[0] = x; s[1] = xd; s[2] = th; s[3] = thd;
        term = fabs(x) > 2.4 || fabs(th) > 12.0 * 2.0 * 3.14159265358979323846 / 360.0;
        reward = 1.0;
        limit = 500;
    } else if constexpr (KIND == 1) {
        const float af = reinterpret_cast<const float*>(a.actions)[(int64_t)e * a.A];
        if (a.act_t) reinterpret_cast<float*>(a.act_t)[(int64_t)e * a.A] = af;
        const double max_speed = 8.0, max_torque = 2.0, dt = 0.05, g = 10.0, m = 1.0, l = 1.0, pi = 3.14159265358979323846;
        const double u = fmin(fmax((double)af, -max_torque), max_torque);
        double thn = fmod(s[0] + pi, 2.0 * pi);
        if (thn < 0.0) thn += 2.0 * pi;                                 // python's % is non-negative
        thn -= pi;
        reward = -(thn * thn + 0.1 * s[1] * s[1] + 0.001 * u * u);
        double thd = s[1] + (3.0 * g / (2.0 * l) * sin(s[0]) + 3.0 / (m * l * l) * u) * dt;
        thd = fmin(fmax(thd, -max_speed), max_speed);
        s[1] = thd;
        s[0] = s[0] + thd * dt;
        limit = 200;
    } else if constexpr (KIND == 4) {                                   // Acrobot-v1
        const long long act = reinterpret_cast<const long long*>(a.actions)[e];
        if (a.act_t) reinterpret_cast<int32_t*>(a.act_t)[e] = (int32_t)act;
        const double torque = (double)(act - 1), dt = 0.2, pi = 3.14159265358979323846;
        double k1[4], k2[4], k3[4], k4[4], y[4];
        acrobot_dsdt(s, torque, k1);                                    // rk4 over [0, dt]: y0 + dt / 6 (k1 + 2 k2 + 2 k3 + k4)
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = s[i] + dt / 2.0 * k1[i];
        acrobot_dsdt(y, torque, k2);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = s[i] + dt / 2.0 * k2[i];
        acrobot_dsdt(y, torque, k3);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = s[i] + dt * k3[i];
        acrobot_dsdt(y, torque, k4);
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] = s[i] + dt / 6.0 * (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]);
#pragma unroll
        for (int i = 0; i < 2; ++i) {                                   // Gymnasium's `wrap` into [-pi, pi]: loops, not fmod
            while (s[i] > pi) s[i] = s[i] - 2.0 * pi;
            while (s[i] < -pi) s[i] = s[i] + 2.0 * pi;
        }
        s[2] = fmin(fmax(s[2], -4.0 * pi), 4.0 * pi);
        s[3] = fmin(fmax(s[3], -9.0 * pi), 9.0 * pi);
        term = -cos(s[0]) - cos(s[1] + s[0]) > 1.0;
        reward = term ? 0.0 : -1.0;
        limit = 500;
    } else if constexpr (KIND == 5) {                                   // MountainCar-v0, float64 (no contraction: numpy has none)
        const long long act = reinterpret_cast<const long long*>(a.actions)[e];
        if (a.act_t) reinterpret_cast<int32_t*>(a.act_t)[e] = (int32_t)act;
        double p = s[0], v = s[1];
        v = __dadd_rn(v, __dadd_rn(__dmul_rn((double)(act - 1), 0.001), __dmul_rn(cos(__dmul_rn(3.0, p)), -0.0025)));
        v = fmin(fmax(v, -0.07), 0.07);
        p = fmin(fmax(__dadd_rn(p, v), -1.2), 0.6);
        if (p == -1.2 && v < 0.0) v = 0.0;
        s[0] = p; s[1] = v;
        term = p >= 0.5 && v >= 0.0;
        reward = -1.0;
        limit = 200;
    } else {                                                            // MountainCarContinuous-v0, float32 state
        const float af = reinterpret_cast<const float*>(a.actions)[(int64_t)e * a.A];
        if (a.act_t) reinterpret_cast<float*>(a.act_t)[(int64_t)e * a.A] = af;
        float p = (float)s[0], v = (float)s[1];
        const double c = cos((double)__fmul_rn(3.0f, p));                // math.cos on the float32 product
        // min(max(action[0], -1.0), 1.0) is the float32 action when in range (float32 multiply), a Python float (double) when not
        const float dv = (af > 1.0f || af < -1.0f) ? (float)__dsub_rn(af > 1.0f ? 0.0015 : -0.0015, __dmul_rn(0.0025, c))
                                                   : __fsub_rn(__fmul_rn(af, 0.0015f), (float)__dmul_rn(0.0025, c));
        v = __fadd_rn(v, dv);
        if (v > 0.07f) v = 0.07f;
        if (v < -0.07f) v = -0.07f;
        p = __fadd_rn(p, v);
        if (p > 0.6f) p = 0.6f;
        if (p < -1.2f) p = -1.2f;
        if (p == -1.2f && v < 0.0f) v = 0.0f;
        s[0] = p; s[1] = v;
        term = p >= 0.45f && v >= 0.0f;
        reward = (term ? 100.0 : 0.0) - __dmul_rn(__dmul_rn((double)af, (double)af), 0.1);
        limit = 999;
    }
    a.steps[e] += 1;
    const bool trunc = a.steps[e] >= limit && !term;
    float fin[6];                                                       // NORM: the normalised final observation
    if constexpr (NORM) {
        float o[6];
        write_obs<KIND>(s, o);
        norm_obs<kObsDim<KIND>>(a, e, o, fin);
#pragma unroll
        for (int j = 0; j < kObsDim<KIND>; ++j) a.next_obs_t[(int64_t)e * a.D + j] = fin[j];
        a.rew_t[e] = norm_reward(a, e, reward, term);
        if (a.raw_rew_t) a.raw_rew_t[e] = (float)reward;
    } else {
        write_obs<KIND>(s, a.next_obs_t + (int64_t)e * a.D);           // the true final observation (autoreset disabled)
        a.rew_t[e] = (float)reward;
    }
    a.term_t[e] = term ? 1.0f : 0.0f;
    a.trunc_t[e] = trunc ? 1.0f : 0.0f;
    const double ret = a.ep_return[e] + reward;
    const bool done = term || trunc;
    if (done && a.done_return) a.done_return[e] = (float)ret;
    if (done && a.auto_reset) {
        reset_state<KIND>(a, e, s);                                     // envs.reset(options={"reset_mask": dones}), ppo.py:174-179
        a.ep_return[e] = 0.0;
    } else {
        a.ep_return[e] = ret;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) a.state[(int64_t)e * 4 + i] = s[i];
    if constexpr (NORM) {
        if (done && a.auto_reset) {                                     // the post-reset observation is counted too
            float o[6];
            write_obs<KIND>(s, o);
            norm_obs<kObsDim<KIND>>(a, e, o, fin);
        }                                                               // else cur_obs is next_obs[t], bit for bit
#pragma unroll
        for (int j = 0; j < kObsDim<KIND>; ++j) a.cur_obs[(int64_t)e * a.D + j] = fin[j];
    } else {
        write_obs<KIND>(s, a.cur_obs + (int64_t)e * a.D);
    }
}

// Synthetic environment of the scale benchmark (shape-only stand-in, diamond/envs.py BatchedSyntheticVectorEnv): i.i.d.
// standard-normal observations, reward = 0.1 * obs[0] * sign(action), Bernoulli terminations / truncations.
// One warp per environment; lanes stride over the observation.  NORM: each lane runs its features' NormalizeObservation
// statistics (the count is shared: every lane reads it, lane 0 advances it once the warp is done), lane 0 runs NormalizeReward, and
// the raw observation's first feature, which the reward reads, is kept in state[e, 0] (unused by the synthetic kinds otherwise).
template <bool NORM>
__global__ void synthetic_env_kernel(EnvArgs a, int mode, const unsigned char* __restrict__ mask)
{
    const int e = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (e >= a.N) return;
    const unsigned long long env = (unsigned long long)(a.env_offset + e);
    bool upd = false;
    if constexpr (NORM) upd = a.norm_obs && *a.update != 0;
    float raw0 = 0.f;                                                   // NORM: lane 0's raw first feature of the last draw
    auto fresh = [&](unsigned long long draw, float* dst0, float* dst1) {       // D normals into up to two destinations
        double count = 0.0;
        if constexpr (NORM) if (a.norm_obs) count = a.obs_count[e];
        for (int j0 = 2 * lane; j0 < a.D; j0 += 64) {
            const unsigned long long c = draw * 4096ull + (unsigned long long)(j0 / 2);
            const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)c, (uint32_t)(c >> 32) ^ 0x4F425321u),
                                          make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
            const float rad = sqrtf(-2.0f * logf((float)u01d(r.x)));
            float sn, cs;
            sincosf(6.28318530717958647692f * (float)u01d(r.y), &sn, &cs);
            float v0 = rad * cs, v1 = rad * sn;
            if constexpr (NORM) {
                if (j0 == 0) raw0 = v0;
                if (a.norm_obs) {
                    v0 = norm_feature(a, (int64_t)e * a.D + j0, count, upd, v0);
                    if (j0 + 1 < a.D) v1 = norm_feature(a, (int64_t)e * a.D + j0 + 1, count, upd, v1);
                }
            }
            if (dst0) { dst0[j0] = v0; if (j0 + 1 < a.D) dst0[j0 + 1] = v1; }
            if (dst1) { dst1[j0] = v0; if (j0 + 1 < a.D) dst1[j0 + 1] = v1; }
        }
        if constexpr (NORM) {
            __syncwarp();
            if (upd && lane == 0) a.obs_count[e] = __dadd_rn(count, 1.0);
            __syncwarp();
        }
    };
    float* cur = a.cur_obs + (int64_t)e * a.D;
    if (mode == 1) {
        if (mask == nullptr || mask[e]) {
            const unsigned long long draw = 2ull * (unsigned long long)a.episode[e] + 1ull;
            fresh((draw << 20), cur, nullptr);
            __syncwarp();
            if (lane == 0) { a.episode[e] += 1; a.steps[e] = 0; a.ep_return[e] = 0.0; }
            if (NORM && lane == 0) a.state[(int64_t)e * 4] = raw0;
        }
        return;
    }
    const float o0 = NORM ? (float)a.state[(int64_t)e * 4] : cur[0];
    __syncwarp();
    if (a.obs_t) for (int j = lane; j < a.D; j += 32) a.obs_t[(int64_t)e * a.D + j] = cur[j];
    float asum;
    if (a.A > 0 && a.kind == 3) {                       // continuous synthetic: sum of the action vector
        asum = 0.f;
        for (int j = 0; j < a.A; ++j) {
            const float v = reinterpret_cast<const float*>(a.actions)[(int64_t)e * a.A + j];
            asum += v;
            if (a.act_t && lane == 0) reinterpret_cast<float*>(a.act_t)[(int64_t)e * a.A + j] = v;
        }
    } else {
        const long long act = reinterpret_cast<const long long*>(a.actions)[e];
        if (a.act_t && lane == 0) reinterpret_cast<int32_t*>(a.act_t)[e] = (int32_t)act;
        asum = (float)act;
    }
    const float reward = o0 * (asum > 0.f ? 1.0f : -1.0f) * 0.1f;
    const unsigned long long step_id = ((unsigned long long)a.episode[e] << 20) + (unsigned long long)a.steps[e];
    __syncwarp();
    // next observation: a fresh draw, written to the buffer's final-observation row and (if the episode continues) cur_obs
    const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)step_id, (uint32_t)(step_id >> 32) ^ 0x444F4E45u),
                                  make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
    const bool term = (float)u01d(r.x) < a.p_term;
    const bool trunc = !term && (float)u01d(r.y) < a.p_trunc;
    const bool done = term || trunc;
    fresh(2ull * step_id + 2ull, a.next_obs_t + (int64_t)e * a.D, (done && a.auto_reset) ? nullptr : cur);
    if (done && a.auto_reset) fresh(((2ull * (unsigned long long)(a.episode[e] + 1) + 1ull) << 20) + 7ull, cur, nullptr);
    __syncwarp();
    if (lane == 0) {
        if constexpr (NORM) {
            a.rew_t[e] = norm_reward(a, e, (double)reward, term);
            if (a.raw_rew_t) a.raw_rew_t[e] = reward;
            a.state[(int64_t)e * 4] = raw0;                             // of the observation now in cur_obs
        } else {
            a.rew_t[e] = reward;
        }
        a.term_t[e] = term ? 1.0f : 0.0f;
        a.trunc_t[e] = trunc ? 1.0f : 0.0f;
        const double ret = a.ep_return[e] + (double)reward;
        if (done && a.done_return) a.done_return[e] = (float)ret;
        if (done && a.auto_reset) { a.episode[e] += 1; a.steps[e] = 0; a.ep_return[e] = 0.0; }
        else { a.steps[e] += 1; a.ep_return[e] = ret; }
    }
}

template <bool NORM>
int launch_env_t(dppo_ctx* ctx, const EnvArgs& a, int mode, const unsigned char* mask, cudaStream_t st)
{
    const unsigned grid = (a.N + 127) / 128;
    switch (a.kind) {
    case 0: classic_env_kernel<0, NORM><<<grid, 128, 0, st>>>(a, mode, mask); break;
    case 1: classic_env_kernel<1, NORM><<<grid, 128, 0, st>>>(a, mode, mask); break;
    case 4: classic_env_kernel<4, NORM><<<grid, 128, 0, st>>>(a, mode, mask); break;
    case 5: classic_env_kernel<5, NORM><<<grid, 128, 0, st>>>(a, mode, mask); break;
    case 6: classic_env_kernel<6, NORM><<<grid, 128, 0, st>>>(a, mode, mask); break;
    default:
        synthetic_env_kernel<NORM><<<(unsigned)(((int64_t)a.N * 32 + 255) / 256), 256, 0, st>>>(a, mode, mask);
        DPPO_CHECK_LAUNCH(ctx, "synthetic_env_kernel");
        return 0;
    }
    DPPO_CHECK_LAUNCH(ctx, "classic_env_kernel");
    return 0;
}

int launch_env(dppo_ctx* ctx, const EnvArgs& a, int mode, const unsigned char* mask, cudaStream_t st)
{
    return (a.norm_obs || a.norm_rew) ? launch_env_t<true>(ctx, a, mode, mask, st) : launch_env_t<false>(ctx, a, mode, mask, st);
}

int fill_args(dppo_ctx* ctx, const dppo_env_desc* d, const dppo_env_state* s, EnvArgs& a)
{
    if (!d || !s) DPPO_FAIL(ctx, "env: null descriptor / state");
    if (d->kind < 0 || d->kind > 6 || d->num_envs < 1) DPPO_FAIL(ctx, "env: bad descriptor (kind %d, num_envs %d)", d->kind, d->num_envs);
    static const int kObsDim[7] = {4, 3, 0, 0, 6, 2, 2}, kActDim[7] = {0, 0, 0, 0, 3, 3, 1};   // 0: not checked
    if (kObsDim[d->kind] && d->obs_dim != kObsDim[d->kind])
        DPPO_FAIL(ctx, "env: obs_dim %d does not match kind %d (expected %d)", d->obs_dim, d->kind, kObsDim[d->kind]);
    if (d->obs_dim < 1) DPPO_FAIL(ctx, "env: obs_dim %d does not match kind %d", d->obs_dim, d->kind);
    if (kActDim[d->kind] && d->act_dim != kActDim[d->kind])
        DPPO_FAIL(ctx, "env: act_dim %d does not match kind %d (expected %d)", d->act_dim, d->kind, kActDim[d->kind]);
    if (!s->state || !s->steps || !s->episode || !s->ep_return || !s->cur_obs) DPPO_FAIL(ctx, "env: null state buffer");
    a.kind = d->kind; a.N = d->num_envs; a.D = d->obs_dim; a.A = d->act_dim;
    a.state = s->state; a.steps = s->steps; a.episode = s->episode; a.ep_return = s->ep_return; a.cur_obs = s->cur_obs;
    a.seed = d->seed; a.env_offset = d->env_offset; a.p_term = d->p_term; a.p_trunc = d->p_trunc;
    if (d->normalize & ~(DPPO_ENV_NORMALIZE_OBS | DPPO_ENV_NORMALIZE_REWARD)) DPPO_FAIL(ctx, "env: unknown normalize flags 0x%x", d->normalize);
    a.norm_obs = (d->normalize & DPPO_ENV_NORMALIZE_OBS) != 0;
    a.norm_rew = (d->normalize & DPPO_ENV_NORMALIZE_REWARD) != 0;
    if (a.norm_obs || a.norm_rew) {
        if (!s->update) DPPO_FAIL(ctx, "env: normalisation needs the device update flag");
        if (a.norm_obs && (!s->obs_mean || !s->obs_var || !s->obs_count)) DPPO_FAIL(ctx, "env: observation normalisation needs obs_mean / obs_var / obs_count");
        if (a.norm_rew && !s->ret_stats) DPPO_FAIL(ctx, "env: reward normalisation needs ret_stats");
        if (a.norm_rew && !(d->gamma >= 0.0 && d->gamma <= 1.0)) DPPO_FAIL(ctx, "env: gamma %g outside [0, 1]", d->gamma);
        if (!(d->epsilon > 0.0)) DPPO_FAIL(ctx, "env: epsilon %g must be > 0", d->epsilon);
        if (!(d->clip_observation >= 0.0) || !(d->clip_reward >= 0.0))
            DPPO_FAIL(ctx, "env: clips must be >= 0 (0: no clip); got %g / %g", d->clip_observation, d->clip_reward);
        a.gamma = d->gamma; a.eps = d->epsilon; a.clip_obs = d->clip_observation; a.clip_rew = d->clip_reward;
        a.obs_mean = s->obs_mean; a.obs_var = s->obs_var; a.obs_count = s->obs_count; a.ret_stats = s->ret_stats; a.update = s->update;
    }
    return 0;
}

}  // namespace

extern "C" int dppo_env_reset(dppo_ctx* ctx, const dppo_env_desc* desc, const dppo_env_state* state, const unsigned char* mask,
                              void* stream)
{
    if (!ctx) return 1;
    EnvArgs a = {};
    if (fill_args(ctx, desc, state, a)) return 1;
    return launch_env(ctx, a, 1, mask, (cudaStream_t)stream);
}

extern "C" int dppo_env_step(dppo_ctx* ctx, const dppo_env_desc* desc, const dppo_env_state* state, const void* actions, int t,
                             int auto_reset, float* obs, float* next_obs, void* buf_actions, float* rewards, float* terminations,
                             float* truncations, float* done_return, float* raw_rewards, void* stream)
{
    if (!ctx) return 1;
    EnvArgs a = {};
    if (fill_args(ctx, desc, state, a)) return 1;
    if (!actions || !next_obs || !rewards || !terminations || !truncations || t < 0) DPPO_FAIL(ctx, "env_step: null output / bad step");
    const int64_t N = a.N, D = a.D;
    const int cont = (a.kind == 1 || a.kind == 3 || a.kind == 6);
    a.t = t; a.auto_reset = auto_reset; a.actions = actions;
    a.obs_t = obs ? obs + (int64_t)t * N * D : nullptr;
    a.next_obs_t = next_obs + (int64_t)t * N * D;
    a.act_t = buf_actions ? (cont ? (void*)((float*)buf_actions + (int64_t)t * N * a.A) : (void*)((int32_t*)buf_actions + (int64_t)t * N)) : nullptr;
    a.rew_t = rewards + (int64_t)t * N; a.term_t = terminations + (int64_t)t * N; a.trunc_t = truncations + (int64_t)t * N;
    a.done_return = done_return;
    a.raw_rew_t = raw_rewards ? raw_rewards + (int64_t)t * N : nullptr;
    if (launch_env(ctx, a, 0, nullptr, (cudaStream_t)stream)) return 1;
    if (a.raw_rew_t && !a.norm_obs && !a.norm_rew &&                    // the kernel without normalisation writes no raw row
        cudaMemcpyAsync(a.raw_rew_t, a.rew_t, (size_t)N * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream) != cudaSuccess)
        DPPO_FAIL(ctx, "env_step: raw reward copy failed");
    return 0;
}
