// marlnav_b200/csrc/marlnav_rollout.cu
//
// The two caller-side pieces SURVEY.md section 8(f) ranks next after the environment step
// (rows f-2 and f-3), as device kernels behind the same C ABI:
//
//   marlnav_actor_sample_f32        Actor.forward + dist.sample() + dist.log_prob()
//                                   /root/reference/marlnav/models.py:27-36, 113-115
//   marlnav_discounted_returns_f64  the backward scan of MAPPO._process_rewards
//                                   /root/reference/marlnav/models.py:131-139
//
// The step kernel stays the product's hot path; these remove the ~10 small launches and the
// per-row Cholesky of MultivariateNormal around it, and the 1000-iteration Python loop after it.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/marlnav_b200.h"
#include "marlnav_actor.cuh"
#include "marlnav_launch.cuh"

namespace mnr {

// One thread per (env, agent) row.  The reference's Actor has NO activation after fc1
// (models.py:29-31): h = fc1(x); mu = tanh(fc_mu(h)); "std" = softplus(fc_std(h)), and that
// "std" is used as the diagonal COVARIANCE of MultivariateNormal (models.py:32-34), so the
// standard deviation of the sampled action is sqrt(softplus(.)).
//
// IT: the observations' element type (float, __half, __nv_bfloat16), widened exactly on load.
template <int MAX_S, int MAX_H, class IT = float>
__global__ void __launch_bounds__(128)
actor_sample_kernel(const IT* __restrict__ obs, long long N, int S, int H,
                    const float* __restrict__ w1, const float* __restrict__ b1,
                    const float* __restrict__ w_mu, const float* __restrict__ b_mu,
                    const float* __restrict__ w_std, const float* __restrict__ b_std,
                    const float* __restrict__ eps, uint64_t seed, uint64_t counter,
                    const unsigned long long* __restrict__ counter_dev, uint64_t row_offset,
                    float* __restrict__ actions, float* __restrict__ log_probs,
                    float* __restrict__ mu_out, float* __restrict__ var_out) {
    extern __shared__ float sm[];
    mna::stage_actor_weights(sm, S, H, w1, b1, w_mu, w_std, threadIdx.x, blockDim.x);
    __syncthreads();
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= N) return;

    float x[MAX_S];
#pragma unroll
    for (int k = 0; k < MAX_S; ++k) x[k] = k < S ? mna::widen(obs[row * S + k]) : 0.f;
    if (counter_dev) counter += __ldg(counter_dev);      // host value = offset inside a batch
    const mna::ActorOut o = mna::actor_row<MAX_S>(x, S, H, mna::ActorWeights(sm, S, H), b_mu, b_std, eps, seed, counter, row,
                                                      row_offset + (uint64_t)row);
    actions[row * 2] = o.a0; actions[row * 2 + 1] = o.a1;
    log_probs[row] = o.logp;
    if (mu_out) { mu_out[row * 2] = o.m0; mu_out[row * 2 + 1] = o.m1; }
    if (var_out) { var_out[row * 2] = o.v0; var_out[row * 2 + 1] = o.v1; }
}

// Critic.forward (models.py:39-56): value = fc2(relu(fc1(flatten(x)))), one thread per env.
// IT, in all three critic kernels: the observations' element type, widened exactly on load.
template <int MAX_H, class IT = float>
__global__ void __launch_bounds__(128)
critic_value_kernel(const IT* __restrict__ obs, long long B, int K, int H, const float* __restrict__ w1,
                    const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                    float* __restrict__ values) {
    extern __shared__ float sm[];
    float* s_w1 = sm;                    // transposed to (K,H) so that a thread walks j contiguously
    for (int i = threadIdx.x; i < H * K; i += blockDim.x) { const int j = i / K, k = i - j * K; s_w1[k * H + j] = w1[i]; }
    __syncthreads();
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    float h[MAX_H];
#pragma unroll
    for (int j = 0; j < MAX_H; ++j) h[j] = j < H ? b1[j] : 0.f;
    const IT* x = obs + e * K;
    for (int k = 0; k < K; ++k) {
        const float xk = mna::widen(x[k]);
#pragma unroll
        for (int j = 0; j < MAX_H; ++j)
            if (j < H) h[j] = fmaf(xk, s_w1[k * H + j], h[j]);
    }
    float v = b2[0];
#pragma unroll
    for (int j = 0; j < MAX_H; ++j)
        if (j < H) v = fmaf(fmaxf(h[j], 0.f), w2[j], v);
    values[e] = v;
}

// The same critic for SMALL batches (rollouts at the reference's scale, ~1 000 envs), where one
// thread per env is a 1 800-step serial chain on a handful of warps: here 64 lanes share an env, one
// hidden unit each (K steps), and one lane finishes the H-term output sum.  Same summation orders
// as critic_value_kernel, hence the same bits.  4 envs in flight per CTA.
template <int MAX_H, class IT = float>
__global__ void __launch_bounds__(4 * MAX_H)
critic_value_wide_kernel(const IT* __restrict__ obs, long long B, int K, int H, const float* __restrict__ w1,
                         const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                         float* __restrict__ values) {
    extern __shared__ float sm[];
    float* s_w1 = sm;                    // transposed to (K,H): lane j walks k with stride H, conflict-free
    float* s_h = sm + (size_t)H * K;     // (4, MAX_H) relu(h)
    for (int i = threadIdx.x; i < H * K; i += blockDim.x) { const int j = i / K, k = i - j * K; s_w1[k * H + j] = w1[i]; }
    __syncthreads();
    const int g = threadIdx.x / MAX_H, j = threadIdx.x % MAX_H;
    const long long stride = (long long)gridDim.x * 4;
    for (long long e0 = (long long)blockIdx.x * 4; e0 < B; e0 += stride) {      // uniform trip count per CTA
        const long long e = e0 + g;
        if (e < B && j < H) {
            const IT* x = obs + e * K;
            float h = b1[j];
            for (int k = 0; k < K; ++k) h = fmaf(mna::widen(__ldg(x + k)), s_w1[k * H + j], h);
            s_h[g * MAX_H + j] = fmaxf(h, 0.f);
        }
        __syncthreads();
        if (e < B && j == 0) {
            float v = b2[0];
            for (int jj = 0; jj < H; ++jj) v = fmaf(s_h[g * MAX_H + jj], w2[jj], v);
            values[e] = v;
        }
        __syncthreads();
    }
}

// Mid-sized batches: L = 16 or 4 lanes per env inside one warp, each lane owning the hidden units
// j = l, l + L, ... (independent K-step chains), lane 0 of the group finishing the H-term sum.
// Same summation orders again.
template <int L, int MAX_H, class IT = float>
__global__ void __launch_bounds__(128)
critic_value_group_kernel(const IT* __restrict__ obs, long long B, int K, int H, const float* __restrict__ w1,
                          const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                          float* __restrict__ values) {
    constexpr int PER = (MAX_H + L - 1) / L;             // hidden units per lane
    constexpr int GROUPS = 128 / L;                      // envs in flight per CTA
    extern __shared__ float sm[];
    float* s_w1 = sm;                                    // transposed to (K,H)
    float* s_h = sm + (size_t)H * K;                     // (GROUPS, MAX_H) relu(h)
    for (int i = threadIdx.x; i < H * K; i += blockDim.x) { const int j = i / K, k = i - j * K; s_w1[k * H + j] = w1[i]; }
    __syncthreads();
    const int g = threadIdx.x / L, l = threadIdx.x % L;
    const long long stride = (long long)gridDim.x * GROUPS;
    for (long long e0 = (long long)blockIdx.x * GROUPS; e0 < B; e0 += stride) {     // uniform trip count per CTA
        const long long e = e0 + g;
        if (e < B) {
            const IT* x = obs + e * K;
            float h[PER];
#pragma unroll
            for (int u = 0; u < PER; ++u) h[u] = (l + u * L) < H ? b1[l + u * L] : 0.f;
            for (int k = 0; k < K; ++k) {
                const float xk = mna::widen(__ldg(x + k));
#pragma unroll
                for (int u = 0; u < PER; ++u)
                    if ((l + u * L) < H) h[u] = fmaf(xk, s_w1[k * H + l + u * L], h[u]);
            }
#pragma unroll
            for (int u = 0; u < PER; ++u)
                if ((l + u * L) < H) s_h[g * MAX_H + l + u * L] = fmaxf(h[u], 0.f);
        }
        __syncwarp();
        if (e < B && l == 0) {
            float v = b2[0];
            for (int jj = 0; jj < H; ++jj) v = fmaf(s_h[g * MAX_H + jj], w2[jj], v);
            values[e] = v;
        }
        __syncwarp();
    }
}

// models.py:131-139, literally, in float64: curr = done ? 0 : rew + gamma * curr, backwards in t.
// (T,B) row-major: for a fixed t consecutive threads touch consecutive envs.
__global__ void discounted_returns_kernel(const float* __restrict__ rewards, const uint8_t* __restrict__ done,
                                          double gamma, int T, long long B, double* __restrict__ out) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double curr = 0.0;
    int t = T - 1;
    // the loads do not depend on the recurrence: fetch eight steps ahead of it
    for (; t >= 7; t -= 8) {
        float r[8]; uint8_t d[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const long long i = (long long)(t - u) * B + b;
            r[u] = rewards[i]; d[u] = done[i];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            curr = d[u] ? 0.0 : __dadd_rn((double)r[u], __dmul_rn(gamma, curr));
            out[(long long)(t - u) * B + b] = curr;
        }
    }
    for (; t >= 0; --t) {
        const long long i = (long long)t * B + b;
        curr = done[i] ? 0.0 : __dadd_rn((double)rewards[i], __dmul_rn(gamma, curr));
        out[i] = curr;
    }
}

// Generalised advantage estimation that tells a time-limit truncation (bootstrapped from the
// value of the observation the episode ended on) from a termination (include/marlnav_b200_final.h),
// in float64 with every operation rounded to nearest and no FMA.  Shaped like
// discounted_returns_kernel: a thread per env, the loads eight steps ahead of the recurrence.
__global__ void gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                           const uint8_t* __restrict__ terminated, const uint8_t* __restrict__ truncated,
                           const float* __restrict__ final_values, const float* __restrict__ last_values,
                           double gamma, double lam, int T, long long B, double* __restrict__ adv_out,
                           double* __restrict__ ret_out) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double gl = __dmul_rn(gamma, lam);
    double adv = 0.0;
    double v_next = last_values ? (double)last_values[b] : 0.0;     // values[t+1, b]
    const auto step = [&](long long i, float r, float v, uint8_t te, uint8_t tr, float fv) {
        const double vd = (double)v;
        double nv = v_next;
        bool cont = true;
        if (te) { nv = 0.0; cont = false; }
        else if (tr) { nv = (double)fv; cont = false; }
        const double delta = __dsub_rn(__dadd_rn((double)r, __dmul_rn(gamma, nv)), vd);
        adv = cont ? __dadd_rn(delta, __dmul_rn(gl, adv)) : delta;
        adv_out[i] = adv;
        ret_out[i] = __dadd_rn(adv, vd);
        v_next = vd;
    };
    int t = T - 1;
    for (; t >= 7; t -= 8) {
        float r[8], v[8], fv[8]; uint8_t te[8], tr[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const long long i = (long long)(t - u) * B + b;
            r[u] = rewards[i]; v[u] = values[i]; te[u] = terminated[i]; tr[u] = truncated[i];
            fv[u] = final_values ? final_values[i] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) step((long long)(t - u) * B + b, r[u], v[u], te[u], tr[u], fv[u]);
    }
    for (; t >= 0; --t) {
        const long long i = (long long)t * B + b;
        step(i, rewards[i], values[i], terminated[i], truncated[i], final_values ? final_values[i] : 0.f);
    }
}

}  // namespace mnr

namespace {
thread_local char g_err2[256] = "";

int cuda_fail(cudaError_t e, const char* where) {
    snprintf(g_err2, sizeof g_err2, "%s: %s", where, cudaGetErrorString(e));
    return (int)e;
}

// critic_value_group_kernel: few enough CTAs per SM that the per-CTA weight staging amortises
// over several env groups
constexpr int kCriticGroupCtasPerSm = 4;

// The bodies of the `_f32` and `_typed` rollout entries; IT = the observations' element type and
// `fn` the entry's name for the error message.
template <class IT>
int actor_sample(const char* fn, const IT* obs, long long N, int S, int H, const float* w1, const float* b1,
                 const float* w_mu, const float* b_mu, const float* w_std, const float* b_std,
                 const float* eps, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                 uint64_t row_offset,
                 float* actions, float* log_probs, float* mu_out, float* var_out, void* stream) {
    if (!obs || !w1 || !b1 || !w_mu || !b_mu || !w_std || !b_std || !actions || !log_probs || N < 1) {
        snprintf(g_err2, sizeof g_err2, "%s: NULL pointer or empty batch", fn);
        return MARLNAV_ERR_BAD_ARG;
    }
    if (S < 1 || S > 64 || H < 1 || H > 256) {
        snprintf(g_err2, sizeof g_err2, "%s: need 1 <= obs_size <= 64 and 1 <= hidden <= 256", fn);
        return MARLNAV_ERR_BAD_SHAPE;
    }
    const int threads = 128;
    const long long grid = (N + threads - 1) / threads;
    const size_t smem = (size_t)(H * S + H + 4 * H) * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    // same shared-memory carveout as the step kernels it alternates with, and room for the largest
    // advertised shape (S = 64, H = 256: 69 KiB of weights)
    const size_t max_smem = (256 * 64 + 5 * 256) * sizeof(float);
    cudaError_t e = S <= 16 ? mnl::set_attributes_once<mnr::actor_sample_kernel<16, 256, IT>>(max_smem, true)
                            : mnl::set_attributes_once<mnr::actor_sample_kernel<64, 256, IT>>(max_smem, true);
    if (e != cudaSuccess) return cuda_fail(e, "actor_sample attributes");
    if (S <= 16)
        mnr::actor_sample_kernel<16, 256, IT><<<(unsigned)grid, threads, smem, st>>>(
            obs, N, S, H, w1, b1, w_mu, b_mu, w_std, b_std, eps, seed, counter,
            reinterpret_cast<const unsigned long long*>(counter_dev), row_offset, actions, log_probs, mu_out, var_out);
    else
        mnr::actor_sample_kernel<64, 256, IT><<<(unsigned)grid, threads, smem, st>>>(
            obs, N, S, H, w1, b1, w_mu, b_mu, w_std, b_std, eps, seed, counter,
            reinterpret_cast<const unsigned long long*>(counter_dev), row_offset, actions, log_probs, mu_out, var_out);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "actor_sample launch");
}

template <class IT>
int critic_value(const char* fn, const IT* obs, long long B, int K, int H, const float* w1, const float* b1,
                 const float* w2, const float* b2, float* values, void* stream) {
    if (!obs || !w1 || !b1 || !w2 || !b2 || !values || B < 1) {
        snprintf(g_err2, sizeof g_err2, "%s: NULL pointer or empty batch", fn);
        return MARLNAV_ERR_BAD_ARG;
    }
    if (K < 1 || H < 1 || H > 64 || (size_t)H * K * sizeof(float) > 200 * 1024) {
        snprintf(g_err2, sizeof g_err2, "%s: need hidden <= 64 and hidden*inputs*4 <= 200 KiB", fn);
        return MARLNAV_ERR_BAD_SHAPE;
    }
    if (B > 2048 && B <= 262144 && (size_t)(H * K + 32 * 64) * sizeof(float) <= 48 * 1024) {
        // mid-sized batches: 16 or 4 lanes per env (see critic_value_group_kernel)
        const bool l16 = B <= 32768;
        cudaError_t e = l16 ? mnl::set_attributes_once<mnr::critic_value_group_kernel<16, 64, IT>>(0, true)
                            : mnl::set_attributes_once<mnr::critic_value_group_kernel<4, 64, IT>>(0, true);
        if (e != cudaSuccess) return cuda_fail(e, "critic_value_group attributes");
        const int groups = l16 ? 8 : 32;
        const long long want = (B + groups - 1) / groups;
        const long long cap = 148 * kCriticGroupCtasPerSm;
        const unsigned grid = (unsigned)(want < cap ? want : cap);
        const size_t smem = (size_t)(H * K + groups * 64) * sizeof(float);
        if (l16)
            mnr::critic_value_group_kernel<16, 64, IT><<<grid, 128, smem, (cudaStream_t)stream>>>(obs, B, K, H, w1, b1, w2, b2, values);
        else
            mnr::critic_value_group_kernel<4, 64, IT><<<grid, 128, smem, (cudaStream_t)stream>>>(obs, B, K, H, w1, b1, w2, b2, values);
        e = cudaGetLastError();
        return e == cudaSuccess ? 0 : cuda_fail(e, "critic_value_group launch");
    }
    if (B <= 2048 && (size_t)(H * K + 4 * 64) * sizeof(float) <= 48 * 1024) {
        // rollout-sized batches: 64 lanes per env (see critic_value_wide_kernel)
        const long long want = (B + 3) / 4;
        const unsigned grid = (unsigned)(want < 148 * 8 ? want : 148 * 8);
        // same shared-memory carveout as the step kernels: SMs need not drain and reconfigure when
        // this runs beside them on a forked stream (collect_rollout)
        cudaError_t e = mnl::set_attributes_once<mnr::critic_value_wide_kernel<64, IT>>(0, true);
        if (e != cudaSuccess) return cuda_fail(e, "critic_value_wide attributes");
        mnr::critic_value_wide_kernel<64, IT><<<grid, 256, (size_t)(H * K + 4 * 64) * sizeof(float), (cudaStream_t)stream>>>(
            obs, B, K, H, w1, b1, w2, b2, values);
        e = cudaGetLastError();
        return e == cudaSuccess ? 0 : cuda_fail(e, "critic_value_wide launch");
    }
    const int threads = 128;
    const size_t smem = (size_t)H * K * sizeof(float);
    if (smem > 48 * 1024) {
        if (cudaError_t e = mnl::set_attributes_once<mnr::critic_value_kernel<64, IT>>(200 * 1024, false))
            return cuda_fail(e, "critic_value attributes");
    }
    mnr::critic_value_kernel<64, IT><<<(unsigned)((B + threads - 1) / threads), threads, smem, (cudaStream_t)stream>>>(
        obs, B, K, H, w1, b1, w2, b2, values);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "critic_value launch");
}

bool obs_dtype_ok(int obs_dtype) {
    if (obs_dtype == MARLNAV_OBS_F32 || obs_dtype == MARLNAV_OBS_F16 || obs_dtype == MARLNAV_OBS_BF16) return true;
    snprintf(g_err2, sizeof g_err2,
             "obs_dtype must be MARLNAV_OBS_F32 (0), MARLNAV_OBS_F16 (1) or MARLNAV_OBS_BF16 (2), got %d", obs_dtype);
    return false;
}

}  // namespace

extern "C" {

const char* marlnav_rollout_last_error(void) { return g_err2; }

int marlnav_actor_sample_f32(const float* obs, long long N, int S, int H, const float* w1, const float* b1,
                             const float* w_mu, const float* b_mu, const float* w_std, const float* b_std,
                             const float* eps, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                             uint64_t row_offset,
                             float* actions, float* log_probs, float* mu_out, float* var_out, void* stream) {
    return actor_sample("marlnav_actor_sample_f32", obs, N, S, H, w1, b1, w_mu, b_mu, w_std, b_std, eps, seed,
                        counter, counter_dev, row_offset, actions, log_probs, mu_out, var_out, stream);
}

int marlnav_actor_sample_typed(const void* obs, int obs_dtype, long long N, int S, int H, const float* w1,
                               const float* b1, const float* w_mu, const float* b_mu, const float* w_std,
                               const float* b_std, const float* eps, uint64_t seed, uint64_t counter,
                               const uint64_t* counter_dev, uint64_t row_offset,
                               float* actions, float* log_probs, float* mu_out, float* var_out, void* stream) {
    if (!obs_dtype_ok(obs_dtype)) return MARLNAV_ERR_BAD_ARG;
    const char* fn = "marlnav_actor_sample_typed";
    switch (obs_dtype) {
        case MARLNAV_OBS_F16:
            return actor_sample(fn, static_cast<const __half*>(obs), N, S, H, w1, b1, w_mu, b_mu, w_std, b_std, eps,
                                seed, counter, counter_dev, row_offset, actions, log_probs, mu_out, var_out, stream);
        case MARLNAV_OBS_BF16:
            return actor_sample(fn, static_cast<const __nv_bfloat16*>(obs), N, S, H, w1, b1, w_mu, b_mu, w_std, b_std,
                                eps, seed, counter, counter_dev, row_offset, actions, log_probs, mu_out, var_out, stream);
        default:
            return actor_sample(fn, static_cast<const float*>(obs), N, S, H, w1, b1, w_mu, b_mu, w_std, b_std, eps,
                                seed, counter, counter_dev, row_offset, actions, log_probs, mu_out, var_out, stream);
    }
}

int marlnav_critic_value_f32(const float* obs, long long B, int K, int H, const float* w1, const float* b1,
                             const float* w2, const float* b2, float* values, void* stream) {
    return critic_value("marlnav_critic_value_f32", obs, B, K, H, w1, b1, w2, b2, values, stream);
}

int marlnav_critic_value_typed(const void* obs, int obs_dtype, long long B, int K, int H, const float* w1,
                               const float* b1, const float* w2, const float* b2, float* values, void* stream) {
    if (!obs_dtype_ok(obs_dtype)) return MARLNAV_ERR_BAD_ARG;
    const char* fn = "marlnav_critic_value_typed";
    switch (obs_dtype) {
        case MARLNAV_OBS_F16:
            return critic_value(fn, static_cast<const __half*>(obs), B, K, H, w1, b1, w2, b2, values, stream);
        case MARLNAV_OBS_BF16:
            return critic_value(fn, static_cast<const __nv_bfloat16*>(obs), B, K, H, w1, b1, w2, b2, values, stream);
        default:
            return critic_value(fn, static_cast<const float*>(obs), B, K, H, w1, b1, w2, b2, values, stream);
    }
}

int marlnav_discounted_returns_f64(const float* rewards, const uint8_t* done, double gamma, int T, long long B,
                                   double* out, void* stream) {
    if (!rewards || !done || !out || T < 1 || B < 1) {
        snprintf(g_err2, sizeof g_err2, "marlnav_discounted_returns_f64: NULL pointer or empty buffer");
        return MARLNAV_ERR_BAD_ARG;
    }
    const int threads = 128;
    mnr::discounted_returns_kernel<<<(unsigned)((B + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        rewards, done, gamma, T, B, out);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "discounted_returns launch");
}

int marlnav_gae_f64(const float* rewards, const float* values, const uint8_t* terminated,
                    const uint8_t* truncated, const float* final_values, const float* last_values,
                    double gamma, double lam, int T, long long B,
                    double* advantages, double* returns, void* stream) {
    if (!rewards || !values || !terminated || !truncated || !advantages || !returns || T < 1 || B < 1) {
        snprintf(g_err2, sizeof g_err2, "marlnav_gae_f64: NULL pointer or empty buffer");
        return MARLNAV_ERR_BAD_ARG;
    }
    if (advantages == returns) {
        snprintf(g_err2, sizeof g_err2, "marlnav_gae_f64: advantages and returns must be different buffers");
        return MARLNAV_ERR_BAD_ARG;
    }
    const int threads = 128;
    mnr::gae_kernel<<<(unsigned)((B + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        rewards, values, terminated, truncated, final_values, last_values, gamma, lam, T, B, advantages, returns);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "gae launch");
}

}  // extern "C"
