// marlnav_b200/csrc/marlnav_actor.cuh
//
// One row of the reference's Actor (/root/reference/marlnav/models.py:27-36) with its
// diagonal-Gaussian sample and log-prob (models.py:113-115), as ONE device function shared by
// the stand-alone actor kernel (marlnav_rollout.cu) and the fused {actor -> step} kernel
// (marlnav_step_env.cu, marlnav_step_team.cu), so that both produce the same bits:
//
//   h = fc1(x)  (NO activation, models.py:29-31);  mu = tanh(fc_mu(h));  var = softplus(fc_std(h))
//   dist = MultivariateNormal(mu, covariance_matrix=diag(var))   -> std dev = sqrt(var)
//   a = mu + sqrt(var) * eps;   log_prob(a), k = 2
//
// eps: given (parity tests), or Philox4x32-10 + Box-Muller addressed by (seed; GLOBAL row, counter).
// Weights in shared memory in torch.nn.Linear layout: w1 (H,S), b1 (H), w_mu/w_std (2,H).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace mna {

// An observation as the policy and the critic read it: float32 as stored, a 16-bit one widened to
// float32 (exact for half and bfloat16), so a 16-bit input gives the bits of its .float() copy.
__device__ __forceinline__ float widen(float x) { return x; }
__device__ __forceinline__ float widen(__half x) { return __half2float(x); }
__device__ __forceinline__ float widen(__nv_bfloat16 x) { return __bfloat162float(x); }

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

struct ActorWeights {            // shared-memory pointers
    const float *w1, *b1, *wm, *ws;
    __device__ __forceinline__ static size_t floats(int S, int H) { return (size_t)H * S + H + 4 * (size_t)H; }
    __device__ __forceinline__ ActorWeights(const float* base, int S, int H)
        : w1(base), b1(base + H * S), wm(base + H * S + H), ws(base + H * S + H + 2 * H) {}
};

// cooperative copy of the six weight tensors into shared memory (caller synchronises afterwards)
__device__ __forceinline__ void stage_actor_weights(float* base, int S, int H, const float* __restrict__ w1,
                                                    const float* __restrict__ b1, const float* __restrict__ w_mu,
                                                    const float* __restrict__ w_std, int tid, int nthreads) {
    float* s_w1 = base;
    float* s_b1 = s_w1 + H * S;
    float* s_wm = s_b1 + H;
    float* s_ws = s_wm + 2 * H;
    for (int i = tid; i < H * S; i += nthreads) s_w1[i] = w1[i];
    for (int i = tid; i < H; i += nthreads) s_b1[i] = b1[i];
    for (int i = tid; i < 2 * H; i += nthreads) { s_wm[i] = w_mu[i]; s_ws[i] = w_std[i]; }
}

struct ActorOut { float a0, a1, logp, m0, m1, v0, v1; };

template <int MAX_S>
__device__ __forceinline__ ActorOut actor_row(const float (&x)[MAX_S], int S, int H, const ActorWeights& w,
                                              const float* __restrict__ b_mu, const float* __restrict__ b_std,
                                              const float* __restrict__ eps, uint64_t seed, uint64_t counter,
                                              long long row, uint64_t grow /* global row: Philox address */) {
    float m0 = b_mu[0], m1 = b_mu[1], v0 = b_std[0], v1 = b_std[1];
    for (int j = 0; j < H; ++j) {
        float h = w.b1[j];
#pragma unroll
        for (int k = 0; k < MAX_S; ++k)
            if (k < S) h = fmaf(x[k], w.w1[j * S + k], h);
        m0 = fmaf(h, w.wm[j], m0); m1 = fmaf(h, w.wm[H + j], m1);
        v0 = fmaf(h, w.ws[j], v0); v1 = fmaf(h, w.ws[H + j], v1);
    }
    m0 = tanhf(m0); m1 = tanhf(m1);
    v0 = v0 > 20.f ? v0 : log1pf(expf(v0));          // F.softplus, beta 1, threshold 20
    v1 = v1 > 20.f ? v1 : log1pf(expf(v1));

    float e0, e1;
    if (eps) { e0 = eps[row * 2]; e1 = eps[row * 2 + 1]; }
    else {
        const uint4 r = philox4x32_10((uint32_t)grow, (uint32_t)(grow >> 32), (uint32_t)counter,
                                      0x41435452u /* 'ACTR' */, (uint32_t)seed,
                                      (uint32_t)(seed >> 32) ^ (uint32_t)(counter >> 32));
        const float u1 = ((float)(r.x >> 8) + 1.0f) * 5.9604644775390625e-08f;      // (0, 1]
        const float u2 = (float)(r.y >> 8) * 5.9604644775390625e-08f;               // [0, 1)
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincospif(2.0f * u2, &sn, &cs);
        e0 = rad * cs; e1 = rad * sn;
    }
    ActorOut o;
    o.a0 = fmaf(sqrtf(v0), e0, m0); o.a1 = fmaf(sqrtf(v1), e1, m1);
    // MultivariateNormal(mu, diag(v)).log_prob(a), k = 2
    const float d0 = o.a0 - m0, d1 = o.a1 - m1;
    const float maha = d0 * d0 / v0 + d1 * d1 / v1;
    o.logp = -0.5f * maha - 0.5f * (logf(v0) + logf(v1)) - 1.8378770664093453f;
    o.m0 = m0; o.m1 = m1; o.v0 = v0; o.v1 = v1;
    return o;
}

}  // namespace mna
