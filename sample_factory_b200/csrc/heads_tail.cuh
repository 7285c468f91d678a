// Row tails of the policy/value heads, shared by heads.cu (stand-alone kernels, sampler step tail) and rollout_fused.cu (the
// persistent rollout kernel): lane a of a warp holds output a of one row (0 = value, 1.. = distribution_linear rows).
#pragma once
#include <curand_kernel.h>

#include "common.cuh"

namespace sfb {

struct HeadsOut {
    float* values; int64_t values_stride;
    float* logits; int64_t logits_stride;
    float* actions_f32; int64_t actions_stride;
    int32_t* env_actions;
    float* log_prob; int64_t log_prob_stride;
    float* pv_out; int64_t pv_stride;
    // continuous (diagonal Gaussian) action space: dist 0 = categorical, 1 = Gaussian with state-dependent log-stddev
    // (the linear layer has 2*act_dim rows), 2 = Gaussian with one learned log-stddev vector (act_dim rows)
    int dist; int act_dim; const float* learned_log_std; float tanh_scale; float* env_actions_f32;
    // Tuple(Discrete(n_0), ..., Discrete(n_{K-1})) action space (action_distributions.py:197-286): K independent
    // categorical heads over consecutive logit segments; num_seg <= 1 means one plain categorical
    int num_seg; int seg_len[8];
    // sampling mode (sfb200_set_sampling_mode): action_mask[row * mask_stride + a] == 0 forbids action a of a plain
    // Discrete space (masked_softmax / masked_log_softmax, action_distributions.py:84-95); deterministic = argmax of the
    // probabilities / the Gaussian means instead of a draw (enjoy.py:165-171 eval_deterministic)
    const uint8_t* action_mask = nullptr; int64_t mask_stride = 0; int deterministic = 0;
};

constexpr float kStddevMin = 1e-4f, kStddevMax = 1e4f;   // action_distributions.py:291-292
constexpr float kHalfLog2Pi = 0.91893853320467274178f;   // log(sqrt(2 pi))

// ContinuousActionDistribution (action_distributions.py:290-323) on the lanes: lane j in 1..act_dim owns action
// dimension j-1.  Stored `logits` are the distribution parameters [means | log_std] (2*act_dim floats) exactly as the
// reference's action_parameterization returns them (tanh-scaled means and the repeated learned vector when
// adaptive_stddev=False, action_parameterization.py:64-78).
__device__ __forceinline__ void gaussian_row_tail(float mine, int lane, int64_t row, const HeadsOut& out,
                                                  const float* __restrict__ noise, uint64_t seed, uint64_t offset,
                                                  float pv) {
    const int Ad = out.act_dim;
    const bool is_dim = lane >= 1 && lane <= Ad;
    float mean = mine, log_std;
    if (out.dist == 1) {
        const int src = lane + Ad;
        log_std = __shfl_sync(0xffffffffu, mine, src < 32 ? src : 31);
    } else {
        log_std = is_dim ? out.learned_log_std[lane - 1] : 0.f;
        if (out.tanh_scale > 0.f) mean = tanhf(__fdiv_rn(mine, out.tanh_scale)) * out.tanh_scale;
    }
    if (out.logits && is_dim) {
        out.logits[row * out.logits_stride + (lane - 1)] = mean;
        out.logits[row * out.logits_stride + Ad + (lane - 1)] = log_std;
    }
    if (out.actions_f32 == nullptr) return;   // values / distribution parameters only (warp-uniform)
    const float sd = clampf(expf(log_std), kStddevMin, kStddevMax);
    float eps = 0.f;
    if (is_dim && !out.deterministic) {
        if (noise) eps = noise[row * Ad + (lane - 1)];
        else {
            curandStatePhilox4_32_10_t st;
            curand_init(seed, (unsigned long long)(row * Ad + (lane - 1)), offset, &st);
            eps = curand_normal(&st);
        }
    }
    // Normal.sample(): eps * std + mean, product and sum rounded separately (SURVEY App.C)
    const float a = __fadd_rn(__fmul_rn(eps, sd), mean);
    const float d = a - mean;
    const float lpj = is_dim ? (-(d * d) / (2.f * (sd * sd)) - logf(sd) - kHalfLog2Pi) : 0.f;   // normal.py:84-94
    const float lp = warp_sum(lpj);                                                              // Independent(.., 1)
    if (is_dim) {
        out.actions_f32[row * out.actions_stride + (lane - 1)] = a;
        if (out.env_actions_f32) out.env_actions_f32[row * Ad + (lane - 1)] = a;
    }
    if (lane == 0) {
        if (out.log_prob) out.log_prob[row * out.log_prob_stride] = lp;
        if (out.pv_out) out.pv_out[row * out.pv_stride] = pv;
    }
}

__device__ __forceinline__ void tuple_row_tail(float mine, int lane, int A, int64_t row, const HeadsOut& out,
                                               const float* __restrict__ noise, uint64_t seed, uint64_t offset, float pv);

// Lane a of the warp holds output a of one row (0 = value, 1..A = logits, bias included): store them and, in sampling
// mode, run CategoricalActionDistribution (action_distributions.py:110-148) on the lanes.
// Returns the sampled action index of a plain Discrete space (the same value in every lane), -1 otherwise.
__device__ __forceinline__ int heads_row_tail(float mine, int lane, int A, int64_t row, const HeadsOut& out,
                                              const float* __restrict__ noise, uint64_t seed, uint64_t offset, float pv) {
    if (lane == 0) out.values[row * out.values_stride] = mine;
    if (out.dist != 0) {
        gaussian_row_tail(mine, lane, row, out, noise, seed, offset, pv);
        return -1;
    }
    const bool is_logit = lane >= 1 && lane <= A;
    if (out.logits && is_logit) out.logits[row * out.logits_stride + (lane - 1)] = mine;
    if (out.actions_f32 == nullptr) return -1;   // values / logits only (warp-uniform)
    if (out.num_seg > 1) {
        tuple_row_tail(mine, lane, A, row, out, noise, seed, offset, pv);
        return -1;
    }

    const bool masked = out.action_mask != nullptr;
    const float mk = (masked && is_logit && out.action_mask[row * out.mask_stride + (lane - 1)] != 0) ? 1.f : 0.f;
    // masked_softmax / masked_log_softmax :84-95: a forbidden logit gets -1e9 added (an allowed one -0.0: unchanged)
    const float x = is_logit ? ((masked && mk == 0.f) ? __fadd_rn(mine, -1.0e9f) : mine) : -INFINITY;
    const float m = warp_max(x);
    const float e = is_logit ? expf(x - m) : 0.f;
    const float s = warp_sum(e);
    float p = __fdiv_rn(e, s);                          // softmax :116
    const float logp = (x - m) - logf(s);               // log_softmax :125
    if (masked) {
        p = __fmul_rn(p, mk);                                              // :88
        p = __fdiv_rn(p, __fadd_rn(warp_sum(p), 1.0e-13f));                // :89
        if (__ballot_sync(0xffffffffu, p > 0.f) == 0u) p = 1.0e-6f;        // :137-140 nothing allowed: uniform fallback
    }
    float q = 1.f;
    if (is_logit && !out.deterministic) {
        if (noise) q = noise[row * A + (lane - 1)];
        else {
            curandStatePhilox4_32_10_t st;
            curand_init(seed, (unsigned long long)(row * A + (lane - 1)), offset, &st);
            q = -logf(curand_uniform(&st));             // Exp(1); uniform is in (0, 1]
            q = fmaxf(q, 1.0e-30f);
        }
    }
    // torch.multinomial(p, 1, True) == argmax(p / q) (first index on ties)
    float best = is_logit ? __fdiv_rn(p, q) : -INFINITY;
    int idx = is_logit ? (lane - 1) : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ob > best || (ob == best && oi < idx)) { best = ob; idx = oi; }
    }
    const float lp = __shfl_sync(0xffffffffu, logp, idx + 1);   // log_prob :145-148
    if (lane == 0) {
        out.actions_f32[row * out.actions_stride] = (float)idx;
        if (out.env_actions) out.env_actions[row] = idx;
        if (out.log_prob) out.log_prob[row * out.log_prob_stride] = lp;
        if (out.pv_out) out.pv_out[row * out.pv_stride] = pv;
    }
    return idx;
}

// TupleActionDistribution on the lanes: every head runs the categorical recipe on its own lane range; actions_f32 gets K
// floats per row (one index per head), env_actions K int32, log_prob the sum over the heads (:231-241).
__device__ __forceinline__ void tuple_row_tail(float mine, int lane, int A, int64_t row, const HeadsOut& out,
                                               const float* __restrict__ noise, uint64_t seed, uint64_t offset, float pv) {
    const bool is_logit = lane >= 1 && lane <= A;
    float q = 1.f;
    if (is_logit && !out.deterministic) {
        if (noise) q = noise[row * A + (lane - 1)];
        else {
            curandStatePhilox4_32_10_t st;
            curand_init(seed, (unsigned long long)(row * A + (lane - 1)), offset, &st);
            q = fmaxf(-logf(curand_uniform(&st)), 1.0e-30f);
        }
    }
    float lp_total = 0.f;
    int start = 0;
    const int K = out.num_seg;
    for (int k = 0; k < K; ++k) {
        const int n = out.seg_len[k];
        const bool in_seg = (lane - 1) >= start && (lane - 1) < start + n;
        const float x = in_seg ? mine : -INFINITY;
        const float m = warp_max(x);
        const float e = in_seg ? expf(x - m) : 0.f;
        const float s = warp_sum(e);
        const float p = __fdiv_rn(e, s);
        const float logp = (x - m) - logf(s);
        float best = in_seg ? __fdiv_rn(p, q) : -INFINITY;
        int idx = in_seg ? (lane - 1 - start) : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (ob > best || (ob == best && oi < idx)) { best = ob; idx = oi; }
        }
        lp_total += __shfl_sync(0xffffffffu, logp, start + idx + 1);
        if (lane == 0) {
            out.actions_f32[row * out.actions_stride + k] = (float)idx;
            if (out.env_actions) out.env_actions[row * K + k] = idx;
        }
        start += n;
    }
    if (lane == 0) {
        if (out.log_prob) out.log_prob[row * out.log_prob_stride] = lp_total;
        if (out.pv_out) out.pv_out[row * out.pv_stride] = pv;
    }
}


// partial head dot products left by the fused GEMM epilogue: part[p][row][kHeadPartPad]
constexpr int kHeadPartPad = 12;

// everything the finishing step of the heads needs besides the partials
struct HeadsFinish {
    HeadsOut out;
    const float* bv;
    const float* ba;
    const float* noise;
    uint64_t seed, offset_host;
    const int64_t* offset_dev;
    const float* pv_scalar;
    int A;               // rows of distribution_linear
};

// one warp finishes one row: fixed-order sum of the P partials (deterministic) + bias, then the distribution tail
__device__ __forceinline__ int heads_finish_row(const float* __restrict__ part, int P, int64_t rows, int64_t row, int lane,
                                                const HeadsFinish& f, float pv, uint64_t offset) {
    float mine = 0.f;
    if (lane <= f.A) {
        for (int p = 0; p < P; ++p) mine += part[((int64_t)p * rows + row) * kHeadPartPad + lane];
    }
    mine += (lane == 0) ? f.bv[0] : (lane <= f.A ? f.ba[lane - 1] : 0.f);
    return heads_row_tail(mine, lane, f.A, row, f.out, f.noise, f.seed, offset, pv);
}

}  // namespace sfb
