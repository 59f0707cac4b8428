// reduce.cuh — sum of the per-block gradient partials (+ Adam): argument block and per-entry epilogue shared by
// reduce_adam_kernel and allreduce_adam_kernel (trainer.cu).
//
// Replaces loss.backward()'s accumulation over the batch and optimizer.step() (ac_nets.py:70-72, 117-119) for the
// fused trainer.  The gradient kernels leave one partial row per block; the rows are summed in a FIXED order
// (32 interleaved slices, each ascending, then the slices ascending).
// (A variant that fused this reduction into the tail of the producing kernel — last block to finish sums and steps —
// was measured at 2x the step time: one block cannot keep enough loads in flight; the launch gap it was meant to
// remove is hidden by programmatic dependent launch instead, common.cuh.)
#pragma once

#include "common.cuh"

namespace ia2c {

struct ReduceArgs {
    const float* partials;
    int n_blocks, P;
    float* grad;            // [N, P+1]
    float* grad_accum;      // [N, P] or null
    float* params; float* m; float* v;
    int32_t* step;          // [N], already incremented for this update
    float* loss_out;        // [N]
    float loss_scale;       // 1 / (T * E_total)
    double lr;
    int apply_adam, from_partials;
};

__host__ __device__ inline ReduceArgs make_reduce_args(const ia2c_episode_desc& d, int which, int n_blocks) {
    ReduceArgs R;
    R.partials = d.partials;
    R.n_blocks = n_blocks;
    R.P = which == 0 ? kCriticP : kActorP;
    R.grad = which == 0 ? d.critic_grad : d.actor_grad;
    R.grad_accum = which == 0 ? nullptr : d.actor_grad_accum;
    R.params = which == 0 ? d.critic_params : d.actor_params;
    R.m = which == 0 ? d.critic_m : d.actor_m;
    R.v = which == 0 ? d.critic_v : d.actor_v;
    R.step = which == 0 ? d.critic_step : d.actor_step;
    R.loss_out = d.loss_out + (which == 0 ? 0 : d.N);
    R.loss_scale = 1.f / (float)((int64_t)d.T * d.E_total);
    R.lr = which == 0 ? d.lr_critic : d.lr_actor;
    R.apply_adam = !(d.flags & IA2C_FLAG_SKIP_ADAM);
    R.from_partials = 1;
    return R;
}

// Per-run learning rates of a batch of runs (reduce_adam_kernel<true>): net n belongs to run n / N; lr == NULL -> ReduceArgs.lr.
struct ReduceRuns {
    const double* lr;
    int N;
};
template <bool RUNS>
using ReduceRunsArg = std::conditional_t<RUNS, ReduceRuns, NoRuns>;
template <bool RUNS>
__device__ __forceinline__ double reduce_lr(const ReduceArgs& R, const ReduceRunsArg<RUNS>& rr, int n) {
    if constexpr (RUNS) {
        return rr.lr ? rr.lr[n / rr.N] : R.lr;
    } else {
        return R.lr;
    }
}

// b^t by binary exponentiation: about 2 log2(t) DMULs, two of them per step independent, instead of pow()'s log/exp sequence.
// Every multiply rounds once, so the relative error stays below 2 log2(t) * 2^-53 (< 7e-15 for any int32 t): far inside the
// float rounding the bias corrections get below.
__device__ __forceinline__ double pow_uint(double b, unsigned t) {
    double r = 1.0;
    for (; t; t >>= 1) {
        if (t & 1u) r *= b;
        b *= b;
    }
    return r;
}

// Adam's bias corrections for step t: {lr / (1 - b1^t) as float, sqrt(1 - b2^t) as float}.  They depend on the step counter the
// gradient kernel has just bumped, so the reduce kernel computes them after its wait, in ONE thread per block whose result the
// others pick up from shared memory: the powers by squaring keep that chain short.
struct AdamBias { float step_size, bc2_sqrt; };
__device__ __forceinline__ AdamBias adam_bias(int t, double lr) {
    const double b1 = 0.9, b2 = 0.999;
    const double bc1 = 1.0 - pow_uint(b1, (unsigned)t), bc2 = 1.0 - pow_uint(b2, (unsigned)t);
    AdamBias a;
    a.step_size = (float)(lr / bc1);
    a.bc2_sqrt = (float)sqrt(bc2);
    return a;
}
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, const AdamBias& a) {
    const double b1 = 0.9, b2 = 0.999;
    const float mi = m + (g - m) * (float)(1.0 - b1);
    const float vi = v * (float)b2 + (float)(1.0 - b2) * g * g;
    m = mi;
    v = vi;
    p = p - a.step_size * (mi / (sqrtf(vi) / a.bc2_sqrt + 1e-8f));
}

constexpr int kReduceSlices = 32;


// Adam operands of entry i of agent n (zero where the entry is not stepped).  Loaded right after the kernel's wait, together with
// the partial rows, so that their memory round trip (from HBM when the cache is cold) is not a second one after the sum.
struct AdamIn { float p, m, v, accum; };
__device__ __forceinline__ AdamIn load_adam_in(const ReduceArgs& R, int n, int i) {
    AdamIn a = {0.f, 0.f, 0.f, 0.f};
    if (R.apply_adam && i < R.P) {
        const int64_t k = (int64_t)n * R.P + i;
        a.p = R.params[k];
        a.m = R.m[k];
        a.v = R.v[k];
        if (R.grad_accum) a.accum = R.grad_accum[k];
    }
    return a;
}

// what happens to entry i of agent n once its sum s is known; `in` = load_adam_in(R, n, i)
__device__ __forceinline__ void finish_entry(const ReduceArgs& R, int n, int i, float s, const AdamBias& bias, const AdamIn& in) {
    const int P = R.P;
    if (R.from_partials) {
        if (i == P) s *= R.loss_scale;
        R.grad[(int64_t)n * (P + 1) + i] = s;
    }
    if (i == P) {
        R.loss_out[n] = s;
    } else if (R.apply_adam) {
        const int64_t k = (int64_t)n * P + i;
        float g = s;
        if (R.grad_accum) {                  // the reference's actor never zeroes its gradients (Q2)
            g += in.accum;
            R.grad_accum[k] = g;
        }
        float p = in.p, m = in.m, v = in.v;
        adam_update(p, m, v, g, bias);
        R.params[k] = p;
        R.m[k] = m;
        R.v[k] = v;
    }
}

}  // namespace ia2c
