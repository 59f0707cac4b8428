// a2c.cu — the native trainer of a2c_org_test.py:43-92: one update of R independent runs x E envs in four launches.
//
// The loop is a single joint agent (9 actions) on Org with no reset after construction and no TimeLimit (SURVEY.md Q6), the
// stored pair is (post-step observation, action taken) (Q4), masks are 0 so the critic target is the reward (Q5), and the
// advantage Q[a] - sum(Q * pi) carries gradient into the actor through pi (Q7).  oracle/a2c_envs.py restates one update for
// E envs (one row per env); tests/test_gpu_a2c.py pins these kernels to it and to the unmodified reference's run.
//
// Kernels in this file (one thread per env, 32 envs per block; grid (ceil(E / 32), R): run r's envs are partitioned as an
// R = 1 call partitions them, so every fixed-order sum is the same sum)
//   a2c_rollout_kernel     T env steps per env: Org step with the pending action, actor forward + sample of the next action
//                          (Philox or injected tape), trajectory stores; the critic gradient of the update's rows rides along
//                          (the critic does not change during the rollout) and is block-reduced into the partials.
//   a2c_actor_grad_kernel  the actor phase over the same rows: Q from the UPDATED critic, V = sum(Q * pi), the policy-gradient
//                          + entropy loss with the Q7 term through V, closed-form backward, partials.
// Between and after them reduce_adam_kernel (trainer.cu) sums each run's partial rows and takes the Adam step (the actor on its
// never-zeroed running sum, Q2).
#include "common.cuh"
#include "mlp_f2.cuh"
#include "reduce.cuh"

namespace ia2c {
int reduce_adam_runs_launch(const ReduceArgs& A, const double* lr_per_net, int nets, cudaStream_t s);   // trainer.cu

namespace {

constexpr int J = IA2C_JOINT_ACTIONS, P = kCriticP;
constexpr int kA2CThreads = 32;                 // envs per block
constexpr uint32_t kStreamA2CAction = 3;        // Philox stream of the A2C action sampler (DESIGN.md §4)
constexpr float kEpsClamp = 1.1920928955078125e-07f;   // torch.finfo(float32).eps: Categorical clamps probs to [eps, 1-eps]

__device__ __forceinline__ void onehot_obs(int prev_cls, int cur_cls, float (&x)[kIn]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x[k] = (k == prev_cls) ? 1.f : 0.f;
        x[3 + k] = (k == cur_cls) ? 1.f : 0.f;
    }
}

// The observation row as the rollout stored it (this launch's predecessor wrote it: L2 path, after the wait).
__device__ __forceinline__ void load_obs6_cg(const float* p, float (&x)[kIn]) {
    const float2* p2 = reinterpret_cast<const float2*>(p);
    const float2 a = __ldcg(p2), b = __ldcg(p2 + 1), c = __ldcg(p2 + 2);
    x[0] = a.x; x[1] = a.y; x[2] = b.x; x[3] = b.y; x[4] = c.x; x[5] = c.y;
}

// Next action from the actor's distribution at observation x: the injected tape's slot, or the inverse CDF at the Philox
// uniform u (drawn off the dependency chain by the caller).
__device__ __forceinline__ int next_action(const float* wa, const float (&x)[kIn], float u, const uint8_t* inj) {
    if (inj) return *inj;
    float2 h1[3], h2[3];
    float p[J];
    fwd_f2<J>(wa, x, h1, h2, p);
    softmax_inplace<J>(p);
    return sample_inverse_cdf<J>(p, u);
}

__device__ __forceinline__ float action_uniform(uint64_t seed, uint32_t update, int slot, int64_t e) {
    return philox_uniform_f32(seed, kStreamA2CAction, update, (uint32_t)slot, (uint64_t)e);
}

__global__ void __launch_bounds__(kA2CThreads) a2c_rollout_kernel(const __grid_constant__ ia2c_a2c_desc d) {
    constexpr int GN = F2<J>::G2;   // 148 floats: the critic gradient and the loss slot
    __shared__ __align__(16) float wa[SmemNet<J>::size];
    __shared__ __align__(16) float wc[SmemNet<J>::size];
    __shared__ float red[(kA2CThreads / 32) * (P + 1)];
    pdl_prologue();
    const int run = blockIdx.y;
    stage_smemnet<J>(wa, d.actor_params + (int64_t)run * P);
    stage_smemnet<J>(wc, d.critic_params + (int64_t)run * P);
    if (blockIdx.x == 0 && threadIdx.x == 0) d.critic_step[run] += 1;
    __syncthreads();
    const int64_t E = d.E, ES = E * d.R;
    const int64_t e = (int64_t)blockIdx.x * kA2CThreads + threadIdx.x;   // env within the run (Philox counter)
    const int T = d.T;
    const float inv_b = 1.f / (float)((int64_t)T * E);
    float2 g2[GN];
#pragma unroll
    for (int i = 0; i < GN; ++i) g2[i] = make_float2(0.f, 0.f);
    float loss = 0.f;
    if (e < E) {
        const int64_t ge = (int64_t)run * E + e;                        // env in the stacked axis
        const uint64_t seed = d.seed[run];
        const uint32_t upd = d.update;
        int s = __ldcg(d.env_state + ge);
        double hist = __ldcg(d.env_hist + ge);
        const uchar2 c2 = __ldcg(reinterpret_cast<const uchar2*>(d.env_cls) + ge);
        int prev_cls = c2.x, cur_cls = c2.y;
        int pending;
        if (upd == 0) {   // a2c_org_test.py:56-60: the first action is drawn from the reset observation
            float x0[kIn];
            onehot_obs(prev_cls, cur_cls, x0);
            pending = next_action(wa, x0, d.inj_actions ? 0.f : action_uniform(seed, upd, 0, e), d.inj_actions ? d.inj_actions + ge : nullptr);
        } else {
            pending = __ldcg(d.pending_action + ge);
        }
        double ret = 0.0;
        float u_next = d.inj_actions ? 0.f : action_uniform(seed, upd, 1, e);
        for (int t = 0; t < T; ++t) {
            // Org.step(pending) (Org.py:51-126): the reference's joint code, two lever counts
            const int a1 = pending / 3, a2 = pending - 3 * (pending / 3);
            int s2;
            double base;
            org_transition(s, (a1 == 0) + (a2 == 0), (a1 == 1) + (a2 == 1), (a1 == 2) + (a2 == 2), 2, s2, base);
            hist = org_reward(base, hist);
            prev_cls = cur_cls;
            cur_cls = org_obs_class(s2);
            s = s2;
            float x[kIn];
            onehot_obs(prev_cls, cur_cls, x);
            // next action from the post-step observation (a2c_org_test.py:69): the chain that bounds the update
            const float u = u_next;
            if (!d.inj_actions && t + 1 < T) u_next = action_uniform(seed, upd, t + 2, e);
            const int nxt = next_action(wa, x, u, d.inj_actions ? d.inj_actions + (int64_t)(t + 1) * ES + ge : nullptr);
            // trajectory (a2c_org_test.py:70-77) and the fp64 return, off the chain
            const float r32 = (float)hist;
            ret += hist;
            const int64_t row = (int64_t)t * ES + ge;
            float2* o2 = reinterpret_cast<float2*>(d.obs + row * kIn);
            o2[0] = make_float2(x[0], x[1]);
            o2[1] = make_float2(x[2], x[3]);
            o2[2] = make_float2(x[4], x[5]);
            d.act[row] = (uint8_t)pending;
            d.reward[row] = r32;
            // critic gradient of this row: target = reward (masks = 0, Q5), L = mean((r - Q(S)[a])^2)
            float2 h1[3], h2[3];
            float q[J];
            fwd_f2<J>(wc, x, h1, h2, q);
            const float delta = r32 - select_out<J>(q, pending);
            loss = fmaf(delta, delta, loss);
            const float gq = -2.f * delta * inv_b;
            const int a = pending;
            bwd_f2<J>(wc, x, h1, h2, [&](int o) { return o == a ? gq : 0.f; }, g2);
            pending = nxt;
        }
        d.env_state[ge] = s;
        d.env_hist[ge] = hist;
        *reinterpret_cast<uchar2*>(d.env_cls + 2 * ge) = make_uchar2((unsigned char)prev_cls, (unsigned char)cur_cls);
        d.env_elapsed[ge] = __ldcg(d.env_elapsed + ge) + T;
        d.pending_action[ge] = (uint8_t)pending;
        d.ep_return[ge] = ret;
    }
    float g[2 * GN];
    unpack_g2(g2, g);
    g[P] = loss;
    block_reduce_store<P + 1>(reinterpret_cast<float(&)[P + 1]>(g), red,
                              d.partials + ((int64_t)run * gridDim.x + blockIdx.x) * (P + 1));
}

__global__ void __launch_bounds__(kA2CThreads) a2c_actor_grad_kernel(const __grid_constant__ ia2c_a2c_desc d) {
    constexpr int GN = F2<J>::G2;
    __shared__ __align__(16) float wa[SmemNet<J>::size];
    __shared__ __align__(16) float wc[SmemNet<J>::size];
    __shared__ float red[(kA2CThreads / 32) * (P + 1)];
    pdl_prologue();
    const int run = blockIdx.y;
    stage_smemnet<J>(wa, d.actor_params + (int64_t)run * P);
    stage_smemnet<J>(wc, d.critic_params + (int64_t)run * P);   // updated by the critic's reduce + Adam
    if (blockIdx.x == 0 && threadIdx.x == 0) d.actor_step[run] += 1;
    __syncthreads();
    const int64_t E = d.E, ES = E * d.R;
    const int64_t e = (int64_t)blockIdx.x * kA2CThreads + threadIdx.x;
    const int T = d.T;
    const float inv_b = 1.f / (float)((int64_t)T * E);
    const float beta = d.beta_run ? d.beta_run[run] : d.beta;
    float2 g2[GN];
#pragma unroll
    for (int i = 0; i < GN; ++i) g2[i] = make_float2(0.f, 0.f);
    float loss = 0.f;
    if (e < E) {
        const int64_t ge = (int64_t)run * E + e;
        for (int t = 0; t < T; ++t) {
            const int64_t row = (int64_t)t * ES + ge;
            float x[kIn];
            load_obs6_cg(d.obs + row * kIn, x);
            const int a = __ldcg(d.act + row);
            float q[J];
            {
                float2 h1[3], h2[3];
                fwd_f2<J>(wc, x, h1, h2, q);   // Q(S) of the updated critic, no gradient (a2c_org_test.py:86)
            }
            float2 h1[3], h2[3];
            float p[J];
            fwd_f2<J>(wa, x, h1, h2, p);
            softmax_inplace<J>(p);               // d = actor.action_distribution(S, grad=True) (a2c_org_test.py:87)
            float V = 0.f;
#pragma unroll
            for (int o = 0; o < J; ++o) V = fmaf(q[o], p[o], V);
            const float adv = select_out<J>(q, a) - V;   // Q_cur - V, differentiable through d (Q7)
            // Categorical(probs=d): qv = d / sum(d); logit = log(clamp(qv)); loss_row = adv * (-logit[a]) - beta * H
            float sp = 0.f;
#pragma unroll
            for (int o = 0; o < J; ++o) sp += p[o];
            float ent = 0.f, qg = 0.f, neglogp = 0.f, gqv[J], qq[J];
#pragma unroll
            for (int o = 0; o < J; ++o) {
                const float qv = p[o] / sp;
                const bool inside = (qv >= kEpsClamp) && (qv <= 1.f - kEpsClamp);
                const float logit = logf(fminf(fmaxf(qv, kEpsClamp), 1.f - kEpsClamp));
                ent -= logit * qv;
                float go = beta * (logit + (inside ? 1.f : 0.f));
                if (o == a) {
                    neglogp = -logit;
                    if (inside) go -= adv / qv;
                }
                gqv[o] = go;
                qq[o] = qv;
                qg = fmaf(qv, go, qg);
            }
            loss += adv * neglogp - beta * ent;
            // dL/dy: the policy-gradient + entropy term through normalise + softmax, plus the advantage's own gradient
            // dL/dadv * dadv/dy_o = (neglogp / B) * (-d_o (Q_o - V))
            float dy[J];
#pragma unroll
            for (int o = 0; o < J; ++o) dy[o] = (qq[o] * (gqv[o] - qg) - neglogp * p[o] * (q[o] - V)) * inv_b;
            bwd_f2<J>(wa, x, h1, h2, [&](int o) { return dy[o]; }, g2);
        }
    }
    float g[2 * GN];
    unpack_g2(g2, g);
    g[P] = loss;
    block_reduce_store<P + 1>(reinterpret_cast<float(&)[P + 1]>(g), red,
                              d.partials + ((int64_t)run * gridDim.x + blockIdx.x) * (P + 1));
}

int64_t a2c_blocks_per_run(int64_t E) { return (E + kA2CThreads - 1) / kA2CThreads; }

ReduceArgs a2c_reduce_args(const ia2c_a2c_desc& d, int which) {
    ReduceArgs A;
    A.partials = d.partials;
    A.n_blocks = (int)a2c_blocks_per_run(d.E);
    A.P = P;
    A.grad = which == 0 ? d.critic_grad : d.actor_grad;
    A.grad_accum = which == 0 ? nullptr : d.actor_grad_accum;   // the actor never zeroes its gradient (Q2)
    A.params = which == 0 ? d.critic_params : d.actor_params;
    A.m = which == 0 ? d.critic_m : d.actor_m;
    A.v = which == 0 ? d.critic_v : d.actor_v;
    A.step = which == 0 ? d.critic_step : d.actor_step;
    A.loss_out = d.loss_out + (which == 0 ? 0 : d.R);
    A.loss_scale = 1.f / (float)((int64_t)d.T * d.E);
    A.lr = which == 0 ? d.lr_critic : d.lr_actor;
    A.apply_adam = 1;
    A.from_partials = 1;
    return A;
}

int validate_a2c(const ia2c_a2c_desc* d, const char* who) {
    IA2C_REQUIRE(d != nullptr, "%s: null descriptor", who);
    IA2C_REQUIRE(d->R >= 1 && d->R <= IA2C_A2C_MAX_RUNS, "%s: R=%d outside 1..%d", who, d->R, IA2C_A2C_MAX_RUNS);
    IA2C_REQUIRE(d->E >= 1 && d->E <= IA2C_A2C_MAX_ENVS, "%s: E=%lld outside 1..%d", who, (long long)d->E, IA2C_A2C_MAX_ENVS);
    IA2C_REQUIRE((int64_t)d->R * d->E <= IA2C_A2C_MAX_ENVS, "%s: R * E = %lld above %d", who, (long long)d->R * d->E,
                 IA2C_A2C_MAX_ENVS);
    IA2C_REQUIRE(d->T >= 1 && d->T <= IA2C_A2C_MAX_STEPS, "%s: T=%d outside 1..%d", who, d->T, IA2C_A2C_MAX_STEPS);
    IA2C_REQUIRE(d->seed != nullptr, "%s: null seed array (one Philox key per run)", who);
    IA2C_REQUIRE(d->actor_params && d->actor_grad && d->actor_grad_accum && d->actor_m && d->actor_v && d->actor_step &&
                     d->critic_params && d->critic_grad && d->critic_m && d->critic_v && d->critic_step && d->loss_out,
                 "%s: null network/optimiser pointer", who);
    IA2C_REQUIRE(d->env_state && d->env_hist && d->env_cls && d->env_elapsed && d->pending_action && d->ep_return,
                 "%s: null env pointer", who);
    IA2C_REQUIRE(d->obs && d->act && d->reward, "%s: null trajectory pointer", who);
    IA2C_REQUIRE(d->partials && d->partials_floats >= ia2c_a2c_partials_floats(d), "%s: partials workspace too small (%zu < %zu)",
                 who, d->partials_floats, ia2c_a2c_partials_floats(d));
    return 0;
}

}  // namespace
}  // namespace ia2c

using namespace ia2c;

extern "C" size_t ia2c_a2c_partials_floats(const ia2c_a2c_desc* d) {
    if (d == nullptr || d->R < 1 || d->E < 1) return 0;
    return (size_t)d->R * (size_t)a2c_blocks_per_run(d->E) * (size_t)(P + 1);
}

extern "C" int ia2c_a2c_train_update(const ia2c_a2c_desc* d, void* stream) {
    if (int rc = validate_a2c(d, "ia2c_a2c_train_update")) return rc;
    cudaStream_t s = as_stream(stream);
    const dim3 grid((unsigned)a2c_blocks_per_run(d->E), (unsigned)d->R);
    if (int rc = launch_pdl("a2c_rollout_kernel", a2c_rollout_kernel, grid, dim3(kA2CThreads), 0, s, *d)) return rc;
    if (int rc = reduce_adam_runs_launch(a2c_reduce_args(*d, 0), d->lr_critic_run, d->R, s)) return rc;
    if (int rc = launch_pdl("a2c_actor_grad_kernel", a2c_actor_grad_kernel, grid, dim3(kA2CThreads), 0, s, *d)) return rc;
    return reduce_adam_runs_launch(a2c_reduce_args(*d, 1), d->lr_actor_run, d->R, s);
}
