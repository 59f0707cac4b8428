// trainer.cu — the fused IA2C episode: rollout, critic phase, actor phase (N agents, E envs).
//
// Replaces the episode body of ia2c.py:62-129:
//   rollout        ia2c.py:72-102   (env step, 2N actor forwards + samples, belief updates, trajectory)
//   critic phase   ia2c.py:104-114  (+ CriticNetwork.batch_update, ac_nets.py:62-72)
//   actor phase    ia2c.py:116-129  (+ ActorNetwork.batch_update, ac_nets.py:112-119, no zero_grad)
// generalised from 2 to N agents as specified in DESIGN.md ("Org-N"; identical to the reference at N=2).
//
// Kernels in this file
//   env_step_kernel        one Org step for all envs (general N): action counts of step t-1 reduced by warp shuffles
//                          (agents in lanes) -> true-partner mode, transition, reward, observation classes.
//   actor_step_kernel      every agent's actor forward + sample -> act[t]; block = one agent x a strip of envs, the
//                          agent's weights warp-uniform in registers (FFMA2).  (N <= 8 uses the persistent pipelined
//                          kernel of rollout_fused.cu instead of these two.)
//   critic_grad_kernel     a thread walks a time chunk of one (agent, env): ONE critic forward and ONE backward per
//                          observation (TD target with gradient through both passes: residual gradient, SURVEY.md
//                          Q8), FFMA2 math, accumulators in registers, block-reduced to partials (fixed order).
//                          Skipped when the fused rollout already produced the critic partials.
//   actor_grad_kernel      same walk: advantage from the updated critic, actor forward, Categorical
//                          log-prob/entropy loss, closed-form backward, partials.  (Many-agent configs use the
//                          warp-specialised actor_pipe_kernel of actor_pipe.cu; IA2C_FLAG_ACTOR_COLUMNS selects.)
//   reduce_adam_kernel     sums the partials, writes grad (+loss), applies Adam (actor: accumulating gradient
//                          buffer, SURVEY.md Q2).
//   allreduce_adam_kernel  multi-GPU: the same plus the gradient exchange over NVLink peer memory, in one kernel.
// The belief update between steps is belief_pairs(_table)_kernel (belief.cu).
#include <algorithm>
#include <chrono>
#include <cstdlib>

#include "common.cuh"
#include "mlp_f2.cuh"
#include "reduce.cuh"

namespace ia2c {
int rollout_fused_supported(int N, int M);                                  // rollout_fused.cu
int rollout_fused_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, const EnvPartners* p, cudaStream_t s);
int64_t rollout_fused_blocks(int64_t E, int N);
int actor_pipe_launch(const ia2c_episode_desc* d, cudaStream_t s);
int reduce_adam_runs_launch(const ReduceArgs& A, const double* lr_per_net, int nets, cudaStream_t s);   // used by a2c.cu
int64_t actor_pipe_blocks(int64_t E, int N);
int belief_pairs_episode_runs_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, cudaStream_t s);   // belief.cu
int validate_env_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p, const char* who);   // partners.cu
EnvPartners env_partners_arg(const ia2c_env_partner_desc* p);

namespace {

constexpr int F = IA2C_OBS_FEATURES, A = IA2C_AGENT_ACTIONS, J = IA2C_JOINT_ACTIONS;
constexpr int kRolloutThreads = 128;
constexpr int kGradThreads = 128;
#ifdef IA2C_STAGE_CLOCKS
// diagnostic build only: stamps of the update kernels of the LAST episode (0-3 critic reduce / exchange: left the wait, local
// reduction done, all ranks' words in, block 0 done; 4-7 actor gradient: entry, left the wait, rows done, block 0 done;
// 10-13 actor reduce / exchange).  Read back with ia2c_debug_kclocks.
__device__ unsigned long long g_kclock[16];
#endif
constexpr float kEpsClamp = 1.1920928955078125e-07f;

__device__ __forceinline__ int mode3(int c0, int c1, int c2) {
    int best = 0, bc = c0;
    if (c1 > bc) { best = 1; bc = c1; }
    if (c2 > bc) { best = 2; }
    return best;
}

// joint index for agent i: lower agent index is the high digit, partner (i+1) mod N (SURVEY.md Q9)
__device__ __forceinline__ int joint_index(int i, int n, int own, int other) {
    return (i < (i + 1) % n) ? own * A + other : other * A + own;
}

// ------------------------------------------------------------------------------------------------
struct StepArgs {
    ia2c_episode_desc d;
    int t;
    int G;   // lanes per env (power of two, min(32, pow2ceil(N)))
};

__device__ __forceinline__ uint32_t pack_count(int a) { return a == 0 ? 1u : (a == 1 ? (1u << 10) : (1u << 20)); }

// env_step_kernel, step t in 0..T+1: G lanes per env.  t == 0 resets; 1 <= t <= T counts the actions of step t-1
// (agents strided over the group's lanes, counts reduced by shuffles), writes partner_true[t-1] (mode of the OTHERS'
// actions) and advances the env; t == T+1 only writes partner_true[T].
__global__ void __launch_bounds__(kRolloutThreads) env_step_kernel(StepArgs S) {
    pdl_prologue();
    const ia2c_episode_desc& d = S.d;
    const int N = d.N, G = S.G, t = S.t;
    const int lane = threadIdx.x & 31;
    const int sub = lane & (G - 1);
    const int epw = 32 / G;                                        // envs per warp
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t e = warp_global * epw + (lane / G);
    const bool live = e < d.E;                                     // whole group shares this
    const int64_t E = d.E;

    int prev_cls = 1, cur_cls = 1;
    if (t > 0) {
        uint32_t packed = 0;
        const uint8_t* a_prev = d.act + ((int64_t)(t - 1) * E + (live ? e : 0)) * N;
        if (live) {
            for (int i = sub; i < N; i += G) packed += pack_count(a_prev[i]);
        }
        for (int off = G >> 1; off > 0; off >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, off);
        const int c0 = packed & 1023, c1 = (packed >> 10) & 1023, c2 = (packed >> 20) & 1023;
        if (live) {
            uint8_t* pt = d.partner_true + ((int64_t)(t - 1) * E + e) * N;
            for (int i = sub; i < N; i += G) {
                const int a = a_prev[i];
                pt[i] = (uint8_t)mode3(c0 - (a == 0), c1 - (a == 1), c2 - (a == 2));
            }
        }
        if (t > d.T) return;
        if (live && sub == 0) {
            const int s = d.env_state[e];
            int s2;
            double base;
            org_transition(s, c0, c1, c2, N, s2, base);
            double r = org_reward(base, d.env_hist[e]);
            prev_cls = d.env_cls[2 * e + 1];
            cur_cls = org_obs_class(s2);
            d.reward[(int64_t)(t - 1) * E + e] = (float)r;         // float32(r) as stored by ia2c.py:99
            d.ep_return[e] += r;                                   // fp64, in step order (ia2c.py:102)
            if (d.state_trace) d.state_trace[(int64_t)(t - 1) * E + e] = s2;
            if (d.reward_f64) d.reward_f64[(int64_t)(t - 1) * E + e] = r;
            int el = d.env_elapsed[e] + 1;
            if (d.max_episode_steps > 0 && el >= d.max_episode_steps) {  // same-step autoreset (Q14)
                s2 = 2; r = 0.0; prev_cls = 1; cur_cls = 1; el = 0;
            }
            d.env_state[e] = s2;
            d.env_hist[e] = r;
            d.env_elapsed[e] = el;
            *reinterpret_cast<uchar2*>(d.env_cls + 2 * e) = make_uchar2((unsigned char)prev_cls, (unsigned char)cur_cls);
        }
    } else if (live && sub == 0) {
        d.env_state[e] = 2;
        d.env_hist[e] = 0.0;
        d.env_elapsed[e] = 0;
        d.ep_return[e] = 0.0;
        *reinterpret_cast<uchar2*>(d.env_cls + 2 * e) = make_uchar2(1, 1);
    }
    const int leader = lane & ~(G - 1);
    prev_cls = __shfl_sync(0xffffffffu, prev_cls, leader);
    cur_cls = __shfl_sync(0xffffffffu, cur_cls, leader);
    if (live && sub < F) {
        for (int k = sub; k < F; k += G)
            d.obs[((int64_t)t * E + e) * F + k] = (k < 3 ? k == prev_cls : k - 3 == cur_cls) ? 1.f : 0.f;
    }
}

// actor_step_kernel, step t in 0..T: every agent's actor forward + sample (ac_nets.py:94-102).  Block = one agent
// (blockIdx.y) x a strip of envs, lane = env: the agent's weights are warp-uniform and live in registers (FFMA2,
// mlp_f2.cuh), each thread walks up to kActorEnvsPerThread envs.
constexpr int kActorThreads = 256, kActorEnvsPerThread = 4;
__global__ void __launch_bounds__(kActorThreads) actor_step_kernel(StepArgs S) {
    pdl_prologue();
    const ia2c_episode_desc& d = S.d;
    const int N = d.N, t = S.t, i = blockIdx.y;
    const int64_t E = d.E;
    RegNet<A> net;
    if (!d.inj_actions) load_regnet<A>(net, d.actor_params + (int64_t)i * kActorP);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = ((int64_t)t * E + e) * N + i;
        int a;
        if (d.inj_actions) {
            a = d.inj_actions[row];
        } else {
            const uchar2 cls = *reinterpret_cast<const uchar2*>(d.env_cls + 2 * e);
            float x[F], y[A];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                x[k] = (k == cls.x) ? 1.f : 0.f;
                x[3 + k] = (k == cls.y) ? 1.f : 0.f;
            }
            forward_regnet<A>(net, x, y);
            softmax_inplace<A>(y);
            const float u = d.inj_u_action ? d.inj_u_action[row]
                                           : philox_uniform_f32(d.seed, kStreamAction, d.episode, (uint32_t)t,
                                                                (uint64_t)((d.env_offset + e) * N + i));
            a = sample_inverse_cdf<A>(y, u);
        }
        d.act[row] = (uint8_t)a;
    }
}

// rollout_many_kernel (9 <= N <= 256): the T+1 env / actor steps of an episode in ONE persistent launch instead of 2(T+1)
// launches of env_step_kernel / actor_step_kernel — same functions, same order of operations, same Philox counters, so the
// trajectory bytes are identical.  Envs are independent: a block owns a chunk of envs for the whole episode, thread = agent
// (its actor in registers, FFMA2), and a step is
//   (1) every agent samples its action for each env of the chunk; per-warp action counts by ballots;
//   (2) the chunk's first threads (one per env) total the counts, advance the env (transition, fp64 reward recurrence,
//       same-step autoreset) and publish the next observation classes;
//   (3) every agent derives the mode of the OTHERS' actions (partner_true)
// with two block barriers per step.  The belief update of the whole episode follows as one kernel (belief.cu).
// RUNS: a batch of independent runs (ia2c_train_episode_runs_many), blockIdx.y = run.  A block's chunk lies inside one run (its
// threads hold that run's actors, rows run * N + i); the run's envs are columns [run * E, (run + 1) * E) of an env axis of
// length R * E (stride ES), and `e` stays the env's index within its run, which keys its Philox counters.
// PARTNERS: frozen partners per env (ia2c_train_episode_env_partners).  The chunk's owner threads draw their envs' teams into
// shared memory and log them; a partner-seat thread samples from its env's pool row of the policy table (Org has 9 observation
// classes; the table holds what forward_regnet + softmax_inplace compute, so the samples are those of the row's actor).
constexpr int kManyMaxEnvs = 32;     // envs per block
template <bool RUNS, bool PARTNERS = false>
__global__ void __launch_bounds__(256) rollout_many_kernel(const __grid_constant__ ia2c_episode_desc d, int envs_per_block, RunsArg<RUNS> ra,
                                                           const __grid_constant__ PartnerArg<PARTNERS> pa) {
    extern __shared__ __align__(16) unsigned char many_smem[];
    const int N = d.N, T = d.T, i = threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int64_t E = d.E, e0 = (int64_t)blockIdx.x * envs_per_block;
    const int run = RUNS ? (int)blockIdx.y : 0;
    const int64_t ES = RUNS ? E * gridDim.y : E, g0 = RUNS ? (int64_t)run * E + e0 : e0;   // g0: the chunk's first column
    const int EC = (int)min((int64_t)envs_per_block, E - e0);
    uint32_t* warp_cnt = reinterpret_cast<uint32_t*>(many_smem);                 // [EC][n_warps] packed 3 x 10 bits
    uint32_t* tot_cnt = warp_cnt + kManyMaxEnvs * 8;                              // [EC]
    int* cls_s = reinterpret_cast<int*>(tot_cnt + kManyMaxEnvs);                  // [EC] prev | cur << 2
    uint8_t* act_s = reinterpret_cast<uint8_t*>(cls_s + kManyMaxEnvs);            // [EC][blockDim]
    pdl_prologue();
    const bool agent = i < N;
    RegNet<A> net;
    if (agent && !d.inj_actions) load_regnet<A>(net, d.actor_params + (int64_t)(RUNS ? run * N + i : i) * kActorP);
    // env state of env el lives in the registers of thread el
    int s = 2, prev_cls = 1, cur_cls = 1, elapsed = 0;
    double hist = 0.0, ep_ret = 0.0;
    const bool owner = i < EC;
    __shared__ int team_s[PARTNERS ? kManyMaxEnvs : 1];
    int slot = -1;   // this agent's partner-seat slot
    const int32_t* partner_teams = nullptr;
    const float* partner_policy = nullptr;
    int partner_S = 0;
    auto team_of = [&](int el) { return PARTNERS ? team_s[el] : -1; };
    if constexpr (PARTNERS) {
        partner_teams = pa.teams, partner_policy = pa.policy, partner_S = pa.S;
        if (owner) {
            team_s[i] = env_team(pa, run_seed<RUNS>(d, ra, run), d.episode, e0 + i, N);
            pa.log[g0 + i] = team_s[i];
        }
        if (agent) slot = env_partner_slot(pa, i);
    }
    if (owner) {
        cls_s[i] = 1 | (1 << 2);
        float* o = d.obs + (g0 + i) * F;
#pragma unroll
        for (int k = 0; k < F; ++k) o[k] = (k == 1 || k == 4) ? 1.f : 0.f;        // reset observation [0,1,0,0,1,0] (Org.py:128-148)
    }
    __syncthreads();
    for (int t = 0; t <= T; ++t) {
        // ---- (1) actions of step t
        for (int el = 0; el < EC; ++el) {
            const int64_t e = e0 + el;
            int a = 3;   // no action (threads beyond N)
            if (agent) {
                const int64_t row = ((int64_t)t * ES + (RUNS ? g0 + el : e)) * N + i;
                if (d.inj_actions) {
                    a = d.inj_actions[row];
                } else {
                    const int packed = cls_s[el];
                    float y[A];
                    if (PARTNERS && slot >= 0 && team_of(el) >= 0) {
                        const int64_t row = __ldcg(partner_teams + (int64_t)team_of(el) * partner_S + slot);
                        const float* pr = partner_policy + (row * 9 + 3 * (packed & 3) + (packed >> 2)) * A;
#pragma unroll
                        for (int k = 0; k < A; ++k) y[k] = __ldcg(pr + k);
                    } else {
                        float x[F];
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            x[k] = (k == (packed & 3)) ? 1.f : 0.f;
                            x[3 + k] = (k == (packed >> 2)) ? 1.f : 0.f;
                        }
                        forward_regnet<A>(net, x, y);
                        softmax_inplace<A>(y);
                    }
                    const float u = d.inj_u_action ? d.inj_u_action[row]
                                                   : philox_uniform_f32(run_seed<RUNS>(d, ra, run), kStreamAction, d.episode, (uint32_t)t,
                                                                        (uint64_t)((d.env_offset + e) * N + i));
                    a = sample_inverse_cdf<A>(y, u);
                }
                d.act[row] = (uint8_t)a;
            }
            act_s[el * blockDim.x + i] = (uint8_t)a;
            const uint32_t c0 = __popc(__ballot_sync(0xffffffffu, a == 0)), c1 = __popc(__ballot_sync(0xffffffffu, a == 1)),
                           c2 = __popc(__ballot_sync(0xffffffffu, a == 2));
            if (lane == 0) warp_cnt[el * 8 + warp] = c0 | (c1 << 10) | (c2 << 20);
        }
        __syncthreads();
        // ---- (2) totals, env transition (steps 0..T-1 advance the env; after step T only partner_true[T] is due)
        if (owner) {
            uint32_t packed = 0u;
            for (int w = 0; w < n_warps; ++w) packed += warp_cnt[i * 8 + w];
            tot_cnt[i] = packed;
            if (t < T) {
                const int64_t e = g0 + i;
                const int c0 = packed & 1023, c1 = (packed >> 10) & 1023, c2 = (packed >> 20) & 1023;
                int s2;
                double base;
                org_transition(s, c0, c1, c2, N, s2, base);
                double r = org_reward(base, hist);
                prev_cls = cur_cls;
                cur_cls = org_obs_class(s2);
                d.reward[(int64_t)t * ES + e] = (float)r;         // float32(r) as stored by ia2c.py:99
                ep_ret += r;                                     // fp64, in step order (ia2c.py:102)
                if (d.state_trace) d.state_trace[(int64_t)t * ES + e] = s2;
                if (d.reward_f64) d.reward_f64[(int64_t)t * ES + e] = r;
                ++elapsed;
                if (d.max_episode_steps > 0 && elapsed >= d.max_episode_steps) {   // same-step autoreset (Q14)
                    s2 = 2; r = 0.0; prev_cls = 1; cur_cls = 1; elapsed = 0;
                }
                s = s2;
                hist = r;
                cls_s[i] = prev_cls | (cur_cls << 2);
                float* o = d.obs + ((int64_t)(t + 1) * ES + e) * F;
#pragma unroll
                for (int k = 0; k < F; ++k) o[k] = (k < 3 ? k == prev_cls : k - 3 == cur_cls) ? 1.f : 0.f;
            }
        }
        __syncthreads();
        // ---- (3) mode of the others' actions at step t
        if (agent) {
            for (int el = 0; el < EC; ++el) {
                const uint32_t packed = tot_cnt[el];
                const int a = act_s[el * blockDim.x + i];
                const int c0 = packed & 1023, c1 = (packed >> 10) & 1023, c2 = (packed >> 20) & 1023;
                d.partner_true[((int64_t)t * ES + g0 + el) * N + i] = (uint8_t)mode3(c0 - (a == 0), c1 - (a == 1), c2 - (a == 2));
            }
        }
        // (the next step's writes to warp_cnt / act_s come after these reads only per thread for act_s — own entries — and after
        //  the next barrier for tot_cnt; warp_cnt is rewritten before that barrier but was last read before this step's second one)
    }
    if (owner) {   // persist the final env state exactly as the per-step path leaves it
        const int64_t e = g0 + i;
        d.env_state[e] = s;
        d.env_hist[e] = hist;
        d.env_elapsed[e] = elapsed;
        d.ep_return[e] = ep_ret;
        *reinterpret_cast<uchar2*>(d.env_cls + 2 * e) = make_uchar2((unsigned char)prev_cls, (unsigned char)cur_cls);
    }
}

// ---- gradient kernels: one thread per (agent, env, time chunk), packed fp32 math (mlp_f2.cuh) ----------
// next_obs[t] IS obs[t+1] (trajectory layout), so a thread that walks a chunk [t0,t1) of one env's
// time axis evaluates the critic ONCE per observation (L+1 forwards for L rows instead of 2L) and, in the
// critic phase, back-propagates ONCE per observation with the two output-gradient contributions it
// receives — as Q(obs_t)[jt_t] of row t and as the bootstrap Q(next_obs_{t-1})[nja_{t-1}] of row t-1 —
// added together first (L+1 backward passes instead of 2L).  Same sums, fewer passes.
struct ChunkPlan { int chunk_len, n_chunks; };
__host__ __device__ inline ChunkPlan chunk_plan(int T, int64_t E, int N) {
    // enough (env, chunk) items per agent for one resident wave of 148 SMs x 2 blocks x 128 threads over N agents
    const int64_t target = (int64_t)kSMs * 2 * 128;
    int64_t c = target / (E * N);   // floor: all items must fit in ONE pass of the resident wave
    if (c < 1) c = 1;
    if (c > T) c = T;
    ChunkPlan p;
    p.chunk_len = (int)((T + c - 1) / c);
    p.n_chunks = (T + p.chunk_len - 1) / p.chunk_len;
    return p;
}

// partial row layout: P gradient entries then the loss partial.
// RUNS: a batch of independent runs (ia2c_train_episode_runs_many), laid out as actor_grad_kernel<true> lays them out:
// blockIdx.y = run * N + agent is the net row, the run's envs are columns [run * E, (run + 1) * E) of an env axis of length R * E.
template <bool RUNS>
__global__ void __launch_bounds__(kGradThreads) critic_grad_kernel(ia2c_episode_desc d, float* __restrict__ partials, RunsArg<RUNS> ra) {
    constexpr int P = kCriticP, GN = F2<J>::G2;   // 148 floats = 74 float2
    __shared__ __align__(16) float w[SmemNet<J>::size];
    __shared__ float red[(kGradThreads / 32) * (P + 1)];
    pdl_prologue();
    const int N = d.N, n = RUNS ? (int)blockIdx.y % N : blockIdx.y;   // n: the agent
    const int run = RUNS ? (int)blockIdx.y / N : 0;
    stage_smemnet<J>(w, d.critic_params + (int64_t)(RUNS ? blockIdx.y : n) * P);
    if (blockIdx.x == 0 && threadIdx.x == 0 && !(d.flags & IA2C_FLAG_SKIP_ADAM)) d.critic_step[RUNS ? blockIdx.y : n] += 1;
    __syncthreads();
    const int64_t E = d.E, rows = (int64_t)d.T * E;
    const int64_t ES = RUNS ? E * (gridDim.y / N) : E;
    const ChunkPlan cp = chunk_plan(d.T, E, N);
    const int64_t items = E * cp.n_chunks;
    const float inv_b = 1.f / (float)((int64_t)d.T * d.E_total);
    float2 g2[GN];
#pragma unroll
    for (int i = 0; i < GN; ++i) g2[i] = make_float2(0.f, 0.f);
    float loss = 0.f;
    for (int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = RUNS ? (int64_t)run * E + item % E : item % E;
        const int t0 = (int)(item / E) * cp.chunk_len;
        const int t1 = min(d.T, t0 + cp.chunk_len);
        float x[kIn], q[J];
        float2 h1[3], h2[3];
        load_obs6(d.obs + ((int64_t)t0 * ES + e) * kIn, x);
        fwd_f2<J>(w, x, h1, h2, q);
        int carry_idx = -1;          // pending bootstrap gradient for the CURRENT observation (from row t-1)
        float carry_val = 0.f;
        for (int t = t0; t < t1; ++t) {
            const int64_t r = (int64_t)t * ES + e;
            float xn[kIn], qn[J];
            float2 h1n[3], h2n[3];
            load_obs6(d.obs + (r + ES) * kIn, xn);                   // next_obs[t] = obs[t+1]
            fwd_f2<J>(w, xn, h1n, h2n, qn);
            const int own = d.act[r * N + n], own_n = d.act[(r + ES) * N + n];
            const int jt = joint_index(n, N, own, d.partner_true[r * N + n]);            // ia2c.py:112
            const int nja = joint_index(n, N, own_n, d.partner_pred[(r + ES) * N + n]);  // ia2c.py:104-105
            // RUNS spells out, with rounding intrinsics, what nvcc 12.9 makes of the standalone instantiation (read off its SASS:
            // FFMA for reward + gamma * Q', FMULs rounding 2 * gamma * delta and then * inv_b): with gamma loaded per run the
            // compiler may contract differently, and the batch's runs would drift from the standalone runs in the last bit.
            const float gamma = run_gamma<RUNS>(d, ra, run);
            const float target = RUNS ? __fmaf_rn(gamma, select_out<J>(qn, nja), d.reward[r])
                                      : d.reward[r] + gamma * select_out<J>(qn, nja);   // ia2c.py:110 (Q8)
            const float delta = target - select_out<J>(q, jt);
            if (d.target_dump) d.target_dump[(int64_t)n * rows + r] = target;   // never in a batch (refused)
            loss = fmaf(delta, delta, loss);
            const float gq = RUNS ? __fmul_rn(-2.f * delta, inv_b) : -2.f * delta * inv_b;   // dL/dQ(obs_t)[jt]
            bwd_f2<J>(w, x, h1, h2, [&](int o) { return (o == jt ? gq : 0.f) + (o == carry_idx ? carry_val : 0.f); }, g2);
            carry_idx = nja;
            carry_val = RUNS ? __fmul_rn(__fmul_rn(2.f * gamma, delta), inv_b)   // dL/dQ(next_obs_t)[nja]: residual gradient
                             : 2.f * gamma * delta * inv_b;
#pragma unroll
            for (int k = 0; k < kIn; ++k) x[k] = xn[k];
#pragma unroll
            for (int k = 0; k < 3; ++k) { h1[k] = h1n[k]; h2[k] = h2n[k]; }
#pragma unroll
            for (int o = 0; o < J; ++o) q[o] = qn[o];
        }
        bwd_f2<J>(w, x, h1, h2, [&](int o) { return o == carry_idx ? carry_val : 0.f; }, g2);
    }
    float g[2 * GN];
    unpack_g2(g2, g);
    g[P] = loss;
    block_reduce_store<P + 1>(reinterpret_cast<float(&)[P + 1]>(g), red, partials + ((int64_t)(RUNS ? blockIdx.y : n) * gridDim.x + blockIdx.x) * (P + 1));
}

// RUNS: a batch of independent runs (ia2c_train_episode_runs): blockIdx.y = run * N + agent is the net row, the run's envs are
// columns [run * E, (run + 1) * E) of an env axis of length R * E (stride ES).
template <bool RUNS>
__global__ void __launch_bounds__(kGradThreads) actor_grad_kernel(ia2c_episode_desc d, float* __restrict__ partials, RunsArg<RUNS> ra) {
    constexpr int P = kActorP, PC = kCriticP, GN = F2<A>::G2;   // 106 floats = 53 float2
    __shared__ __align__(16) float wc[SmemNet<J>::size];
    __shared__ __align__(16) float w[SmemNet<A>::size];
    __shared__ float red[(kGradThreads / 32) * (P + 1)];
    KCLOCK(k_entry);
    KSTAMP(g_kclock, 4);
    pdl_prologue();
    KCLOCK(k_waited);
    KSTAMP(g_kclock, 5);
    const int N = d.N, n = RUNS ? (int)blockIdx.y % N : blockIdx.y;   // n: the agent
    const int run = RUNS ? (int)blockIdx.y / N : 0;
    stage_smemnet<J>(wc, d.critic_params + (int64_t)(RUNS ? blockIdx.y : n) * PC);
    stage_smemnet<A>(w, d.actor_params + (int64_t)(RUNS ? blockIdx.y : n) * P);
    if (blockIdx.x == 0 && threadIdx.x == 0 && !(d.flags & IA2C_FLAG_SKIP_ADAM)) d.actor_step[RUNS ? blockIdx.y : n] += 1;
    __syncthreads();
    KCLOCK(k_staged);
    const int64_t E = d.E, rows = (int64_t)d.T * E;
    const int64_t ES = RUNS ? E * (gridDim.y / N) : E;
    const ChunkPlan cp = chunk_plan(d.T, E, N);
    const int64_t items = E * cp.n_chunks;
    const float inv_b = 1.f / (float)((int64_t)d.T * d.E_total);
    float2 g2[GN];
#pragma unroll
    for (int i = 0; i < GN; ++i) g2[i] = make_float2(0.f, 0.f);
    float loss = 0.f;
    for (int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; item < items; item += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = RUNS ? (int64_t)run * E + item % E : item % E;
        const int t0 = (int)(item / E) * cp.chunk_len;
        const int t1 = min(d.T, t0 + cp.chunk_len);
        float x[kIn], q[J];
        load_obs6(d.obs + ((int64_t)t0 * ES + e) * kIn, x);
        {
            float2 h1[3], h2[3];
            fwd_f2<J>(wc, x, h1, h2, q);
        }
        // The row's inputs are fetched ONE ITERATION AHEAD (the kernel was stalled on these L2 round trips: ncu long_scoreboard
        // 1.8 per issue): iteration t consumes {next observation, next own action, next predicted partner, reward} loaded
        // during iteration t-1 and carries its own action / predicted partner over from the previous row.
        struct RowIn { float xn[kIn]; int own_n, pp_n; float rew; };
        auto fetch = [&](int t, RowIn& in) {
            const int64_t r = (int64_t)t * ES + e;
            load_obs6(d.obs + (r + ES) * kIn, in.xn);                 // next_obs[t] = obs[t+1]
            in.own_n = d.act[(r + ES) * N + n];
            in.pp_n = d.partner_pred[(r + ES) * N + n];
            in.rew = d.reward[r];
        };
        RowIn cur;
        fetch(t0, cur);
        int own = d.act[((int64_t)t0 * ES + e) * N + n], pp = d.partner_pred[((int64_t)t0 * ES + e) * N + n];
        for (int t = t0; t < t1; ++t) {
            const int64_t r = (int64_t)t * ES + e;
            RowIn nxt = cur;
            if (t + 1 < t1) fetch(t + 1, nxt);
            float qn[J];
            {
                float2 h1[3], h2[3];
                fwd_f2<J>(wc, cur.xn, h1, h2, qn);                   // UPDATED critic, no gradient (ia2c.py:116-127)
            }
            const int own_n = cur.own_n;
            const int ja = joint_index(n, N, own, pp);                                   // ia2c.py:120-121
            const int nja = joint_index(n, N, own_n, cur.pp_n);
            // RUNS spells out, with rounding intrinsics, the contractions nvcc 12.9 makes in the standalone instantiation (read
            // off its SASS: FFMA for rew + gamma * Q', for adv * (-log q) - beta * H, for the entropy terms and for the own
            // action's beta * (..) - adv / q except at the last action): with gamma / beta loaded per run instead of read from
            // the parameter bank the compiler contracts differently, and the batch's runs would drift from the standalone runs
            // in the last bit.  tests/test_gpu_runs.py checks the two byte for byte.
            const float adv = RUNS ? __fmaf_rn(run_gamma<RUNS>(d, ra, run), select_out<J>(qn, nja), cur.rew) - select_out<J>(q, ja)
                                   : (cur.rew + run_gamma<RUNS>(d, ra, run) * select_out<J>(qn, nja)) - select_out<J>(q, ja);
            if (d.adv_dump) d.adv_dump[(int64_t)n * rows + r] = adv;   // never in a batch (refused)
            float2 h1[3], h2[3];
            float p[A];
            fwd_f2<A>(w, x, h1, h2, p);
            softmax_inplace<A>(p);
            // Categorical(probs=p): q = p/sum(p); logit = log(clamp(q)); loss_row = adv*(-logit[a]) - beta*H
            float s = 0.f;
#pragma unroll
            for (int o = 0; o < A; ++o) s += p[o];
            float ent = 0.f, qg = 0.f, neglogp = 0.f, gq[A], qq[A];
#pragma unroll
            for (int o = 0; o < A; ++o) {
                const float qv = p[o] / s;
                const bool inside = (qv >= kEpsClamp) && (qv <= 1.f - kEpsClamp);
                const float logit = logf(fminf(fmaxf(qv, kEpsClamp), 1.f - kEpsClamp));
                float go;
                if constexpr (RUNS) {
                    const float beta = run_beta<RUNS>(d, ra, run), lc = logit + (inside ? 1.f : 0.f);
                    ent = __fmaf_rn(-logit, qv, ent);
                    if (o == own && inside)   // (the standalone build fuses this for the first two actions, not the last)
                        go = o < A - 1 ? __fmaf_rn(beta, lc, -__fdiv_rn(adv, qv)) : __fsub_rn(__fmul_rn(beta, lc), __fdiv_rn(adv, qv));
                    else
                        go = __fmul_rn(beta, lc);
                    if (o == own) neglogp = -logit;
                } else {
                    ent -= logit * qv;
                    go = run_beta<RUNS>(d, ra, run) * (logit + (inside ? 1.f : 0.f));
                    if (o == own) {
                        neglogp = -logit;
                        if (inside) go -= adv / qv;
                    }
                }
                gq[o] = go;
                qq[o] = qv;
                qg = fmaf(qv, go, qg);
            }
            if constexpr (RUNS) loss += __fmaf_rn(adv, neglogp, -__fmul_rn(run_beta<RUNS>(d, ra, run), ent));
            else loss += adv * neglogp - run_beta<RUNS>(d, ra, run) * ent;
            float dy[A];
#pragma unroll
            for (int o = 0; o < A; ++o) dy[o] = qq[o] * (gq[o] - qg) * inv_b;   // through normalise + softmax
            bwd_f2<A>(w, x, h1, h2, [&](int o) { return dy[o]; }, g2);
#pragma unroll
            for (int k = 0; k < kIn; ++k) x[k] = cur.xn[k];
#pragma unroll
            for (int o = 0; o < J; ++o) q[o] = qn[o];
            own = own_n;
            pp = cur.pp_n;
            cur = nxt;
        }
    }
    KCLOCK(k_loop_end);
    KSTAMP(g_kclock, 6);
    float g[2 * GN];
    unpack_g2(g2, g);
    g[P] = loss;
    block_reduce_store<P + 1>(reinterpret_cast<float(&)[P + 1]>(g), red, partials + ((int64_t)(RUNS ? blockIdx.y : n) * gridDim.x + blockIdx.x) * (P + 1));
    KSTAMP(g_kclock, 7);
    KCLOCK_PRINT(d.episode == 5 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) && blockIdx.y == 0 && threadIdx.x == 0,
                 "actor_grad block %3d entry %llu: waited +%llu, staged +%llu, rows done +%llu, exit +%llu ns\n", (int)blockIdx.x,
                 k_entry % 1000000000ull, k_waited - k_entry, k_staged - k_entry, k_loop_end - k_entry, stage_ns() - k_entry);
}

// Sum partials over blocks (fixed order) -> grad[n][0..P] (slot P = loss); optionally Adam.  (reduce.cuh holds
// ReduceArgs and the per-entry epilogue with the Adam step.)
// grid (N, ceil((P+1)/32)); block 1024 = 32 entries x 32 slices of the partial blocks; fixed-order sums.
// The partials are L2-resident, so a thread's chain of dependent adds costs one L2 round trip per term: many
// short slices (<= 8 terms at 256 partial blocks, loads issued back to back) instead of few long ones.
// Everything the update reads is requested right after the wait — the partial rows (every slice), the Adam operands (slice 0)
// and the step counter (the bias thread) — so the kernel costs one memory round trip before its barrier and none after it.
// RUNS: the R * N nets of a batch of runs (ia2c_train_episode_runs); net n belongs to run n / N and steps with that run's lr.
template <bool RUNS>
__global__ void __launch_bounds__(32 * kReduceSlices) reduce_adam_kernel(ReduceArgs R, ReduceRunsArg<RUNS> rr) {
    pdl_prologue();
    KSTAMP(g_kclock, R.P == kCriticP ? 0 : 10);
    const int n = blockIdx.x, P = R.P;
    const int col = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int i = blockIdx.y * 32 + col;
    __shared__ float part[kReduceSlices][33];
    __shared__ AdamBias bias;
    const bool bias_thread = threadIdx.x == blockDim.x - 1 && R.apply_adam;
    const int t = bias_thread ? __ldcg(R.step + n) : 0;   // step[n] was already incremented by the gradient kernel / apply entry
    const AdamIn in = (slice == 0 && i <= P) ? load_adam_in(R, n, i) : AdamIn{0.f, 0.f, 0.f, 0.f};
    float s = 0.f;
    if (i <= P) {
        if (R.from_partials) {
            const float* src = R.partials + (int64_t)n * R.n_blocks * (P + 1) + i;
            float v[8];
            for (int b0 = slice; b0 < R.n_blocks; b0 += 8 * kReduceSlices) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int b = b0 + u * kReduceSlices;
                    v[u] = b < R.n_blocks ? src[(int64_t)b * (P + 1)] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) s += v[u];
            }
        } else if (slice == 0) {
            s = R.grad[(int64_t)n * (P + 1) + i];
        }
    }
    if (bias_thread) bias = adam_bias(t, reduce_lr<RUNS>(R, rr, n));
    part[slice][col] = s;
    __syncthreads();
    if (slice != 0 || i > P) return;
#pragma unroll
    for (int k = 1; k < kReduceSlices; ++k) s += part[k][col];
    finish_entry(R, n, i, s, bias, in);
    KSTAMP(g_kclock, R.P == kCriticP ? 3 : 13);
}

__global__ void bump_steps_kernel(int32_t* step, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) step[i] += 1;
}

// Blocks per agent for the gradient kernels: one resident wave (2 blocks of 128 threads per SM at 255
// registers) shared by the N agents, grid-stride over the (env, time chunk) items.
int grad_blocks(const ia2c_episode_desc* d) {
    const ChunkPlan cp = chunk_plan(d->T, d->E, d->N);
    const int64_t items = d->E * cp.n_chunks;
    const int64_t by_items = (items + kGradThreads - 1) / kGradThreads;
    const int64_t by_wave = std::max<int64_t>(1, (int64_t)kSMs * 2 / std::max(1, d->N));
    return (int)std::max<int64_t>(1, std::min(by_items, by_wave));
}

// Launch shape of rollout_many_kernel for `runs` runs of d->E envs.  A block walks its envs one after the other, so an episode
// costs (waves of resident blocks) x (envs per block) — take the envs per block c that minimises it over all runs * ceil(E / c)
// blocks (1024 x 256: 7 envs = one wave of 147 blocks instead of two waves of 4).  Envs are independent (no sum crosses an env),
// so the choice changes no result.
struct ManyPlan { int threads, envs_per_block; size_t smem; int64_t blocks; };   // blocks: per run (grid x)
template <bool RUNS, bool PARTNERS = false>
ManyPlan many_plan(const ia2c_episode_desc* d, int runs) {
    ManyPlan p;
    p.threads = ((d->N + 31) / 32) * 32;
    p.smem = (size_t)kManyMaxEnvs * (8 + 1 + 1) * 4 + (size_t)kManyMaxEnvs * p.threads;
    static int resident_per_sm[9] = {0};     // per instantiation, by threads / 32; the same on every B200 of the box
    int& per_sm = resident_per_sm[p.threads / 32];
    if (per_sm == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rollout_many_kernel<RUNS, PARTNERS>, p.threads, p.smem) != cudaSuccess) per_sm = 1;
    const int64_t resident = (int64_t)kSMs * std::max(1, per_sm);
    p.envs_per_block = 1;
    int64_t best = INT64_MAX;
    for (int c = 1; c <= std::min(kManyMaxEnvs, p.threads); ++c) {   // one owner thread per env of the chunk
        const int64_t blocks = runs * ((d->E + c - 1) / c), cost = ((blocks + resident - 1) / resident) * c;
        if (cost <= best) { best = cost; p.envs_per_block = c; }   // ties: the larger chunk (fewer blocks, weights loaded once per more envs)
    }
    p.blocks = (d->E + p.envs_per_block - 1) / p.envs_per_block;
    return p;
}

int validate(const ia2c_episode_desc* d, const char* who) {
    IA2C_REQUIRE(d != nullptr, "%s: null descriptor", who);
    IA2C_REQUIRE(d->E > 0 && d->E_total >= d->E && d->T > 0 && d->T < 65535, "%s: E=%lld E_total=%lld T=%d", who,
                 (long long)d->E, (long long)d->E_total, d->T);
    IA2C_REQUIRE(d->N >= 2 && d->N <= 1023, "%s: N=%d outside 2..1023", who, d->N);
    IA2C_REQUIRE(d->M >= 2 && d->M <= IA2C_MAX_MODELS, "%s: M=%d outside 2..%d", who, d->M, IA2C_MAX_MODELS);
    IA2C_REQUIRE(d->actor_params && d->critic_params && d->obs && d->reward && d->act && d->partner_true &&
                     d->partner_pred, "%s: null network/trajectory pointer", who);
    return 0;
}

}  // namespace
}  // namespace ia2c

using namespace ia2c;

static bool fused_critic(const ia2c_episode_desc* d) {
    return (d->flags & IA2C_FLAG_FUSED_ROLLOUT) && (d->flags & IA2C_FLAG_FUSED_CRITIC);
}
// partial rows per agent written by the critic-gradient producer (fused rollout stage or critic_grad_kernel)
static int critic_partial_blocks(const ia2c_episode_desc* d) {
    return fused_critic(d) ? (int)rollout_fused_blocks(d->E, d->N) : grad_blocks(d);
}

// the actor-gradient producer: the pipelined kernel (actor_pipe.cu) unless the caller asks for the column kernel
static bool actor_columns(const ia2c_episode_desc* d) { return d->flags & IA2C_FLAG_ACTOR_COLUMNS; }
static int actor_partial_blocks(const ia2c_episode_desc* d) {
    return actor_columns(d) ? grad_blocks(d) : (int)actor_pipe_blocks(d->E, d->N);
}
static int launch_actor_grad(const ia2c_episode_desc* d, cudaStream_t s) {
    if (!actor_columns(d)) return actor_pipe_launch(d, s);
    dim3 grid(grad_blocks(d), d->N);
    return launch_pdl("actor_grad_kernel", actor_grad_kernel<false>, grid, dim3(kGradThreads), 0, s, *d, d->partials, NoRuns{});
}

extern "C" size_t ia2c_episode_partials_floats(const ia2c_episode_desc* d) {
    if (!d || d->N < 1 || d->E < 1 || d->T < 1) return 0;
    const size_t blocks = (size_t)std::max<int64_t>(std::max<int64_t>(grad_blocks(d), (d->E + 31) / 32),
                                                    rollout_fused_blocks(d->E, std::min(d->N, 8)));
    return (size_t)d->N * blocks * (kCriticP + 1);
}

extern "C" int ia2c_rollout_fused_supported(int32_t N, int32_t M) { return rollout_fused_supported(N, M); }

static int check_rollout(const ia2c_episode_desc* d, const char* who) {
    if (int rc = validate(d, who)) return rc;
    IA2C_REQUIRE(d->env_state && d->env_hist && d->env_cls && d->env_elapsed && d->ep_return && d->belief_records &&
                     d->filter_action, "%s: null env/belief pointer", who);
    if (d->flags & IA2C_FLAG_FUSED_ROLLOUT) {
        IA2C_REQUIRE(rollout_fused_supported(d->N, d->M), "%s: IA2C_FLAG_FUSED_ROLLOUT needs N<=8 with M=5 (or N=2, M=3); got N=%d M=%d", who, d->N, d->M);
        if (d->flags & IA2C_FLAG_FUSED_CRITIC) {
            IA2C_REQUIRE(d->partials && d->partials_floats >= ia2c_episode_partials_floats(d) && d->critic_step,
                         "%s: IA2C_FLAG_FUSED_CRITIC needs the partials workspace and critic_step", who);
        }
    }
    return 0;
}

// The rollout of ia2c_rollout; p != nullptr: the PARTNERS instantiations (the path was checked by validate_env_partners).
static int rollout_launch(const ia2c_episode_desc* d, const EnvPartners* p, void* stream) {
    cudaStream_t s = as_stream(stream);
    if (d->flags & IA2C_FLAG_FUSED_ROLLOUT) return rollout_fused_launch(d, nullptr, p, s);
    const bool episode_beliefs = !(d->flags & IA2C_FLAG_BELIEF_PER_STEP) && ia2c_belief_supports_episode(d->N, d->M);
    if (p || (episode_beliefs && !(d->flags & IA2C_FLAG_ROLLOUT_PER_STEP) && d->N <= 256)) {
        // ONE persistent kernel for the T+1 env / actor steps, then ONE kernel for the episode's belief updates
        const ManyPlan mp = p ? many_plan<false, true>(d, 1) : many_plan<false>(d, 1);
        const int rc = p ? launch_pdl("rollout_many_kernel", rollout_many_kernel<false, true>, dim3((unsigned)mp.blocks), dim3(mp.threads),
                                      mp.smem, s, *d, mp.envs_per_block, NoRuns{}, *p)
                         : launch_pdl("rollout_many_kernel", rollout_many_kernel<false>, dim3((unsigned)mp.blocks), dim3(mp.threads),
                                      mp.smem, s, *d, mp.envs_per_block, NoRuns{}, NoPartners{});
        if (rc) return rc;
        return ia2c_belief_update_pairs_episode(d->belief_records, d->filter_action, d->act, d->inj_u_belief, d->pred_dump, d->belief_dump,
                                                d->partner_pred, d->E, d->N, d->M, d->T + 1, d->seed, d->episode, d->env_offset, stream);
    }
    StepArgs S;
    S.d = *d;
    int G = 1;
    while (G < d->N && G < 32) G <<= 1;
    S.G = G;
    const int epw = 32 / G;
    const int64_t warps = (d->E + epw - 1) / epw;
    const int blocks = ceil_div(warps * 32, kRolloutThreads);
    // up to kActorEnvsPerThread envs per thread (amortises the weight load) once that still leaves two waves of blocks
    const int64_t ept = std::max<int64_t>(1, std::min<int64_t>(kActorEnvsPerThread, d->E * d->N / ((int64_t)kActorThreads * 2 * kSMs)));
    dim3 actor_grid((unsigned)ceil_div(d->E, (int64_t)kActorThreads * ept), (unsigned)d->N);
    const int64_t EN = d->E * d->N, K = d->N - 1;
    // Nothing reads a belief before the update phase (ia2c.py:72-102 vs :104-121), so with many modelled others the T+1 env /
    // actor steps run first and ONE kernel then carries every belief record through the whole episode in registers
    // (belief.cu: belief_pairs_episode_kernel) instead of streaming the records once per step.
    for (int t = 0; t <= d->T + 1; ++t) {
        S.t = t;
        if (int rc = launch_pdl("env_step_kernel", env_step_kernel, dim3(blocks), dim3(kRolloutThreads), 0, s, S)) return rc;
        if (t > d->T) break;   // the last call only completes partner_true[T]
        if (int rc = launch_pdl("actor_step_kernel", actor_step_kernel, actor_grid, dim3(kActorThreads), 0, s, S)) return rc;
        if (episode_beliefs) continue;
        int rc = ia2c_belief_update_pairs(
            d->belief_records, d->filter_action, d->act + (int64_t)t * EN,
            d->inj_u_belief ? d->inj_u_belief + (int64_t)t * EN * K : nullptr,
            d->pred_dump ? d->pred_dump + (int64_t)t * EN * K : nullptr,
            d->belief_dump ? d->belief_dump + (int64_t)t * EN * K * d->M : nullptr,
            d->partner_pred + (int64_t)t * EN, d->E, d->N, d->M, /*reset_prior=*/t == 0, d->seed, d->episode,
            (uint32_t)t, d->env_offset, stream);
        if (rc) return rc;
    }
    if (episode_beliefs)
        return ia2c_belief_update_pairs_episode(d->belief_records, d->filter_action, d->act, d->inj_u_belief, d->pred_dump, d->belief_dump,
                                                d->partner_pred, d->E, d->N, d->M, d->T + 1, d->seed, d->episode, d->env_offset, stream);
    return 0;
}

extern "C" int ia2c_rollout(const ia2c_episode_desc* d, void* stream) {
    if (int rc = check_rollout(d, "ia2c_rollout")) return rc;
    return rollout_launch(d, nullptr, stream);
}

static int run_reduce(const ia2c_episode_desc* d, int which, int from_partials, int apply, cudaStream_t s) {
    ReduceArgs R = make_reduce_args(*d, which, which == 0 ? critic_partial_blocks(d) : actor_partial_blocks(d));
    R.apply_adam = apply;
    R.from_partials = from_partials;
    if (!from_partials && apply) {   // ia2c_apply_adam: the gradient kernel did not bump the step counter
        bump_steps_kernel<<<ceil_div(d->N, 256), 256, 0, s>>>(R.step, d->N);
        if (int rc = check_launch("bump_steps_kernel")) return rc;
    }
    dim3 grid(d->N, ceil_div(R.P + 1, 32));
    return launch_pdl("reduce_adam_kernel", reduce_adam_kernel<false>, grid, dim3(32 * kReduceSlices), 0, s, R, NoRuns{});
}

// ------------------------------------------------------------------------------------------------
// Fused gradient all-reduce + Adam over NVLink peer memory (multi-GPU, one process per GPU).
//
// Per optimiser phase every rank holds locally summed gradients (already scaled by the GLOBAL 1/(T*E_total)).
// Instead of reduce kernel -> NCCL all-reduce -> Adam kernel (three launches and a ~20 us small-message
// collective), ONE kernel per rank does all of it over peer-mapped ("symmetric") buffers:
//   1. sum this rank's per-block partials for a chunk of 32 entries              (fixed order)
//   2. PUSH each sum into every peer's inbox slot [parity][my rank] as ONE naturally aligned 64-bit word
//      {epoch << 32 | float bits} with a single st.relaxed.sys.u64 (single-copy atomic: the word cannot tear), so the
//      message carries its own flag — no separate flag store, no system-scope fence, no second NVLink hop.  With a
//      multicast (NVLS) mapping one multimem.st reaches all inboxes through the switch instead of `world` stores
//   3. poll (bounded by a wall-clock budget) the world's words for this entry in the own inbox until each carries
//      this epoch
//   4. add the contributions in RANK order (every rank computes bit-identical sums) and apply Adam.
// Chunks are independent, so transfer and arithmetic of different chunks overlap; the grid is persistent
// (<= one resident wave) so a block never waits for a peer block that cannot be scheduled.  Inboxes are
// double-buffered by epoch parity: kernels are stream-ordered on every rank, so when a rank has finished exchange e
// every peer has at least started e (i.e. finished e-1) — a peer can be at most one exchange ahead, and a slot's
// previous content carries epoch - 2, never this epoch.  Epoch 0 is the empty inbox.
// Failure: a chunk whose words do not all arrive in time applies NOTHING (no gradient, no Adam, no step counter),
// the block stops, and the error word of EVERY rank is raised; a rank whose error word is set turns all later
// exchanges into no-ops, so parameters are never stepped with a stale or partial sum and the run fails loudly at the
// host's next check (trainer.py: check_comm — before statistics, checkpoints and after bench regions).
struct PeerArgs {
    int rank, world;
    unsigned long long* inbox[IA2C_MAX_RANKS];   // 64-bit words {epoch << 32 | float bits}
    unsigned long long* mc_inbox;   // multicast mapping or null
    int32_t* error[IA2C_MAX_RANKS];
    uint32_t epoch;
    int t;                          // Adam step number of this update (host-tracked in the multi-rank path)
    int64_t stride;                 // words per (parity, rank) slot = N * (kCriticP + 1)
    unsigned long long timeout_ns;
};

__device__ __forceinline__ void st_word_sys(unsigned long long* p, unsigned long long w) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ void st_word_multicast(unsigned long long* p, unsigned long long w) {
    asm volatile("multimem.st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ unsigned long long ld_word_sys(const unsigned long long* p) {
    unsigned long long w;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
    return w;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __launch_bounds__(32 * kReduceSlices) allreduce_adam_kernel(ReduceArgs R, PeerArgs X, int total_chunks,
                                                                            int chunks_per_agent) {
    __shared__ float part[kReduceSlices][33];
    __shared__ AdamBias bias;
    pdl_release();
    if (threadIdx.x == blockDim.x - 1) bias = adam_bias(X.t, R.lr);   // from launch arguments only: overlaps the predecessor's tail
    pdl_wait();
    KSTAMP(g_kclock, R.P == kCriticP ? 0 : 10);
    if (X.error[X.rank] && *reinterpret_cast<volatile int32_t*>(X.error[X.rank]) != 0) return;   // a previous exchange failed: no-op
    const int P = R.P, col = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int parity = (int)(X.epoch & 1u);
    for (int c = blockIdx.x; c < total_chunks; c += gridDim.x) {
        const int n = c / chunks_per_agent, i = (c % chunks_per_agent) * 32 + col;
        float s = 0.f;
        if (i <= P) {
            const float* src = R.partials + (int64_t)n * R.n_blocks * (P + 1) + i;
            float v[8];
            for (int b0 = slice; b0 < R.n_blocks; b0 += 8 * kReduceSlices) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int b = b0 + u * kReduceSlices;
                    v[u] = b < R.n_blocks ? src[(int64_t)b * (P + 1)] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) s += v[u];
            }
        }
        part[slice][col] = s;
        __syncthreads();
        KSTAMP(g_kclock, R.P == kCriticP ? 1 : 11);
        float g = 0.f;
        int late = 0;
        // Warp 0 owns the chunk's 32 entries (poll, sum in rank order, Adam); warp 1 computes the same local sums (same order:
        // bit-identical) and PUSHES them, then waits for the remote stores to be acknowledged (fence.sys) while warp 0 is already
        // polling.  Without that the acknowledgements were collected at grid completion and the next kernel left its
        // griddepcontrol.wait 2-3 us later than after a kernel without peer stores (profiles/r02_timeline.md).
        const bool owner = slice == 0 && i <= P, pusher = slice == 1 && i <= P;
        const int64_t idx = (int64_t)n * (P + 1) + i;
        if (owner || pusher) {
            s = part[0][col];
#pragma unroll
            for (int k = 1; k < kReduceSlices; ++k) s += part[k][col];
            if (i == P) s *= R.loss_scale;
        }
        if (pusher) {
            const int64_t mine = ((int64_t)parity * X.world + X.rank) * X.stride + idx;
            const unsigned long long word = ((unsigned long long)X.epoch << 32) | (unsigned long long)__float_as_uint(s);
            if (X.mc_inbox) {
                st_word_multicast(X.mc_inbox + mine, word);                                  // one store, fanned out by the switch
            } else {
                for (int p = 0; p < X.world; ++p) st_word_sys(X.inbox[p] + mine, word);      // NVLink stores (self included)
            }
            __threadfence_system();
        }
        if (owner) {
            // first look at every rank's word at once (independent loads: one L2 round trip instead of `world` in a row), then
            // wait, in rank order, only for the ones that have not arrived
            const unsigned long long* w0 = X.inbox[X.rank] + (int64_t)parity * X.world * X.stride + idx;
            unsigned long long m[IA2C_MAX_RANKS];
#pragma unroll
            for (int r = 0; r < IA2C_MAX_RANKS; ++r) m[r] = r < X.world ? ld_word_sys(w0 + (int64_t)r * X.stride) : 0ull;
            unsigned long long t_start = 0;
#pragma unroll
            for (int r = 0; r < IA2C_MAX_RANKS; ++r) {                       // rank order: identical sums on every rank
                if (r >= X.world || late) continue;
                int spins = 0;
                while ((uint32_t)(m[r] >> 32) != X.epoch) {
                    __nanosleep(32);
                    if ((++spins & 63) == 0) {                               // wall-clock budget, checked every 64 polls
                        const unsigned long long now = global_ns();
                        if (t_start == 0) t_start = now;
                        else if (now - t_start > X.timeout_ns) { late = 1; break; }
                    }
                    m[r] = ld_word_sys(w0 + (int64_t)r * X.stride);
                }
                if (!late) g += __uint_as_float((uint32_t)m[r]);
            }
        }
        KSTAMP(g_kclock, R.P == kCriticP ? 2 : 12);
        if (__syncthreads_or(late)) {      // block-uniform: nothing of this chunk is applied, the block stops
            if (threadIdx.x == 0)
                for (int p = 0; p < X.world; ++p)
                    if (X.error[p]) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(X.error[p]), "r"(1) : "memory");
            return;
        }
        if (owner) {
            R.grad[idx] = g;
            if (i == P) {
                R.loss_out[n] = g;
                R.step[n] = X.t;                                             // device-side counter follows the host's
            } else {
                const int64_t k = (int64_t)n * P + i;
                if (R.grad_accum) {                                          // actor gradients accumulate (Q2)
                    g += R.grad_accum[k];
                    R.grad_accum[k] = g;
                }
                adam_update(R.params[k], R.m[k], R.v[k], g, bias);
            }
        }
        KSTAMP(g_kclock, R.P == kCriticP ? 3 : 13);
    }
}

static int check_update_ptrs(const ia2c_episode_desc* d, const char* who) {
    IA2C_REQUIRE(d->partials && d->partials_floats >= ia2c_episode_partials_floats(d), "%s: partials workspace too small", who);
    IA2C_REQUIRE(d->critic_grad && d->actor_grad && d->critic_m && d->critic_v && d->actor_m && d->actor_v &&
                     d->actor_grad_accum && d->critic_step && d->actor_step && d->loss_out, "%s: null optimiser pointer", who);
    return 0;
}

extern "C" int ia2c_critic_phase(const ia2c_episode_desc* d, void* stream) {
    if (int rc = validate(d, "ia2c_critic_phase")) return rc;
    if (int rc = check_update_ptrs(d, "ia2c_critic_phase")) return rc;
    cudaStream_t s = as_stream(stream);
    if (!fused_critic(d)) {   // otherwise the rollout kernel's critic stage already wrote the partials
        dim3 grid(grad_blocks(d), d->N);
        if (int rc = launch_pdl("critic_grad_kernel", critic_grad_kernel<false>, grid, dim3(kGradThreads), 0, s, *d, d->partials, NoRuns{})) return rc;
    }
    if (d->flags & IA2C_FLAG_GRAD_ONLY) return 0;
    return run_reduce(d, 0, 1, !(d->flags & IA2C_FLAG_SKIP_ADAM), s);
}

extern "C" int ia2c_actor_phase(const ia2c_episode_desc* d, void* stream) {
    if (int rc = validate(d, "ia2c_actor_phase")) return rc;
    if (int rc = check_update_ptrs(d, "ia2c_actor_phase")) return rc;
    cudaStream_t s = as_stream(stream);
    if (int rc = launch_actor_grad(d, s)) return rc;
    if (d->flags & IA2C_FLAG_GRAD_ONLY) return 0;
    return run_reduce(d, 1, 1, !(d->flags & IA2C_FLAG_SKIP_ADAM), s);
}

extern "C" int ia2c_apply_adam(const ia2c_episode_desc* d, int32_t which, void* stream) {
    if (int rc = validate(d, "ia2c_apply_adam")) return rc;
    if (int rc = check_update_ptrs(d, "ia2c_apply_adam")) return rc;
    IA2C_REQUIRE(which == 0 || which == 1, "ia2c_apply_adam: which=%d", which);
    return run_reduce(d, which, 0, 1, as_stream(stream));
}

// One standalone episode; p != nullptr: with frozen partners per env (the caller checked everything before the first CUDA call).
static int train_episode_impl(const ia2c_episode_desc* d, const EnvPartners* p, void* stream) {
    if (int rc = p ? rollout_launch(d, p, stream) : ia2c_rollout(d, stream)) return rc;
    if (int rc = ia2c_critic_phase(d, stream)) return rc;
    return ia2c_actor_phase(d, stream);
}

extern "C" int ia2c_train_episode(const ia2c_episode_desc* d, void* stream) { return train_episode_impl(d, nullptr, stream); }

// One episode of a multi-GPU run in ONE call per rank: rollout, critic gradient, fused NVLink all-reduce + Adam
// (epoch0 + 1), actor gradient, fused all-reduce + Adam (epoch0 + 2).  desc.flags = SKIP_ADAM | GRAD_ONLY.
extern "C" int ia2c_train_episode_p2p(const ia2c_episode_desc* d, const ia2c_peer_desc* peers, uint32_t epoch0, void* stream) {
    IA2C_REQUIRE(d && peers, "ia2c_train_episode_p2p: null descriptor");
    IA2C_REQUIRE((d->flags & IA2C_FLAG_GRAD_ONLY) && (d->flags & IA2C_FLAG_SKIP_ADAM),
                 "ia2c_train_episode_p2p: desc.flags must carry SKIP_ADAM | GRAD_ONLY");
    const int32_t adam_step = (int32_t)d->episode + 1;   // one Adam step per net per episode
    if (int rc = ia2c_rollout(d, stream)) return rc;
    if (int rc = ia2c_critic_phase(d, stream)) return rc;
    if (int rc = ia2c_allreduce_adam(d, 0, peers, epoch0 + 1, adam_step, stream)) return rc;
    if (int rc = ia2c_actor_phase(d, stream)) return rc;
    return ia2c_allreduce_adam(d, 1, peers, epoch0 + 2, adam_step, stream);
}

extern "C" int ia2c_train_episode_host(const ia2c_episode_desc* d, const float* host_u_action,
                                       const double* host_u_belief, float* host_loss_out, double* host_ep_return,
                                       void* stream) {
    if (int rc = validate(d, "ia2c_train_episode_host")) return rc;
    IA2C_REQUIRE(!(d->flags & IA2C_FLAG_SKIP_ADAM), "ia2c_train_episode_host: single-rank entry point (SKIP_ADAM set)");
    cudaStream_t s = as_stream(stream);
    const size_t n_act = (size_t)(d->T + 1) * d->E * d->N;
    if (host_u_action) {
        IA2C_REQUIRE(d->inj_u_action, "ia2c_train_episode_host: desc.inj_u_action staging buffer missing");
        if (cudaMemcpyAsync(const_cast<float*>(d->inj_u_action), host_u_action, n_act * sizeof(float), cudaMemcpyHostToDevice, s) != cudaSuccess)
            return check_launch("memcpy H2D u_action");
    }
    if (host_u_belief) {
        IA2C_REQUIRE(d->inj_u_belief, "ia2c_train_episode_host: desc.inj_u_belief staging buffer missing");
        if (cudaMemcpyAsync(const_cast<double*>(d->inj_u_belief), host_u_belief, n_act * (d->N - 1) * sizeof(double), cudaMemcpyHostToDevice, s) != cudaSuccess)
            return check_launch("memcpy H2D u_belief");
    }
    if (int rc = ia2c_train_episode(d, stream)) return rc;
    if (host_loss_out && cudaMemcpyAsync(host_loss_out, d->loss_out, 2 * (size_t)d->N * sizeof(float), cudaMemcpyDeviceToHost, s) != cudaSuccess)
        return check_launch("memcpy D2H loss");
    if (host_ep_return && cudaMemcpyAsync(host_ep_return, d->ep_return, (size_t)d->E * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess)
        return check_launch("memcpy D2H ep_return");
    if (cudaStreamSynchronize(s) != cudaSuccess) return check_launch("stream sync");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Pipelined host-buffer entry point: n_episodes episodes whose injected uniforms live in (pinned) HOST
// memory.  The H2D copy of episode k+1 runs on the pipe's copy stream while episode k computes; every
// episode's losses and returns are read back to its own host slot on the pipe's download stream; one host sync
// at the end.  The streams and events are owned by a caller-held handle (ia2c_host_pipe_create / _destroy): the
// library keeps no hidden per-thread state.
constexpr int kMaxStages = 8;
struct ia2c_host_pipe {
    cudaStream_t copy = nullptr, down = nullptr;
    cudaEvent_t copied[kMaxStages] = {}, consumed[kMaxStages] = {};          // one pair per staging region
    cudaEvent_t done[2] = {nullptr, nullptr}, downloaded[2] = {nullptr, nullptr};
    int device = -1;
    int stages = 2;   // staging regions in use: desc.inj_u_action + (stages - 1) consecutive regions at stage_b
};

extern "C" int ia2c_host_pipe_destroy(ia2c_host_pipe* p) {
    if (!p) return 0;
    if (p->copy) { cudaStreamSynchronize(p->copy); cudaStreamDestroy(p->copy); }
    if (p->down) { cudaStreamSynchronize(p->down); cudaStreamDestroy(p->down); }
    for (int i = 0; i < kMaxStages; ++i)
        for (cudaEvent_t ev : {p->copied[i], p->consumed[i]})
            if (ev) cudaEventDestroy(ev);
    for (int i = 0; i < 2; ++i)
        for (cudaEvent_t ev : {p->done[i], p->downloaded[i]})
            if (ev) cudaEventDestroy(ev);
    delete p;
    cudaGetLastError();
    return 0;
}

extern "C" int ia2c_host_pipe_create(ia2c_host_pipe** out) {
    IA2C_REQUIRE(out != nullptr, "ia2c_host_pipe_create: null output");
    *out = nullptr;
    ia2c_host_pipe* p = new ia2c_host_pipe();
    bool ok = cudaGetDevice(&p->device) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&p->copy, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&p->down, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < kMaxStages && ok; ++i)
        for (cudaEvent_t* ev : {&p->copied[i], &p->consumed[i]})
            ok = ok && cudaEventCreateWithFlags(ev, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
        for (cudaEvent_t* ev : {&p->done[i], &p->downloaded[i]})
            ok = ok && cudaEventCreateWithFlags(ev, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        const int rc = check_launch("ia2c_host_pipe_create");
        ia2c_host_pipe_destroy(p);
        return rc ? rc : IA2C_ERR_CUDA;
    }
    *out = p;
    return 0;
}

static inline size_t align8(size_t x) { return (x + 7) & ~size_t(7); }

// Depth of the staging ring: `stages` regions in all (2..8) — desc.inj_u_action plus stages - 1 consecutive regions of
// ia2c_host_stage_stride(desc) bytes each at stage_b.  More regions let the copy engine run further ahead of the kernels:
// on a multi-GPU box an episode's kernels wait for the slowest rank in the gradient exchange, and with only two regions
// every such wait also idles this rank's copy engine.
extern "C" int ia2c_host_pipe_set_stages(ia2c_host_pipe* p, int32_t stages) {
    IA2C_REQUIRE(p && stages >= 2 && stages <= kMaxStages, "ia2c_host_pipe_set_stages: stages=%d outside 2..%d", stages, kMaxStages);
    p->stages = stages;
    return 0;
}

extern "C" size_t ia2c_host_tape_bytes(const ia2c_episode_desc* d) {
    if (!d) return 0;
    const size_t n_act = (size_t)(d->T + 1) * d->E * d->N;
    return align8(n_act * sizeof(float)) + n_act * (d->N - 1) * sizeof(double);
}
extern "C" size_t ia2c_host_stage_stride(const ia2c_episode_desc* d) { return (ia2c_host_tape_bytes(d) + 255) & ~size_t(255); }
extern "C" size_t ia2c_host_result_bytes(const ia2c_episode_desc* d) {
    if (!d) return 0;
    return align8(2 * (size_t)d->N * sizeof(float)) + (size_t)d->E * sizeof(double);
}

// peers == nullptr: single rank (ia2c_train_episode per episode); otherwise the multi-GPU sequence with the fused
// NVLink all-reduce + Adam after each gradient phase (desc.flags must carry SKIP_ADAM | GRAD_ONLY).
static int episodes_host_impl(const ia2c_episode_desc* d, ia2c_host_pipe* pipe, const ia2c_peer_desc* peers, uint32_t epoch0,
                              void* stage_b, void* result_b, int32_t n_episodes, const void* const* host_tapes,
                              void* host_results, void* stream) {
    if (int rc = validate(d, "ia2c_train_episodes_host")) return rc;
    if (peers) IA2C_REQUIRE((d->flags & IA2C_FLAG_GRAD_ONLY) && (d->flags & IA2C_FLAG_SKIP_ADAM),
                            "ia2c_train_episodes_host_p2p: desc.flags must carry SKIP_ADAM | GRAD_ONLY");
    else IA2C_REQUIRE(!(d->flags & IA2C_FLAG_SKIP_ADAM), "ia2c_train_episodes_host: single-rank entry point (SKIP_ADAM set)");
    IA2C_REQUIRE(pipe && pipe->copy && pipe->down, "ia2c_train_episodes_host: null pipe (ia2c_host_pipe_create)");
    IA2C_REQUIRE(n_episodes > 0 && host_tapes && host_results, "ia2c_train_episodes_host: null host pointer or n_episodes=%d", n_episodes);
    int dev = -1;
    cudaGetDevice(&dev);
    IA2C_REQUIRE(dev == pipe->device, "ia2c_train_episodes_host: pipe was created on device %d, current device is %d", pipe->device, dev);
    const size_t n_act = (size_t)(d->T + 1) * d->E * d->N;
    const size_t off_b = align8(n_act * sizeof(float)), tape_bytes = ia2c_host_tape_bytes(d);
    const size_t off_ret = align8(2 * (size_t)d->N * sizeof(float)), res_bytes = ia2c_host_result_bytes(d);
    // ONE copy per direction per episode: the two uniform tapes share a staging region, losses and returns a result region
    IA2C_REQUIRE(d->inj_u_action && stage_b && (const char*)d->inj_u_belief == (const char*)d->inj_u_action + off_b,
                 "ia2c_train_episodes_host: inj_u_belief must follow inj_u_action in one staging region (ia2c_host_tape_bytes)");
    IA2C_REQUIRE((const char*)d->ep_return == (const char*)d->loss_out + off_ret,
                 "ia2c_train_episodes_host: ep_return must follow loss_out in one result region (ia2c_host_result_bytes)");
    cudaStream_t s = as_stream(stream);
    ia2c_host_pipe& g = *pipe;
    const int S = g.stages;
    char* stage[kMaxStages];
    stage[0] = reinterpret_cast<char*>(const_cast<float*>(d->inj_u_action));
    for (int b = 1; b < S; ++b) stage[b] = reinterpret_cast<char*>(stage_b) + (size_t)(b - 1) * ia2c_host_stage_stride(d);
    // with a second result region the D2H of episode k runs on its own stream while episode k+1 computes
    char* result[2] = {reinterpret_cast<char*>(d->loss_out), result_b ? reinterpret_cast<char*>(result_b) : reinterpret_cast<char*>(d->loss_out)};
    ia2c_episode_desc e = *d;
    const bool trace = getenv("IA2C_TRACE_HOST") != nullptr;   // diagnostics: host enqueue time vs total
    const auto t_begin = std::chrono::steady_clock::now();
    auto cuda_ok = [](cudaError_t err, const char* what) { return err == cudaSuccess ? 0 : check_launch(what); };
    // trace only: timing events around every H2D copy (copy stream) and every episode's kernels (compute stream)
    constexpr int kTraceMax = 64;
    cudaEvent_t tr_ev[kTraceMax][4] = {};
    const int n_traced = trace ? std::min<int>(n_episodes, kTraceMax) : 0;
    for (int k = 0; k < n_traced; ++k)
        for (int j = 0; j < 4; ++j) cudaEventCreate(&tr_ev[k][j]);
    auto enqueue = [&]() -> int {
        // the copy stream must not overwrite a staging set that earlier work on `s` may still read
        for (int b = 0; b < S; ++b)
            if (int rc = cuda_ok(cudaEventRecord(g.consumed[b], s), "cudaEventRecord")) return rc;
        for (int k = 0; k < n_episodes; ++k) {
            const int b = k % S;        // staging region
            const int rb = k & 1;       // result region
            cudaStreamWaitEvent(g.copy, g.consumed[b], 0);
            if (k < n_traced) cudaEventRecord(tr_ev[k][0], g.copy);
            if (int rc = cuda_ok(cudaMemcpyAsync(stage[b], host_tapes[k], tape_bytes, cudaMemcpyHostToDevice, g.copy), "memcpy H2D uniforms")) return rc;
            if (k < n_traced) cudaEventRecord(tr_ev[k][1], g.copy);
            cudaEventRecord(g.copied[b], g.copy);
            cudaStreamWaitEvent(s, g.copied[b], 0);
            if (result_b && k >= 2) cudaStreamWaitEvent(s, g.downloaded[rb], 0);   // region rb was read back before it is rewritten
            e.inj_u_action = reinterpret_cast<const float*>(stage[b]);
            e.inj_u_belief = reinterpret_cast<const double*>(stage[b] + off_b);
            e.loss_out = reinterpret_cast<float*>(result[rb]);
            e.ep_return = reinterpret_cast<double*>(result[rb] + off_ret);
            e.episode = d->episode + (uint32_t)k;
            if (k < n_traced) cudaEventRecord(tr_ev[k][2], s);
            if (!peers) {
                if (int rc = ia2c_train_episode(&e, stream)) return rc;
            } else {
                if (int rc = ia2c_train_episode_p2p(&e, peers, epoch0 + 2 * (uint32_t)k, stream)) return rc;
            }
            if (k < n_traced) cudaEventRecord(tr_ev[k][3], s);
            cudaEventRecord(g.consumed[b], s);
            char* host_slot = reinterpret_cast<char*>(host_results) + (size_t)k * res_bytes;
            if (result_b) {
                cudaEventRecord(g.done[rb], s);
                cudaStreamWaitEvent(g.down, g.done[rb], 0);
                if (int rc = cuda_ok(cudaMemcpyAsync(host_slot, result[rb], res_bytes, cudaMemcpyDeviceToHost, g.down), "memcpy D2H results")) return rc;
                cudaEventRecord(g.downloaded[rb], g.down);
            } else if (int rc = cuda_ok(cudaMemcpyAsync(host_slot, result[0], res_bytes, cudaMemcpyDeviceToHost, s), "memcpy D2H results")) {
                return rc;
            }
        }
        if (result_b && !(n_episodes & 1)) {   // leave the last episode's results in the descriptor's own region ...
            // ... once the download stream has finished reading region 0 (episode n-2's D2H may still be in flight)
            cudaStreamWaitEvent(s, g.downloaded[0], 0);
            if (int rc = cuda_ok(cudaMemcpyAsync(result[0], result[1], res_bytes, cudaMemcpyDeviceToDevice, s), "memcpy D2D results")) return rc;
        }
        return 0;
    };
    const int rc_enqueue = enqueue();
    const auto t_enqueued = std::chrono::steady_clock::now();
    // drain everything that was enqueued — also on the error path, so that no copy is in flight into caller memory
    // when this call returns
    const cudaError_t e1 = cudaStreamSynchronize(s), e2 = cudaStreamSynchronize(g.copy), e3 = cudaStreamSynchronize(g.down);
    if (rc_enqueue) return rc_enqueue;
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
        set_error("ia2c_train_episodes_host: stream sync: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
        cudaGetLastError();
        return IA2C_ERR_CUDA;
    }
    if (trace) {
        double copy_ms = 0, comp_ms = 0;
        for (int k = 0; k < n_traced; ++k) {
            float a = 0, b = 0, c0 = 0, c1 = 0;
            cudaEventElapsedTime(&a, tr_ev[k][0], tr_ev[k][1]);
            cudaEventElapsedTime(&b, tr_ev[k][2], tr_ev[k][3]);
            cudaEventElapsedTime(&c0, tr_ev[0][0], tr_ev[k][0]);   // copy start / compute start relative to the first copy
            cudaEventElapsedTime(&c1, tr_ev[0][0], tr_ev[k][2]);
            copy_ms += a;
            comp_ms += b;
            if (k < 8 || k >= n_traced - 2)
                fprintf(stderr, "  episode %2d: H2D starts %8.1f us, takes %6.1f us; kernels start %8.1f us, take %6.1f us\n", k, c0 * 1e3, a * 1e3,
                        c1 * 1e3, b * 1e3);
        }
        if (n_traced) fprintf(stderr, "  mean H2D %.1f us, mean kernels %.1f us per episode\n", copy_ms * 1e3 / n_traced, comp_ms * 1e3 / n_traced);
        for (int k = 0; k < n_traced; ++k)
            for (int j = 0; j < 4; ++j) cudaEventDestroy(tr_ev[k][j]);
        const auto t_done = std::chrono::steady_clock::now();
        fprintf(stderr, "ia2c_train_episodes_host: %d episodes, enqueue %.1f us/episode, total %.1f us/episode\n", n_episodes,
                std::chrono::duration<double, std::micro>(t_enqueued - t_begin).count() / n_episodes,
                std::chrono::duration<double, std::micro>(t_done - t_begin).count() / n_episodes);
    }
    return 0;
}

extern "C" int ia2c_train_episodes_host(const ia2c_episode_desc* d, ia2c_host_pipe* pipe, void* stage_b, void* result_b,
                                        int32_t n_episodes, const void* const* host_tapes, void* host_results, void* stream) {
    return episodes_host_impl(d, pipe, nullptr, 0, stage_b, result_b, n_episodes, host_tapes, host_results, stream);
}

extern "C" int ia2c_train_episodes_host_p2p(const ia2c_episode_desc* d, ia2c_host_pipe* pipe, const ia2c_peer_desc* peers,
                                            uint32_t epoch0, void* stage_b, void* result_b, int32_t n_episodes,
                                            const void* const* host_tapes, void* host_results, void* stream) {
    IA2C_REQUIRE(peers != nullptr, "ia2c_train_episodes_host_p2p: null peer descriptor");
    return episodes_host_impl(d, pipe, peers, epoch0, stage_b, result_b, n_episodes, host_tapes, host_results, stream);
}

// ------------------------------------------------------------------------------------------------
// Profiling entry point: one episode with a CUDA event between every kernel launch group (on the launching
// stream), synchronised at the end.  ms_out[5] = {rollout, critic gradient, critic reduce+Adam, actor gradient,
// actor reduce+Adam} in milliseconds, warm caches — what bench.py reports as per-kernel durations.
extern "C" int ia2c_train_episode_timed(const ia2c_episode_desc* d, float* host_ms_out, void* stream) {
    if (int rc = validate(d, "ia2c_train_episode_timed")) return rc;
    if (int rc = check_update_ptrs(d, "ia2c_train_episode_timed")) return rc;
    IA2C_REQUIRE(host_ms_out != nullptr, "ia2c_train_episode_timed: null output");
    cudaStream_t s = as_stream(stream);
    cudaEvent_t ev[6];
    for (auto& e : ev) if (cudaEventCreate(&e) != cudaSuccess) return check_launch("cudaEventCreate");
    int rc = 0;
    const int apply = !(d->flags & IA2C_FLAG_SKIP_ADAM);
    dim3 grid(grad_blocks(d), d->N);
    cudaEventRecord(ev[0], s);
    rc = ia2c_rollout(d, stream);
    cudaEventRecord(ev[1], s);
    if (!rc && !fused_critic(d)) { critic_grad_kernel<false><<<grid, kGradThreads, 0, s>>>(*d, d->partials, NoRuns{}); rc = check_launch("critic_grad_kernel"); }
    cudaEventRecord(ev[2], s);
    if (!rc) rc = run_reduce(d, 0, 1, apply, s);
    cudaEventRecord(ev[3], s);
    if (!rc) rc = launch_actor_grad(d, s);
    cudaEventRecord(ev[4], s);
    if (!rc) rc = run_reduce(d, 1, 1, apply, s);
    cudaEventRecord(ev[5], s);
    if (cudaStreamSynchronize(s) != cudaSuccess && !rc) rc = check_launch("stream sync");
    for (int i = 0; i < 5 && !rc; ++i) cudaEventElapsedTime(&host_ms_out[i], ev[i], ev[i + 1]);
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
}

extern "C" size_t ia2c_peer_inbox_bytes(const ia2c_episode_desc* d, int32_t world) {
    if (!d || world < 1) return 0;
    return (size_t)2 * world * d->N * (kCriticP + 1) * sizeof(unsigned long long);   // two parities x world slots of N*(P_max+1) words
}

extern "C" int ia2c_allreduce_adam(const ia2c_episode_desc* d, int32_t which, const ia2c_peer_desc* peers, uint32_t epoch,
                                   int32_t adam_step, void* stream) {
    if (int rc = validate(d, "ia2c_allreduce_adam")) return rc;
    if (int rc = check_update_ptrs(d, "ia2c_allreduce_adam")) return rc;
    IA2C_REQUIRE(which == 0 || which == 1, "ia2c_allreduce_adam: which=%d", which);
    IA2C_REQUIRE(peers && peers->world >= 1 && peers->world <= 8 && peers->rank >= 0 && peers->rank < peers->world,
                 "ia2c_allreduce_adam: bad peer descriptor");
    IA2C_REQUIRE(epoch > 0 && adam_step > 0, "ia2c_allreduce_adam: epoch and adam_step start at 1");
    for (int p = 0; p < peers->world; ++p)
        IA2C_REQUIRE(peers->inbox[p] && ((uintptr_t)peers->inbox[p] & 7) == 0, "ia2c_allreduce_adam: null or misaligned peer inbox %d", p);
    IA2C_REQUIRE(((uintptr_t)peers->mc_inbox & 7) == 0, "ia2c_allreduce_adam: misaligned multicast inbox");
    cudaStream_t s = as_stream(stream);
    ReduceArgs R = make_reduce_args(*d, which, which == 0 ? critic_partial_blocks(d) : actor_partial_blocks(d));
    R.apply_adam = 1;
    PeerArgs X;
    X.rank = peers->rank;
    X.world = peers->world;
    for (int p = 0; p < 8; ++p) {
        X.inbox[p] = p < peers->world ? reinterpret_cast<unsigned long long*>(peers->inbox[p]) : nullptr;
        X.error[p] = p < peers->world ? peers->error[p] : nullptr;
    }
    X.mc_inbox = reinterpret_cast<unsigned long long*>(peers->mc_inbox);
    X.epoch = epoch;
    X.t = adam_step;
    X.stride = (int64_t)d->N * (kCriticP + 1);
    X.timeout_ns = (unsigned long long)(peers->timeout_us ? peers->timeout_us : 2000000u) * 1000ull;
    const int chunks_per_agent = ceil_div((which == 0 ? kCriticP : kActorP) + 1, 32);
    const int total = d->N * chunks_per_agent;
    const int grid = std::min(total, kSMs);          // persistent: every block is resident
    return launch_pdl("allreduce_adam_kernel", allreduce_adam_kernel, dim3(grid), dim3(32 * kReduceSlices), 0, s, R, X, total, chunks_per_agent);
}

// ------------------------------------------------------------------------------------------------
// A batch of R independent runs in the four launches of one episode (include/ia2c_b200.h: ia2c_train_episode_runs).  Every
// kernel takes the run as one more grid dimension and partitions each run as a standalone run of E envs is partitioned:
// rollout grid (rollout_fused_blocks(E, N), R), actor-gradient grid (grad_blocks(E), R * N), reduce grid (R * N, chunks).
extern "C" size_t ia2c_runs_partials_floats(const ia2c_episode_desc* d, int32_t runs) {
    if (runs < 1) return 0;
    return (size_t)runs * ia2c_episode_partials_floats(d);
}

static int validate_runs(const ia2c_episode_desc* d, const ia2c_runs_desc* r) {
    const char* who = "ia2c_train_episode_runs";
    if (int rc = validate(d, who)) return rc;
    IA2C_REQUIRE(r != nullptr, "%s: null runs descriptor", who);
    IA2C_REQUIRE(r->runs >= 1, "%s: runs=%d, need at least 1", who, r->runs);
    IA2C_REQUIRE((int64_t)r->runs * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS = %d", who,
                 (long long)r->runs * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(r->seed != nullptr, "%s: null seed array (one Philox key per run)", who);
    auto unsupported = [](const char* what, const char* who) {
        set_error("%s: %s", who, what);
        return IA2C_ERR_UNSUPPORTED;
    };
    if (!rollout_fused_supported(d->N, d->M)) {
        set_error("%s: N=%d M=%d has no fused instantiation (batches need N <= 8 with M = 5, or N = 2 with M = 3)", who, d->N, d->M);
        return IA2C_ERR_UNSUPPORTED;
    }
    if (d->env_offset != 0 || d->E_total != d->E)
        return unsupported("batches run on one GPU: desc.env_offset must be 0 and desc.E_total == desc.E (envs per run)", who);
    if (d->inj_actions || d->inj_u_action || d->inj_u_belief) return unsupported("injected replay tapes are not supported in batches", who);
    if (d->state_trace || d->reward_f64 || d->pred_dump || d->belief_dump || d->adv_dump || d->target_dump)
        return unsupported("parity dumps are not supported in batches", who);
    if (d->flags & ~(IA2C_FLAG_FUSED_ROLLOUT | IA2C_FLAG_FUSED_CRITIC | IA2C_FLAG_ACTOR_COLUMNS))
        return unsupported("desc.flags may carry only FUSED_ROLLOUT, FUSED_CRITIC and ACTOR_COLUMNS", who);
    IA2C_REQUIRE(d->env_state && d->env_hist && d->env_cls && d->env_elapsed && d->ep_return && d->belief_records && d->filter_action,
                 "%s: null env/belief pointer", who);
    IA2C_REQUIRE(d->critic_grad && d->actor_grad && d->critic_m && d->critic_v && d->actor_m && d->actor_v && d->actor_grad_accum &&
                     d->critic_step && d->actor_step && d->loss_out, "%s: null optimiser pointer", who);
    IA2C_REQUIRE(d->partials && d->partials_floats >= ia2c_runs_partials_floats(d, r->runs), "%s: partials workspace too small (%zu < %zu)",
                 who, d->partials_floats, ia2c_runs_partials_floats(d, r->runs));
    return 0;
}

// reduce + Adam of a batch's R * N critics (which = 0) or actors (1), each net with its run's learning rate; `e` carries the
// internal flags, which select the partial-row count of the producing kernel
static int reduce_runs(const ia2c_episode_desc& e, const ia2c_runs_desc* r, int which, cudaStream_t s) {
    const int nets = r->runs * e.N;
    ReduceArgs A = make_reduce_args(e, which, which == 0 ? critic_partial_blocks(&e) : actor_partial_blocks(&e));
    A.loss_out = e.loss_out + (which == 0 ? 0 : nets);
    const ReduceRuns rr = {which == 0 ? r->lr_critic : r->lr_actor, e.N};
    dim3 grid(nets, ceil_div(A.P + 1, 32));
    return launch_pdl("reduce_adam_kernel", reduce_adam_kernel<true>, grid, dim3(32 * kReduceSlices), 0, s, A, rr);
}

// One episode of a batch (N <= 8); p != nullptr: with frozen partners per env.
static int train_runs_impl(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const EnvPartners* p, void* stream) {
    cudaStream_t s = as_stream(stream);
    const int R = r->runs, nets = R * d->N;
    ia2c_episode_desc e = *d;
    e.flags = IA2C_FLAG_FUSED_ROLLOUT | IA2C_FLAG_FUSED_CRITIC | IA2C_FLAG_ACTOR_COLUMNS;
    if (int rc = rollout_fused_launch(&e, r, p, s)) return rc;
    if (int rc = reduce_runs(e, r, 0, s)) return rc;
    dim3 grid(grad_blocks(&e), nets);
    if (int rc = launch_pdl("actor_grad_kernel", actor_grad_kernel<true>, grid, dim3(kGradThreads), 0, s, e, e.partials, *r)) return rc;
    return reduce_runs(e, r, 1, s);
}

extern "C" int ia2c_train_episode_runs(const ia2c_episode_desc* d, const ia2c_runs_desc* r, void* stream) {
    if (int rc = validate_runs(d, r)) return rc;
    return train_runs_impl(d, r, nullptr, stream);
}

// ------------------------------------------------------------------------------------------------
// A batch of R independent Org-N runs (9 <= N <= 256) in the six launches of one episode (include/ia2c_b200.h:
// ia2c_train_episode_runs_many): the standalone N > 8 path of ia2c_rollout + the column actor kernel, every kernel with the run as
// one more grid dimension and each run partitioned exactly as a standalone run of E envs.
static int validate_runs_many(const ia2c_episode_desc* d, const ia2c_runs_desc* r) {
    const char* who = "ia2c_train_episode_runs_many";
    if (int rc = validate(d, who)) return rc;
    IA2C_REQUIRE(r != nullptr, "%s: null runs descriptor", who);
    IA2C_REQUIRE(r->runs >= 1, "%s: runs=%d, need at least 1", who, r->runs);
    IA2C_REQUIRE((int64_t)r->runs * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS = %d", who,
                 (long long)r->runs * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(r->seed != nullptr, "%s: null seed array (one Philox key per run)", who);
    auto unsupported = [](const char* what, const char* who) {
        set_error("%s: %s", who, what);
        return IA2C_ERR_UNSUPPORTED;
    };
    if (d->N <= 8) {
        set_error("%s: N=%d: batches of N <= 8 agents run on the fused path, ia2c_train_episode_runs", who, d->N);
        return IA2C_ERR_UNSUPPORTED;
    }
    if (d->N > 256) {
        set_error("%s: N=%d above 256 (the per-step env / actor kernels have no batched form)", who, d->N);
        return IA2C_ERR_UNSUPPORTED;
    }
    if (d->env_offset != 0 || d->E_total != d->E)
        return unsupported("batches run on one GPU: desc.env_offset must be 0 and desc.E_total == desc.E (envs per run)", who);
    if (d->inj_actions || d->inj_u_action || d->inj_u_belief) return unsupported("injected replay tapes are not supported in batches", who);
    if (d->state_trace || d->reward_f64 || d->pred_dump || d->belief_dump || d->adv_dump || d->target_dump)
        return unsupported("parity dumps are not supported in batches", who);
    if (d->flags != IA2C_FLAG_ACTOR_COLUMNS)
        return unsupported("desc.flags must be exactly ACTOR_COLUMNS (the batch runs the column actor kernel)", who);
    IA2C_REQUIRE(d->env_state && d->env_hist && d->env_cls && d->env_elapsed && d->ep_return && d->belief_records && d->filter_action,
                 "%s: null env/belief pointer", who);
    IA2C_REQUIRE(d->critic_grad && d->actor_grad && d->critic_m && d->critic_v && d->actor_m && d->actor_v && d->actor_grad_accum &&
                     d->critic_step && d->actor_step && d->loss_out, "%s: null optimiser pointer", who);
    IA2C_REQUIRE(d->partials && d->partials_floats >= ia2c_runs_partials_floats(d, r->runs), "%s: partials workspace too small (%zu < %zu)",
                 who, d->partials_floats, ia2c_runs_partials_floats(d, r->runs));
    return 0;
}

// One episode of a batch (9 <= N <= 256); p != nullptr: with frozen partners per env.
static int train_runs_many_impl(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const EnvPartners* p, void* stream) {
    cudaStream_t s = as_stream(stream);
    const int R = r->runs, nets = R * d->N;
    ia2c_episode_desc e = *d;
    e.flags = IA2C_FLAG_ACTOR_COLUMNS;   // both reductions sum grad_blocks(E) partial rows per net
    const ManyPlan mp = p ? many_plan<true, true>(&e, R) : many_plan<true>(&e, R);
    const dim3 many_grid((unsigned)mp.blocks, (unsigned)R);
    if (int rc = p ? launch_pdl("rollout_many_kernel", rollout_many_kernel<true, true>, many_grid, dim3(mp.threads), mp.smem, s, e,
                                mp.envs_per_block, *r, *p)
                   : launch_pdl("rollout_many_kernel", rollout_many_kernel<true>, many_grid, dim3(mp.threads), mp.smem, s, e,
                                mp.envs_per_block, *r, NoPartners{}))
        return rc;
    if (int rc = belief_pairs_episode_runs_launch(&e, r, s)) return rc;
    const dim3 grid(grad_blocks(&e), nets);
    if (int rc = launch_pdl("critic_grad_kernel", critic_grad_kernel<true>, grid, dim3(kGradThreads), 0, s, e, e.partials, *r)) return rc;
    if (int rc = reduce_runs(e, r, 0, s)) return rc;
    if (int rc = launch_pdl("actor_grad_kernel", actor_grad_kernel<true>, grid, dim3(kGradThreads), 0, s, e, e.partials, *r)) return rc;
    return reduce_runs(e, r, 1, s);
}

extern "C" int ia2c_train_episode_runs_many(const ia2c_episode_desc* d, const ia2c_runs_desc* r, void* stream) {
    if (int rc = validate_runs_many(d, r)) return rc;
    return train_runs_many_impl(d, r, nullptr, stream);
}

// ------------------------------------------------------------------------------------------------
// Frozen partners per env (include/ia2c_b200.h: ia2c_train_episode_env_partners): the episode entry points above with the
// PARTNERS instantiations of the rollout kernels; validate_env_partners (partners.cu) refuses every path that has none.
extern "C" int ia2c_rollout_env_partners(const ia2c_episode_desc* d, const ia2c_env_partner_desc* p, void* stream) {
    const char* who = "ia2c_rollout_env_partners";
    if (int rc = validate_env_partners(d, nullptr, p, who)) return rc;
    if (int rc = check_rollout(d, who)) return rc;
    const EnvPartners ep = env_partners_arg(p);
    return rollout_launch(d, &ep, stream);
}

extern "C" int ia2c_train_episode_env_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p,
                                               void* stream) {
    const char* who = "ia2c_train_episode_env_partners";
    if (int rc = validate_env_partners(d, r, p, who)) return rc;
    const EnvPartners ep = env_partners_arg(p);
    if (!r) {
        if (int rc = check_rollout(d, who)) return rc;
        if (int rc = check_update_ptrs(d, who)) return rc;
        return train_episode_impl(d, &ep, stream);
    }
    if (d->N <= 8) {
        if (int rc = validate_runs(d, r)) return rc;
        return train_runs_impl(d, r, &ep, stream);
    }
    if (int rc = validate_runs_many(d, r)) return rc;
    return train_runs_many_impl(d, r, &ep, stream);
}

// reduce_adam_kernel<true> for `nets` nets of P entries with one learning rate per net (lr_per_net, or A.lr where NULL): the
// native A2C trainer (a2c.cu) reduces and steps its R actor and R critic rows with it.
int ia2c::reduce_adam_runs_launch(const ReduceArgs& A, const double* lr_per_net, int nets, cudaStream_t s) {
    const ReduceRuns rr = {lr_per_net, 1};
    const dim3 grid(nets, ceil_div(A.P + 1, 32));
    return launch_pdl("reduce_adam_kernel", reduce_adam_kernel<true>, grid, dim3(32 * kReduceSlices), 0, s, A, rr);
}

#ifdef IA2C_STAGE_CLOCKS
extern "C" int ia2c_debug_kclocks(unsigned long long* out16) {
    return cudaMemcpyFromSymbol(out16, ia2c::g_kclock, sizeof(unsigned long long) * 16) == cudaSuccess ? 0 : -1;
}
#endif
