// evaluate.cu — frozen-policy evaluation of trained IA2C actors: R runs x E envs x K episodes in two launches.
//
// The IA2C actor reads only the observation, never the beliefs (ia2c.py: every sampler draws before a belief exists), and
// Org has 9 distinct observations.  An evaluation therefore needs neither the belief filter nor the critic: each actor's
// action distribution is tabulated once per call, with the forward and softmax the training samplers use (so the table
// holds the very probabilities they sample from), and the episodes sample from the table.  Nothing outside the
// descriptor's outputs is written: training state is untouched.
//
// Kernels in this file
//   eval_policy_kernel          one thread per (net, observation class c = 3 * prev_cls + cur_cls): forward_regnet +
//                               softmax_inplace -> policy[R*N, 9, 3]; the same launch zeroes action_counts.
//   eval_episodes_kernel<WIDE>  one episode of T Org steps per item (episode k, env e) of run blockIdx.y, from the reset
//                               state, with the same-step autoreset at max_episode_steps (Q14) and the fp64 return summed in
//                               step order, as the training rollouts compute them.  The run's table sits in shared memory.
//                               !WIDE (N <= 8): one thread per item.  WIDE: one warp per item; lane l owns the agent quads
//                               q = l + 32 j (agents 4q .. 4q+3), one Philox block each, and every lane steps its copy of
//                               the env from the butterfly-reduced counts (warp-uniform, nothing to broadcast).
//                               Action counts: registers per item, shared memory per block, one u64 atomicAdd per block
//                               and entry (integer sums: the same in any order).
//   lineup_policy_kernel        cross-play (ia2c_evaluate_lineups): the pool's table as eval_policy_kernel computes it, and the
//                               lineups' action_counts zeroed (P * N * 3 of them, independent of the pool's size).
//   lineup_episodes_kernel<WIDE> eval_episodes_kernel's body over lineup p = blockIdx.z * gridDim.y + blockIdx.y, the block's
//                               table gathered from the lineup's pool rows (a row out of range: NaN returns, no counts).
//   lineup_stats_kernel         one warp per lineup: the fixed-order return_sum and return_m2 of its K * E returns.
#include <algorithm>
#include <climits>

#include "common.cuh"
#include "mlp_f2.cuh"

namespace ia2c {
namespace {

constexpr int F = IA2C_OBS_FEATURES, A = IA2C_AGENT_ACTIONS;
constexpr int kClasses = 9;                       // 3 previous x 3 current observation classes
constexpr int kRow = kClasses * A;                // table floats per net
constexpr uint32_t kStreamEval = 4;               // Philox stream of the evaluation sampler (DESIGN.md §4)
constexpr int kPolicyThreads = 128;
constexpr int kEvalThreads = 128;
constexpr int kStatsThreads = 256;                // lineup_stats_kernel: one warp per lineup
constexpr int kNarrowMaxN = 8;                    // one thread per item up to here, one warp per item above
constexpr int kWideChunks = (IA2C_EVAL_MAX_AGENTS + 127) / 128;   // 128 agents (32 lanes x 4) per chunk

__device__ __forceinline__ uint32_t pack_count(int a) { return a == 0 ? 1u : (a == 1 ? (1u << 10) : (1u << 20)); }
// per-item count of one agent: action 0 in the low, action 1 in the high 16 bits (T <= 65535); action 2 is T minus both
__device__ __forceinline__ uint32_t pack_count01(int a) { return a == 0 ? 1u : (a == 1 ? 0x10000u : 0u); }

// the 24-bit uniform philox_uniform_f32 makes of word .x, from any of the four words
__device__ __forceinline__ float word_uniform(uint32_t w) { return (float)(w >> 8) * 5.9604644775390625e-8f; }
__device__ __forceinline__ uint32_t word_of(const uint4& r, int w) { return w == 0 ? r.x : (w == 1 ? r.y : (w == 2 ? r.z : r.w)); }

// argmax with ties to the lowest index (torch.argmax)
__device__ __forceinline__ int argmax3(const float (&p)[A]) {
    int a = 0;
    float m = p[0];
    if (p[1] > m) { a = 1; m = p[1]; }
    if (p[2] > m) a = 2;
    return a;
}

// One action from table row p: greedy, or the inverse CDF at uniform u (the training samplers' function).
__device__ __forceinline__ int eval_action(const float* p, bool greedy, float u) {
    const float pr[A] = {p[0], p[1], p[2]};
    return greedy ? argmax3(pr) : sample_inverse_cdf<A>(pr, u);
}

// One Org step from the step's packed action counts, as rollout_many_kernel / rollout_fused_kernel take it.
__device__ __forceinline__ void eval_env_step(uint32_t packed, int N, int max_steps, int& s, int& prev_cls, int& cur_cls,
                                              int& elapsed, double& hist, double& ret) {
    int s2;
    double base;
    org_transition(s, packed & 1023, (packed >> 10) & 1023, (packed >> 20) & 1023, N, s2, base);
    double r = org_reward(base, hist);
    prev_cls = cur_cls;
    cur_cls = org_obs_class(s2);
    ret += r;                                                    // fp64, in step order (ia2c.py:102)
    ++elapsed;
    if (max_steps > 0 && elapsed >= max_steps) {                 // same-step autoreset (Q14)
        s2 = 2; r = 0.0; prev_cls = 1; cur_cls = 1; elapsed = 0;
    }
    s = s2;
    hist = r;
}

// Table row of thread idx = net * 9 + c: net's softmax at observation class c, into policy[idx * 3 ..].
__device__ __forceinline__ void policy_row(const float* actor_params, float* policy, int64_t idx) {
    const int64_t net = idx / kClasses;
    const int c = (int)(idx - net * kClasses);
    float flat[kActorP];
#pragma unroll
    for (int k = 0; k < kActorP; ++k) flat[k] = __ldcg(actor_params + net * kActorP + k);
    RegNet<A> w;
    load_regnet<A>(w, flat);
    float x[F], y[A];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x[k] = (k == c / 3) ? 1.f : 0.f;
        x[3 + k] = (k == c % 3) ? 1.f : 0.f;
    }
    forward_regnet<A>(w, x, y);
    softmax_inplace<A>(y);
#pragma unroll
    for (int o = 0; o < A; ++o) policy[idx * A + o] = y[o];
}

__global__ void __launch_bounds__(kPolicyThreads) eval_policy_kernel(const __grid_constant__ ia2c_eval_desc d) {
    pdl_prologue();   // the parameters may come from the training kernels just before; counts may still be summed into
    const int64_t nets = (int64_t)d.R * d.N;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < nets * A) d.action_counts[idx] = 0ull;
    if (idx >= nets * kClasses) return;
    policy_row(d.actor_params, d.policy, idx);
}

// The pool's table, and the lineups' counts zeroed: P * N * 3 of them, more or fewer than the pool's nets * 9 rows.
__global__ void __launch_bounds__(kPolicyThreads) lineup_policy_kernel(const __grid_constant__ ia2c_lineup_desc d) {
    pdl_prologue();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < (int64_t)d.P * d.N * A) d.action_counts[idx] = 0ull;
    if (idx < (int64_t)d.nets * kClasses) policy_row(d.actor_params, d.policy, idx);
}

template <bool WIDE>
__global__ void __launch_bounds__(kEvalThreads) eval_episodes_kernel(const __grid_constant__ ia2c_eval_desc d) {
    extern __shared__ __align__(16) float eval_smem[];
    const int N = d.N, T = d.T, run = blockIdx.y;
    float* tab = eval_smem;                                               // [N][9][3] of this run
    uint32_t* cnt = reinterpret_cast<uint32_t*>(eval_smem + N * kRow);    // [N][3] this block's counts
    for (int k = threadIdx.x; k < N * A; k += blockDim.x) cnt[k] = 0u;
    pdl_prologue();
    const float* src = d.policy + (int64_t)run * N * kRow;                // written by eval_policy_kernel: L2 path, after the wait
    for (int k = threadIdx.x; k < N * kRow; k += blockDim.x) tab[k] = __ldcg(src + k);
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const bool greedy = d.greedy != 0;
    const int64_t E = d.E, RE = E * d.R, items = E * d.episodes;
    const int64_t item = WIDE ? (int64_t)blockIdx.x * (kEvalThreads / 32) + (threadIdx.x >> 5)
                              : (int64_t)blockIdx.x * kEvalThreads + threadIdx.x;
    const bool live = item < items;
    const int64_t k = live ? item / E : 0, e = live ? item - k * E : 0;
    const uint32_t episode = d.episode0 + (uint32_t)k;
    const int quads = (N + 3) >> 2;
    const uint64_t row0 = (uint64_t)e * (uint64_t)quads;                  // Philox index of this env's first agent quad
    const float* tape = d.inj_u_action ? d.inj_u_action + ((int64_t)k * T * RE + (int64_t)run * E + e) * N : nullptr;
    int s = 2, prev_cls = 1, cur_cls = 1, elapsed = 0;
    double hist = 0.0, ret = 0.0;

    if constexpr (!WIDE) {
        uint32_t c01[kNarrowMaxN];
#pragma unroll
        for (int i = 0; i < kNarrowMaxN; ++i) c01[i] = 0u;
        if (live) {
            for (int t = 0; t < T; ++t) {
                const float* row = tab + 3 * (3 * prev_cls + cur_cls);
                uint32_t packed = 0u;
#pragma unroll
                for (int q = 0; q < kNarrowMaxN / 4; ++q) {
                    if (4 * q < N) {
                        uint4 r = make_uint4(0u, 0u, 0u, 0u);
                        if (!greedy && !tape) r = philox_draw(d.seed, kStreamEval, episode, (uint32_t)t, row0 + q);
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            const int i = 4 * q + w;
                            if (i < N) {
                                const float u = tape ? __ldcg(tape + i) : word_uniform(word_of(r, w));
                                const int a = eval_action(row + i * kRow, greedy, u);
                                c01[i] += pack_count01(a);
                                packed += pack_count(a);
                            }
                        }
                    }
                }
                eval_env_step(packed, N, d.max_episode_steps, s, prev_cls, cur_cls, elapsed, hist, ret);
                if (tape) tape += RE * N;
            }
#pragma unroll
            for (int i = 0; i < kNarrowMaxN; ++i) {
                if (i < N) {
                    const uint32_t c0 = c01[i] & 0xFFFFu, c1 = c01[i] >> 16;
                    atomicAdd(cnt + 3 * i, c0);
                    atomicAdd(cnt + 3 * i + 1, c1);
                    atomicAdd(cnt + 3 * i + 2, (uint32_t)T - c0 - c1);
                }
            }
            d.returns[(int64_t)run * items + item] = ret;
        }
    } else {
        uint32_t c01[kWideChunks][4];
#pragma unroll
        for (int j = 0; j < kWideChunks; ++j)
#pragma unroll
            for (int w = 0; w < 4; ++w) c01[j][w] = 0u;
        if (live) {   // warp-uniform
            for (int t = 0; t < T; ++t) {
                const float* row = tab + 3 * (3 * prev_cls + cur_cls);
                uint32_t packed = 0u;
#pragma unroll
                for (int j = 0; j < kWideChunks; ++j) {
                    if (128 * j >= N) break;                                   // warp-uniform
                    const int q = lane + 32 * j;
                    if (4 * q < N) {
                        uint4 r = make_uint4(0u, 0u, 0u, 0u);
                        if (!greedy && !tape) r = philox_draw(d.seed, kStreamEval, episode, (uint32_t)t, row0 + q);
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            const int i = 4 * q + w;
                            if (i < N) {
                                const float u = tape ? __ldcg(tape + i) : word_uniform(word_of(r, w));
                                const int a = eval_action(row + i * kRow, greedy, u);
                                c01[j][w] += pack_count01(a);
                                packed += pack_count(a);
                            }
                        }
                    }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, off);
                eval_env_step(packed, N, d.max_episode_steps, s, prev_cls, cur_cls, elapsed, hist, ret);
                if (tape) tape += RE * N;
            }
#pragma unroll
            for (int j = 0; j < kWideChunks; ++j) {
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const int i = 4 * (lane + 32 * j) + w;
                    if (i < N) {
                        const uint32_t c0 = c01[j][w] & 0xFFFFu, c1 = c01[j][w] >> 16;
                        atomicAdd(cnt + 3 * i, c0);
                        atomicAdd(cnt + 3 * i + 1, c1);
                        atomicAdd(cnt + 3 * i + 2, (uint32_t)T - c0 - c1);
                    }
                }
            }
            if (lane == 0) d.returns[(int64_t)run * items + item] = ret;
        }
    }
    __syncthreads();
    unsigned long long* out = d.action_counts + (int64_t)run * N * A;
    for (int i = threadIdx.x; i < N * A; i += blockDim.x)
        if (cnt[i]) atomicAdd(out + i, (unsigned long long)cnt[i]);
}

// Cross-play: eval_episodes_kernel's body over lineup p, with the block's table gathered from the lineup's pool rows (a row
// outside [0, nets): NaN returns, no counts) and outputs and tape indexed by p as a batch indexes its runs.  A copy rather than
// a body shared with eval_episodes_kernel: inlined into it, a shared body changes that kernel's instruction schedule.
template <bool WIDE>
__global__ void __launch_bounds__(kEvalThreads) lineup_episodes_kernel(const __grid_constant__ ia2c_lineup_desc d) {
    extern __shared__ __align__(16) float eval_smem[];
    const int N = d.N, T = d.T, run = (int)(blockIdx.z * gridDim.y + blockIdx.y);   // lineup p: P may exceed 65535
    if (run >= d.P) return;
    float* tab = eval_smem;                                               // [N][9][3] of this lineup
    uint32_t* cnt = reinterpret_cast<uint32_t*>(eval_smem + N * kRow);    // [N][3] this block's counts
    for (int k = threadIdx.x; k < N * A; k += blockDim.x) cnt[k] = 0u;
    pdl_prologue();
    // lineups and table after the wait, through L2 (the table is the previous launch's output)
    int* row_of = reinterpret_cast<int*>(cnt + N * A);               // [N] pool row of each seat
    int miss = 0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const int r = __ldcg(d.lineups + (int64_t)run * N + i);
        miss |= r < 0 || r >= d.nets;
        row_of[i] = r;
    }
    const bool bad = __syncthreads_or(miss) != 0;
    if (!bad)
        for (int k = threadIdx.x; k < N * kRow; k += blockDim.x) {
            const int i = k / kRow;
            tab[k] = __ldcg(d.policy + (int64_t)row_of[i] * kRow + (k - i * kRow));
        }
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const bool greedy = d.greedy != 0;
    const int64_t E = d.E, RE = E * d.P, items = E * d.episodes;
    const int64_t item = WIDE ? (int64_t)blockIdx.x * (kEvalThreads / 32) + (threadIdx.x >> 5)
                              : (int64_t)blockIdx.x * kEvalThreads + threadIdx.x;
    const bool live = item < items;
    const int64_t k = live ? item / E : 0, e = live ? item - k * E : 0;
    const uint32_t episode = d.episode0 + (uint32_t)k;
    const int quads = (N + 3) >> 2;
    const uint64_t row0 = (uint64_t)e * (uint64_t)quads;                  // Philox index of this env's first agent quad
    if (bad) {   // block-uniform: no barrier follows
        if (live && (!WIDE || lane == 0)) d.returns[(int64_t)run * items + item] = __longlong_as_double(0x7FF8000000000000ll);
        return;
    }
    const float* tape = d.inj_u_action ? d.inj_u_action + ((int64_t)k * T * RE + (int64_t)run * E + e) * N : nullptr;
    int s = 2, prev_cls = 1, cur_cls = 1, elapsed = 0;
    double hist = 0.0, ret = 0.0;

    if constexpr (!WIDE) {
        uint32_t c01[kNarrowMaxN];
#pragma unroll
        for (int i = 0; i < kNarrowMaxN; ++i) c01[i] = 0u;
        if (live) {
            for (int t = 0; t < T; ++t) {
                const float* row = tab + 3 * (3 * prev_cls + cur_cls);
                uint32_t packed = 0u;
#pragma unroll
                for (int q = 0; q < kNarrowMaxN / 4; ++q) {
                    if (4 * q < N) {
                        uint4 r = make_uint4(0u, 0u, 0u, 0u);
                        if (!greedy && !tape) r = philox_draw(d.seed, kStreamEval, episode, (uint32_t)t, row0 + q);
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            const int i = 4 * q + w;
                            if (i < N) {
                                const float u = tape ? __ldcg(tape + i) : word_uniform(word_of(r, w));
                                const int a = eval_action(row + i * kRow, greedy, u);
                                c01[i] += pack_count01(a);
                                packed += pack_count(a);
                            }
                        }
                    }
                }
                eval_env_step(packed, N, d.max_episode_steps, s, prev_cls, cur_cls, elapsed, hist, ret);
                if (tape) tape += RE * N;
            }
#pragma unroll
            for (int i = 0; i < kNarrowMaxN; ++i) {
                if (i < N) {
                    const uint32_t c0 = c01[i] & 0xFFFFu, c1 = c01[i] >> 16;
                    atomicAdd(cnt + 3 * i, c0);
                    atomicAdd(cnt + 3 * i + 1, c1);
                    atomicAdd(cnt + 3 * i + 2, (uint32_t)T - c0 - c1);
                }
            }
            d.returns[(int64_t)run * items + item] = ret;
        }
    } else {
        uint32_t c01[kWideChunks][4];
#pragma unroll
        for (int j = 0; j < kWideChunks; ++j)
#pragma unroll
            for (int w = 0; w < 4; ++w) c01[j][w] = 0u;
        if (live) {   // warp-uniform
            for (int t = 0; t < T; ++t) {
                const float* row = tab + 3 * (3 * prev_cls + cur_cls);
                uint32_t packed = 0u;
#pragma unroll
                for (int j = 0; j < kWideChunks; ++j) {
                    if (128 * j >= N) break;                                   // warp-uniform
                    const int q = lane + 32 * j;
                    if (4 * q < N) {
                        uint4 r = make_uint4(0u, 0u, 0u, 0u);
                        if (!greedy && !tape) r = philox_draw(d.seed, kStreamEval, episode, (uint32_t)t, row0 + q);
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            const int i = 4 * q + w;
                            if (i < N) {
                                const float u = tape ? __ldcg(tape + i) : word_uniform(word_of(r, w));
                                const int a = eval_action(row + i * kRow, greedy, u);
                                c01[j][w] += pack_count01(a);
                                packed += pack_count(a);
                            }
                        }
                    }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, off);
                eval_env_step(packed, N, d.max_episode_steps, s, prev_cls, cur_cls, elapsed, hist, ret);
                if (tape) tape += RE * N;
            }
#pragma unroll
            for (int j = 0; j < kWideChunks; ++j) {
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const int i = 4 * (lane + 32 * j) + w;
                    if (i < N) {
                        const uint32_t c0 = c01[j][w] & 0xFFFFu, c1 = c01[j][w] >> 16;
                        atomicAdd(cnt + 3 * i, c0);
                        atomicAdd(cnt + 3 * i + 1, c1);
                        atomicAdd(cnt + 3 * i + 2, (uint32_t)T - c0 - c1);
                    }
                }
            }
            if (lane == 0) d.returns[(int64_t)run * items + item] = ret;
        }
    }
    __syncthreads();
    unsigned long long* out = d.action_counts + (int64_t)run * N * A;
    for (int i = threadIdx.x; i < N * A; i += blockDim.x)
        if (cnt[i]) atomicAdd(out + i, (unsigned long long)cnt[i]);
}

// return_sum / return_m2 of lineup p (one warp each) over its n = episodes * E returns in returns[p] row-major order, in the
// header's order: 256 virtual lanes j (lane l holds j = l + 32 v, v < 8) add x[j], x[j + 256], ... from +0.0, then the
// halving tree s[j] += s[j + w] for w = 128 .. 1 (in registers down to w = 32, then across lanes).
__device__ __forceinline__ double lineup_lane_sum(const double* x, int64_t n, bool sq, double mean) {
    const int lane = threadIdx.x & 31;
    double s[8];
#pragma unroll
    for (int v = 0; v < 8; ++v) s[v] = 0.0;
    for (int64_t j0 = lane; j0 < n; j0 += 256) {
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const int64_t j = j0 + 32 * v;
            if (j < n) {
                double y = __ldcg(x + j);
                if (sq) {
                    y = __dsub_rn(y, mean);
                    y = __dmul_rn(y, y);
                }
                s[v] = __dadd_rn(s[v], y);
            }
        }
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) s[v] = __dadd_rn(s[v], s[v + 4]);
#pragma unroll
    for (int v = 0; v < 2; ++v) s[v] = __dadd_rn(s[v], s[v + 2]);
    double t = __dadd_rn(s[0], s[1]);
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) {
        const double o = __shfl_down_sync(0xffffffffu, t, w);
        if (lane < w) t = __dadd_rn(t, o);
    }
    return __shfl_sync(0xffffffffu, t, 0);
}

__global__ void __launch_bounds__(kStatsThreads) lineup_stats_kernel(const __grid_constant__ ia2c_lineup_desc d) {
    pdl_prologue();   // returns are the previous launch's output: L2 path, after the wait
    const int64_t p = (int64_t)blockIdx.x * (kStatsThreads / 32) + (threadIdx.x >> 5);
    if (p >= d.P) return;   // warp-uniform
    const int64_t n = d.E * d.episodes;
    const double* x = d.returns + p * n;
    const double sum = lineup_lane_sum(x, n, false, 0.0);
    const double mean = __ddiv_rn(sum, (double)n);
    const double m2 = lineup_lane_sum(x, n, true, mean);
    if ((threadIdx.x & 31) == 0) {
        d.return_sum[p] = sum;
        d.return_m2[p] = m2;
    }
}

int64_t eval_items_per_block(int N) { return N > kNarrowMaxN ? kEvalThreads / 32 : kEvalThreads; }
size_t eval_smem_bytes(int N) { return (size_t)N * (kRow + A) * 4; }

int validate_eval(const ia2c_eval_desc* d, const char* who) {
    IA2C_REQUIRE(d != nullptr, "%s: null descriptor", who);
    IA2C_REQUIRE(d->actor_params && d->policy && d->returns && d->action_counts, "%s: null actor_params / policy / returns / "
                 "action_counts pointer", who);
    IA2C_REQUIRE(d->R >= 1 && d->R <= IA2C_EVAL_MAX_RUNS, "%s: R=%d outside 1..%d", who, d->R, IA2C_EVAL_MAX_RUNS);
    IA2C_REQUIRE(d->N >= 2 && d->N <= IA2C_EVAL_MAX_AGENTS, "%s: N=%d outside 2..%d", who, d->N, IA2C_EVAL_MAX_AGENTS);
    IA2C_REQUIRE((int64_t)d->R * d->N <= IA2C_MAX_RUN_NETS, "%s: R * N = %lld above IA2C_MAX_RUN_NETS (%d)", who,
                 (long long)d->R * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(d->E >= 1, "%s: E=%lld must be >= 1", who, (long long)d->E);
    IA2C_REQUIRE(d->episodes >= 1, "%s: episodes=%d must be >= 1", who, d->episodes);
    IA2C_REQUIRE(d->T >= 1 && d->T <= IA2C_EVAL_MAX_STEPS, "%s: T=%d outside 1..%d", who, d->T, IA2C_EVAL_MAX_STEPS);
    IA2C_REQUIRE(d->max_episode_steps >= 0, "%s: max_episode_steps=%d must be >= 0 (0: no time limit)", who, d->max_episode_steps);
    IA2C_REQUIRE(d->E <= (int64_t)INT_MAX * eval_items_per_block(d->N) / d->episodes,
                 "%s: E * episodes = %lld * %d items do not fit one grid", who, (long long)d->E, d->episodes);
    IA2C_REQUIRE((uint64_t)d->episode0 + (uint64_t)d->episodes <= (1ull << 32), "%s: episode0 + episodes = %llu above 2^32", who,
                 (unsigned long long)d->episode0 + (unsigned long long)d->episodes);
    IA2C_REQUIRE(!d->greedy || d->E * d->episodes == 1, "%s: greedy needs E = episodes = 1 (Org is deterministic: every greedy "
                 "episode of a run is the same), got E=%lld episodes=%d", who, (long long)d->E, d->episodes);
    IA2C_REQUIRE(!d->greedy || d->inj_u_action == nullptr, "%s: greedy takes no uniform tape", who);
    IA2C_REQUIRE(d->policy_floats >= ia2c_eval_policy_floats(d), "%s: policy workspace too small (%zu < %zu floats)", who,
                 d->policy_floats, ia2c_eval_policy_floats(d));
    return 0;
}

int validate_lineups(const ia2c_lineup_desc* d) {
    const char* who = "ia2c_evaluate_lineups";
    IA2C_REQUIRE(d != nullptr, "%s: null descriptor", who);
    IA2C_REQUIRE(d->actor_params && d->lineups && d->policy && d->returns && d->action_counts && d->return_sum && d->return_m2,
                 "%s: null actor_params / lineups / policy / returns / action_counts / return_sum / return_m2 pointer", who);
    IA2C_REQUIRE(d->N >= 2 && d->N <= IA2C_EVAL_MAX_AGENTS, "%s: N=%d outside 2..%d", who, d->N, IA2C_EVAL_MAX_AGENTS);
    IA2C_REQUIRE(d->nets >= 1, "%s: nets=%d must be >= 1", who, d->nets);
    IA2C_REQUIRE(d->P >= 1 && d->P <= IA2C_EVAL_MAX_LINEUPS, "%s: P=%d outside 1..%d", who, d->P, IA2C_EVAL_MAX_LINEUPS);
    IA2C_REQUIRE(d->E >= 1, "%s: E=%lld must be >= 1", who, (long long)d->E);
    IA2C_REQUIRE(d->episodes >= 1, "%s: episodes=%d must be >= 1", who, d->episodes);
    IA2C_REQUIRE(d->T >= 1 && d->T <= IA2C_EVAL_MAX_STEPS, "%s: T=%d outside 1..%d", who, d->T, IA2C_EVAL_MAX_STEPS);
    IA2C_REQUIRE(d->max_episode_steps >= 0, "%s: max_episode_steps=%d must be >= 0 (0: no time limit)", who, d->max_episode_steps);
    IA2C_REQUIRE(d->E <= (int64_t)INT_MAX * eval_items_per_block(d->N) / d->episodes,
                 "%s: E * episodes = %lld * %d items do not fit one grid", who, (long long)d->E, d->episodes);
    IA2C_REQUIRE((uint64_t)d->episode0 + (uint64_t)d->episodes <= (1ull << 32), "%s: episode0 + episodes = %llu above 2^32", who,
                 (unsigned long long)d->episode0 + (unsigned long long)d->episodes);
    IA2C_REQUIRE(!d->greedy || d->E * d->episodes == 1, "%s: greedy needs E = episodes = 1 (Org is deterministic: every greedy "
                 "episode of a lineup is the same), got E=%lld episodes=%d", who, (long long)d->E, d->episodes);
    IA2C_REQUIRE(!d->greedy || d->inj_u_action == nullptr, "%s: greedy takes no uniform tape", who);
    IA2C_REQUIRE(d->policy_floats >= (size_t)d->nets * kRow, "%s: policy workspace too small (%zu < nets * 27 = %zu floats)", who,
                 d->policy_floats, (size_t)d->nets * kRow);
    return 0;
}

}  // namespace
}  // namespace ia2c

using namespace ia2c;

extern "C" size_t ia2c_eval_policy_floats(const ia2c_eval_desc* d) {
    if (d == nullptr || d->R < 1 || d->N < 1) return 0;
    return (size_t)d->R * (size_t)d->N * (size_t)kRow;
}

extern "C" int ia2c_evaluate(const ia2c_eval_desc* d, void* stream) {
    if (int rc = validate_eval(d, "ia2c_evaluate")) return rc;
    cudaStream_t s = as_stream(stream);
    const int64_t nets = (int64_t)d->R * d->N;
    if (int rc = launch_pdl("eval_policy_kernel", eval_policy_kernel, dim3((unsigned)ceil_div(nets * kClasses, kPolicyThreads)),
                            dim3(kPolicyThreads), 0, s, *d))
        return rc;
    const int64_t items = d->E * d->episodes;
    const dim3 grid((unsigned)ceil_div(items, eval_items_per_block(d->N)), (unsigned)d->R);
    const size_t smem = eval_smem_bytes(d->N);
    if (d->N > kNarrowMaxN) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(eval_episodes_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return launch_pdl("eval_episodes_kernel<WIDE>", eval_episodes_kernel<true>, grid, dim3(kEvalThreads), smem, s, *d);
    }
    return launch_pdl("eval_episodes_kernel", eval_episodes_kernel<false>, grid, dim3(kEvalThreads), smem, s, *d);
}

extern "C" int ia2c_evaluate_lineups(const ia2c_lineup_desc* d, void* stream) {
    if (int rc = validate_lineups(d)) return rc;
    cudaStream_t s = as_stream(stream);
    const int64_t zero_and_rows = std::max<int64_t>((int64_t)d->nets * kClasses, (int64_t)d->P * d->N * A);
    if (int rc = launch_pdl("lineup_policy_kernel", lineup_policy_kernel, dim3((unsigned)ceil_div(zero_and_rows, kPolicyThreads)),
                            dim3(kPolicyThreads), 0, s, *d))
        return rc;
    const int64_t items = d->E * d->episodes;
    const unsigned gy = (unsigned)std::min<int>(d->P, 65535), gz = (unsigned)ceil_div(d->P, gy);
    const dim3 grid((unsigned)ceil_div(items, eval_items_per_block(d->N)), gy, gz);
    const size_t smem = eval_smem_bytes(d->N) + (size_t)d->N * sizeof(int);   // + the seats' pool rows
    int rc;
    if (d->N > kNarrowMaxN) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(lineup_episodes_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        rc = launch_pdl("lineup_episodes_kernel<WIDE>", lineup_episodes_kernel<true>, grid, dim3(kEvalThreads), smem, s, *d);
    } else {
        rc = launch_pdl("lineup_episodes_kernel", lineup_episodes_kernel<false>, grid, dim3(kEvalThreads), smem, s, *d);
    }
    if (rc) return rc;
    return launch_pdl("lineup_stats_kernel", lineup_stats_kernel, dim3((unsigned)ceil_div(d->P, kStatsThreads / 32)),
                      dim3(kStatsThreads), 0, s, *d);
}
