// rollout_fused.cu — persistent one-launch rollout (+ critic gradient) for small agent counts (N <= 8).
//
// Replaces the rollout part of the episode loop, ia2c.py:72-102, in ONE kernel launch — and, with
// IA2C_FLAG_FUSED_CRITIC, also the gradient computation of the critic phase, ia2c.py:104-114 — with
// everything on-chip: a lane owns one (env, agent) pair for the whole episode.
//
// The block is a WARP-SPECIALISED PIPELINE over the same 32 (env, agent) lanes; warp k works on the time step
// (iteration - offset_k) and the stages meet only through small shared-memory rings and ONE __syncthreads per
// iteration:
//   warp 0  Cf "critic"  (row  it-4)   critic forward on obs[t+1] (FFMA2, weights in registers) and the TD error
//                                      of row t; activations parked in shared memory; owns the W1/b1 gradient.
//   warp 1  A  "actor"   (step it-1)   Org transition -> observation -> actor forward (FFMA2, weights in
//                                      registers) -> sample.  Carries the recurrence env -> action -> env.
//   warp 2  B  "belief"  (step it-2)   the K fp64 belief updates (exact operation order), predicted actions,
//                                      partner mode.  Carries the recurrence posterior(t-1) -> posterior(t).
//   warp 3  R  "draws"   (step it)     the step's belief uniforms — device Philox4x32-10 or the injected tapes (the action
//                                      uniforms are drawn by warp 2, which has the slack); then
//           Cb "backprop"(obs  it-5)   ONE backward per observation with both output-gradient contributions
//                                      it receives (W3/W2 rows in registers); owns the W3/b3/W2/b2 gradient and
//                                      hands dz1 back to warp 0.  147 accumulators stay in registers all episode.
// The kernel is a pure dependent-latency chain (profiles/r01_ncu_full_summary.md: 3 % of peak warps, every
// pipe < 7 %): a single warp issues one instruction every ~3.5 cycles, so an episode costs
// (instructions of the slowest stage) x 3.5 cycles x (T+4) — splitting the work over warps that sit on
// different schedulers is what shortens it; the 140 other SM sub-partitions are idle anyway at E*N = 8192.
// Parameters are frozen during a rollout and envs are independent: no inter-block communication.
// The per-step kernels in trainer.cu / belief.cu remain the general path (any N) and the reference for this
// kernel's parity tests: both must write identical bytes.
#include "common.cuh"
#include "mlp_f2.cuh"

namespace ia2c {
namespace {

constexpr int F = IA2C_OBS_FEATURES, A = IA2C_AGENT_ACTIONS, J = IA2C_JOINT_ACTIONS;
constexpr int kRoles = 4;
constexpr int kBlock = 32 * kRoles;
constexpr int kRing = 8;

// Diagnostic build (-DIA2C_STAGE_CLOCKS, tools/stage_clocks.py): the stage warps of the first and the last block of episode 5
// print when they entered, left griddepcontrol.wait, started / ended the step loop and finished (ns since entry), and the
// cycles they spent between leaving one per-iteration barrier and reaching the next.
#ifdef IA2C_STAGE_CLOCKS
#define STAGE_CLOCK_INIT long long sc_work = 0, sc_t0 = clock64(); KCLOCK(sc_loop)
#define STAGE_SYNC() do { sc_work += clock64() - sc_t0; __syncthreads(); sc_t0 = clock64(); } while (0)
#else
#define STAGE_CLOCK_INIT
#define STAGE_SYNC() __syncthreads()
#endif
#define STAGE_CLOCK_EXIT(name) KCLOCK_PRINT(d.episode == 5 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) && lane == 0, \
    "rollout block %3d stage %-5s entry %llu: waited +%llu, loop +%llu .. +%llu (work %lld cycles), exit +%llu ns\n", (int)blockIdx.x, name, \
    sc_entry % 1000000000ull, sc_waited - sc_entry, sc_loop - sc_entry, sc_loop_end - sc_entry, sc_work, stage_ns() - sc_entry)

__device__ __forceinline__ uint32_t pack_count(int a) { return a == 0 ? 1u : (a == 1 ? (1u << 10) : (1u << 20)); }
__device__ __forceinline__ int mode3(int c0, int c1, int c2) {
    int best = 0, bc = c0;
    if (c1 > bc) { best = 1; bc = c1; }
    if (c2 > bc) { best = 2; }
    return best;
}
__device__ __forceinline__ int joint_index(int i, int n, int own, int other) {
    return (i < (i + 1) % n) ? own * A + other : other * A + own;   // SURVEY.md Q9
}
__device__ __forceinline__ void obs_from_cls(int packed, float (&x)[F]) {
    const int prev = packed & 3, cur = packed >> 2;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x[k] = (k == prev) ? 1.f : 0.f;
        x[3 + k] = (k == cur) ? 1.f : 0.f;
    }
}

// RUNS: a batch of independent runs (ia2c_train_episode_runs), blockIdx.y = run; see `run` below.
// PARTNERS: frozen partners per env (ia2c_train_episode_env_partners): a partner lane loads its env's pool row instead of its own.
template <int N, int M, bool CRITIC, bool RUNS, bool PARTNERS = false>
__global__ void __launch_bounds__(kBlock) rollout_fused_kernel(ia2c_episode_desc d, float* __restrict__ partials, RunsArg<RUNS> ra,
                                                               PartnerArg<PARTNERS> pa) {
    constexpr int K = N - 1;
    constexpr int G = N <= 2 ? 2 : (N <= 4 ? 4 : 8);     // lanes per env
    constexpr int EPW = 32 / G;
    __shared__ double tab[101];                          // k / 100, correctly rounded
    __shared__ double fa_s[N * M * A];
    __shared__ float ua_s[2][32];                        // action uniforms of step t        (slot t & 1)
    __shared__ double ub_s[4][K][32];                    // belief uniforms of step t        (slot t & 3)
    __shared__ int act_s[kRing][32];                     // sampled action of step t         (slot t & 7)
    __shared__ int cls_s[kRing][32];                     // obs classes prev | cur << 2 of step t
    __shared__ int ptrue_s[kRing][32];                   // mode of the others' true actions at step t
    __shared__ int ppred_s[kRing][32];                   // mode of the predicted actions at step t
    __shared__ float rew_s[kRing][32];                   // float32 reward of ROW t (known once step t+1 ran)
    __shared__ float2 hst_s[4][6][CRITIC ? 32 : 1];      // critic activations (h1 | h2 pairs) of obs[t], slot t & 3
    __shared__ float2 dz1_s[2][3][CRITIC ? 32 : 1];      // dL/dz1 of observation t (backprop warp -> W1-gradient owner), slot t & 1
    __shared__ float4 dy_s[4][CRITIC ? 32 : 1];          // row t's output gradients {jt, dQ[jt], nja, dQ'[nja]}, slot t & 3
    __shared__ float red_s[CRITIC ? kCriticP + 1 : 1][33];   // per-lane gradient partials for the block-wide reduction at the end
    KCLOCK(sc_entry);
    // A run of a batch owns net rows [run * N, (run + 1) * N) and env columns [run * E, (run + 1) * E) of an env axis of length
    // R * E (stride ES); `e` stays the env's index within its run, which keys its Philox counters.  ia2c_train_episode_runs
    // refuses replay tapes and parity dumps, so the code that indexes them by `e` and E never runs in a batch.
    const int run = RUNS ? (int)blockIdx.y : 0;
    const int net0 = run * N;
    pdl_release();
    // constants of the run (k/100, the agents' models): staged while the previous kernel of the stream may still be running
    for (int k = threadIdx.x; k <= 100; k += blockDim.x) tab[k] = __ddiv_rn((double)k, 100.0);
    for (int k = threadIdx.x; k < N * M * A; k += blockDim.x) fa_s[k] = d.filter_action[(int64_t)net0 * M * A + k];
    __syncthreads();
    pdl_wait();   // parameters (updated by the previous episode's Adam steps) are read only after this
    KCLOCK(sc_waited);

    const int role = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int sub = lane & (G - 1);
    const int leader = lane & ~(G - 1);
    const int64_t e = (int64_t)blockIdx.x * EPW + (lane / G);
    const int64_t E = d.E;
    const int64_t ES = RUNS ? E * gridDim.y : E;
    const int64_t ge = RUNS ? (int64_t)run * E + e : e;
    const bool live = e < E;            // uniform over the env's lane group
    const bool agent = live && sub < N; // this lane owns agent `sub`
    const int i = sub < N ? sub : 0;
    const int T = d.T;
    const int n_iter = CRITIC ? T + 7 : T + 3;   // steps 0..T through R(0) A(-1) B(-2); rows through Cf(-4), observations through Cb(-5)

    // ---- R: uniforms for step t (device Philox or the injected tapes) -> shared-memory rings, in two halves so that they
    //         can ride on different warps: with the critic stages present the backprop warp (the heaviest: 190
    //         instructions of backward per step) only makes the belief draws and the belief warp makes the action draws.
    // Injected tapes are fetched TWO steps ahead into registers (freshly copied tapes sit in HBM: a load issued in the
    // iteration that needs it would hold the whole block at the barrier for a DRAM round trip).
    const bool inj_a = d.inj_u_action != nullptr, inj_b = d.inj_u_belief != nullptr;
    float tua0 = 0.f, tua1 = 0.f;
    struct TapeB { double ub[K]; } tb0, tb1;
    auto fetch_a = [&](float& ua, int t) {
        if (inj_a && t <= T && agent) ua = __ldg(d.inj_u_action + ((int64_t)t * E + e) * N + i);
    };
    auto fetch_b = [&](TapeB& tp, int t) {
        if (inj_b && t <= T && agent) {
            const int64_t row = ((int64_t)t * E + e) * N + i;
#pragma unroll
            for (int jj = 0; jj < K; ++jj) tp.ub[jj] = __ldg(d.inj_u_belief + row * K + jj);
        }
    };
    auto draw_action_init = [&]() { fetch_a(tua0, 0); fetch_a(tua1, 1); };
    auto draw_belief_init = [&]() { fetch_b(tb0, 0); fetch_b(tb1, 1); };
    auto draw_action_from = [&](float& ua, int t) {
        if (t <= T && agent)
            ua_s[t & 1][lane] = inj_a ? ua
                                      : philox_uniform_f32(run_seed<RUNS>(d, ra, run), kStreamAction, d.episode, (uint32_t)t,
                                                           (uint64_t)((d.env_offset + e) * N + i));
        fetch_a(ua, t + 2);
    };
    auto draw_belief_from = [&](TapeB& tp, int t) {
        if (t <= T && agent) {
            if (inj_b) {
#pragma unroll
                for (int jj = 0; jj < K; ++jj) ub_s[t & 3][jj][lane] = tp.ub[jj];
            } else {
#pragma unroll
                for (int sl = 0; sl < (K + 3) / 4; ++sl) {
                    const uint4 r = philox_belief_quad(run_seed<RUNS>(d, ra, run), d.episode, (uint32_t)t, (uint64_t)((d.env_offset + e) * N + i), K, sl);
                    ub_s[t & 3][4 * sl][lane] = belief_word_to_unit_f64(r.x);
                    if (4 * sl + 1 < K) ub_s[t & 3][4 * sl + 1][lane] = belief_word_to_unit_f64(r.y);
                    if (4 * sl + 2 < K) ub_s[t & 3][4 * sl + 2][lane] = belief_word_to_unit_f64(r.z);
                    if (4 * sl + 3 < K) ub_s[t & 3][4 * sl + 3][lane] = belief_word_to_unit_f64(r.w);
                }
            }
        }
        fetch_b(tp, t + 2);
    };
    auto draw_action = [&](int t) {
        if (t & 1) draw_action_from(tua1, t); else draw_action_from(tua0, t);
    };
    auto draw_belief = [&](int t) {
        if (t & 1) draw_belief_from(tb1, t); else draw_belief_from(tb0, t);
    };

    if (role == 1) {
        // ================================================================ A: env + actor, step t = it - 1
        RegNet<A> net;
        if constexpr (PARTNERS) {   // the env's team, drawn once by every lane of its group; the leader logs it
            const int team = env_team(pa, run_seed<RUNS>(d, ra, run), d.episode, e, N);
            const int slot = team >= 0 && sub < N ? env_partner_slot(pa, i) : -1;
            if (live && sub == 0) pa.log[ge] = team;
            load_regnet<A>(net, slot >= 0 ? pa.rows + (int64_t)__ldcg(pa.teams + (int64_t)team * pa.S + slot) * kActorP
                                          : d.actor_params + (net0 + i) * kActorP);
        } else {
            load_regnet<A>(net, d.actor_params + (net0 + i) * kActorP);
        }
        int s = 2, prev_cls = 1, cur_cls = 1, elapsed = 0;   // env state, replicated in the group's lanes
        double hist = 0.0, ep_ret = 0.0;
        const double rcp10 = drcp_seq(10.0);
        int a = 0;
        // running output pointers (one bump per step instead of 64-bit index arithmetic)
        float* obs_p = d.obs + ge * F;
        uint8_t* act_p = d.act + ge * N + i;
        uint8_t* ptrue_p = d.partner_true + ge * N + i;
        const uint8_t* inj_p = d.inj_actions ? d.inj_actions + e * N + i : nullptr;
        float* rew_p = d.reward + ge;
        int32_t* trace_p = d.state_trace ? d.state_trace + e : nullptr;
        double* rew64_p = d.reward_f64 ? d.reward_f64 + e : nullptr;
        const int max_steps = d.max_episode_steps;
        STAGE_CLOCK_INIT;
        for (int it = 0; it < n_iter; ++it) {
            const int t = it - 1;
            if (t >= 0 && t <= T) {
                if (t > 0) {   // Org step from the actions of t-1 (every lane of the group computes it)
                    uint32_t packed = (sub < N) ? pack_count(a) : 0u;
#pragma unroll
                    for (int off = G >> 1; off > 0; off >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, off);
                    int s2;
                    double base;
                    org_transition(s, packed & 1023, (packed >> 10) & 1023, (packed >> 20) & 1023, N, s2, base);
                    double r = __dadd_rn(base, ddiv_with(hist, 10.0, rcp10));   // r' = base + r/10 (Org.py:55, Q17)
                    prev_cls = cur_cls;
                    cur_cls = org_obs_class(s2);
                    ep_ret += r;
                    rew_s[(t - 1) & (kRing - 1)][lane] = (float)r;
                    if (live && sub == 0) {
                        *rew_p = (float)r;                           // float32(r) as stored by ia2c.py:99
                        if (trace_p) *trace_p = s2;
                        if (rew64_p) *rew64_p = r;
                    }
                    rew_p += ES;
                    if (trace_p) trace_p += E;
                    if (rew64_p) rew64_p += E;
                    ++elapsed;
                    if (max_steps > 0 && elapsed >= max_steps) {     // same-step autoreset (Q14)
                        s2 = 2; r = 0.0; prev_cls = 1; cur_cls = 1; elapsed = 0;
                    }
                    s = s2;
                    hist = r;
                }
                float x[F];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    x[k] = (k == prev_cls) ? 1.f : 0.f;
                    x[3 + k] = (k == cur_cls) ? 1.f : 0.f;
                }
                if (live) {
#pragma unroll
                    for (int k = 0; k < F; ++k)
                        if ((k % G) == sub) obs_p[k] = x[k];
                }
                obs_p += ES * F;
                if (inj_p) {
                    a = agent ? *inj_p : 0;
                    inj_p += E * N;
                } else {
                    float y[A];
                    forward_regnet<A>(net, x, y);
                    softmax_inplace<A>(y);
                    a = sample_inverse_cdf<A>(y, agent ? ua_s[t & 1][lane] : 0.f);
                }
                uint32_t packed = (sub < N) ? pack_count(a) : 0u;
#pragma unroll
                for (int off = G >> 1; off > 0; off >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, off);
                const int c0 = packed & 1023, c1 = (packed >> 10) & 1023, c2 = (packed >> 20) & 1023;
                const int pt = mode3(c0 - (a == 0), c1 - (a == 1), c2 - (a == 2));
                const int slot = t & (kRing - 1);
                act_s[slot][lane] = a;                   // hand-over to the belief / critic warps
                cls_s[slot][lane] = prev_cls | (cur_cls << 2);
                ptrue_s[slot][lane] = pt;
                if (agent) {
                    *act_p = (uint8_t)a;
                    *ptrue_p = (uint8_t)pt;
                }
                act_p += ES * N;
                ptrue_p += ES * N;
            }
            STAGE_SYNC();
        }
        KCLOCK(sc_loop_end);
        if (live && sub == 0) {   // persist the final env state exactly as the per-step path leaves it
            d.env_state[ge] = s;
            d.env_hist[ge] = hist;
            d.env_elapsed[ge] = elapsed;
            d.ep_return[ge] = ep_ret;
            *reinterpret_cast<uchar2*>(d.env_cls + 2 * ge) = make_uchar2((unsigned char)prev_cls, (unsigned char)cur_cls);
        }
        STAGE_CLOCK_EXIT("A");
    } else if (role == 2) {
        // ================================================================ B: beliefs, step t = it - 2
        const double* fa = fa_s + i * M * A;
        int bel[K][M];
        const int prior_k = (int)rint(100.0 / M);        // round(1/M, 2) in hundredths (Q12)
#pragma unroll
        for (int jj = 0; jj < K; ++jj)
#pragma unroll
            for (int m = 0; m < M; ++m) bel[jj][m] = prior_k;
        int last_pred[K];
#pragma unroll
        for (int jj = 0; jj < K; ++jj) last_pred[jj] = 0;
        uint8_t* ppred_p = d.partner_pred + ge * N + i;
        if (CRITIC) draw_action_init();
        STAGE_CLOCK_INIT;
        for (int it = 0; it < n_iter; ++it) {
            if (CRITIC) draw_action(it);      // stage R's action half rides on this warp when the critic stages exist
            const int t = it - 2;
            if (t >= 0 && t <= T) {
                const int64_t row = ((int64_t)t * E + e) * N + i;
                int pc0 = 0, pc1 = 0, pc2 = 0;
#pragma unroll
                for (int jj = 0; jj < K; ++jj) {
                    const int j = jj + (jj >= i);        // modelled others in ascending order, skipping self
                    const int seen = act_s[t & (kRing - 1)][leader + j];
                    double prev[M], lik[A], b[M], pred[A], bp[M];
#pragma unroll
                    for (int m = 0; m < M; ++m) prev[m] = tab[bel[jj][m]];
#pragma unroll
                    for (int k = 0; k < A; ++k) lik[k] = (k == seen) ? 0.8 : 0.1;   // ia2c.py:53-58
                    const double u = ub_s[t & 3][jj][lane];
                    // operation order of SURVEY.md Appendix A.2 (kept in sync with belief.cu)
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        double acc = __dmul_rn(lik[0], __dmul_rn(fa[m * A + 0], prev[m]));
#pragma unroll
                        for (int k = 1; k < A; ++k) acc = __dadd_rn(acc, __dmul_rn(lik[k], __dmul_rn(fa[m * A + k], prev[m])));
                        bp[m] = acc;
                    }
                    double S = bp[0];
#pragma unroll
                    for (int m = 1; m < M; ++m) S = __dadd_rn(S, bp[m]);
                    const double rS = drcp_seq(S);
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        b[m] = ddiv_with(bp[m], S, rS);
                        bel[jj][m] = __double2int_rn(__dmul_rn(b[m], 100.0));   // rounded posterior = next prior (Q10)
                    }
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        double acc = 0.0;
#pragma unroll
                        for (int m = 0; m < M; ++m) acc = __dadd_rn(acc, __dmul_rn(b[m], fa[m * A + k]));
                        pred[k] = acc;
                    }
                    double c = pred[0];
                    int ap = 0;
                    bool found = u < c;
#pragma unroll
                    for (int k = 1; k < A; ++k) {
                        c = __dadd_rn(c, pred[k]);
                        if (!found && u < c) { ap = k; found = true; }
                    }
                    last_pred[jj] = ap;                  // falls through to 0 when u >= cumsum[-1] (Q11)
                    pc0 += (ap == 0); pc1 += (ap == 1); pc2 += (ap == 2);
                    if (agent && d.pred_dump) d.pred_dump[row * K + jj] = (uint8_t)ap;
                    if (agent && d.belief_dump) {
#pragma unroll
                        for (int m = 0; m < M; ++m) d.belief_dump[(row * K + jj) * M + m] = (uint8_t)bel[jj][m];
                    }
                }
                const int pp = mode3(pc0, pc1, pc2);
                ppred_s[t & (kRing - 1)][lane] = pp;
                if (agent) *ppred_p = (uint8_t)pp;
                ppred_p += ES * N;
            }
            STAGE_SYNC();
        }
        KCLOCK(sc_loop_end);
        if (agent) {   // persist the final beliefs exactly as the per-step path leaves them
#pragma unroll
            for (int jj = 0; jj < K; ++jj) {
                uint32_t lo = 0, hi = 0;
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    if (m < 4) lo |= (uint32_t)bel[jj][m] << (8 * m); else hi |= (uint32_t)bel[jj][m] << (8 * (m - 4));
                }
                hi |= (uint32_t)last_pred[jj] << 16;
                *reinterpret_cast<uint2*>(d.belief_records + ((ge * N + i) * (int64_t)K + jj) * IA2C_BELIEF_RECORD) = make_uint2(lo, hi);
            }
        }
        STAGE_CLOCK_EXIT("B");
    } else if (!CRITIC) {
        // ================================================================ R alone: draws (no critic stage)
        if (role == 3) { draw_action_init(); draw_belief_init(); }
        STAGE_CLOCK_INIT;
        for (int it = 0; it < n_iter; ++it) {
            if (role == 3) { draw_action(it); draw_belief(it); }
            STAGE_SYNC();
        }
    } else {
    // ==================================================================== R + Cf / Cb: draws, critic gradient
    constexpr int P = kCriticP, GN = F2<J>::G2;          // 148 floats = 74 float2 (147 gradient entries + the loss)
    const float inv_b = agent ? 1.f / (float)((int64_t)T * d.E_total) : 0.f;   // dead lanes contribute nothing

    if (role == 0) {
        // ================================================================ Cf: critic forward + TD error, row t = it - 4
        // One forward per observation: obs[t+1] is evaluated as the "next" observation of row t, its
        // activations are parked in shared memory for the backward stage, and the two Q values it will be
        // asked for (as bootstrap of row t, as Q(obs)[jt] of row t+1) are selected right away.
        const float gamma = run_gamma<RUNS>(d, ra, run);
        float loss = 0.f;
        float q_cur_jt = 0.f;
        RegNet<J> cnet;                      // this lane's critic, forward-paired weights in registers
        load_regnet<J>(cnet, d.critic_params + (int64_t)(net0 + i) * kCriticP);
        float2 gB[21];                       // W1 | b1 gradient (the backprop warp hands dz1 over, one iteration later)
#pragma unroll
        for (int k = 0; k < 21; ++k) gB[k] = make_float2(0.f, 0.f);
        float* target_p = d.target_dump ? d.target_dump + (int64_t)i * T * E + e : nullptr;
        auto park = [&](int slot, const float2 (&a1)[3], const float2 (&a2)[3]) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { hst_s[slot][k][lane] = a1[k]; hst_s[slot][3 + k][lane] = a2[k]; }
        };
        STAGE_CLOCK_INIT;
        for (int it = 0; it < n_iter; ++it) {
            const int t = it - 4;
            if (t >= 0 && t < T) {
                const int s0 = t & (kRing - 1), s1 = (t + 1) & (kRing - 1);
                const int jt = joint_index(i, N, act_s[s0][lane], ptrue_s[s0][lane]);    // ia2c.py:112
                const int nja = joint_index(i, N, act_s[s1][lane], ppred_s[s1][lane]);   // ia2c.py:104-105
                const int jt_next = joint_index(i, N, act_s[s1][lane], ptrue_s[s1][lane]);
                if (t == 0) {
                    float x0[F], q0[J];
                    float2 a1[3], a2[3];
                    obs_from_cls(cls_s[s0][lane], x0);
                    forward_regnet<J>(cnet, x0, a1, a2, q0);
                    park(0, a1, a2);
                    q_cur_jt = select_out<J>(q0, jt);
                }
                float xn[F], qn[J];
                float2 a1[3], a2[3];
                obs_from_cls(cls_s[s1][lane], xn);                   // next_obs[t] = obs[t+1]
                forward_regnet<J>(cnet, xn, a1, a2, qn);
                park((t + 1) & 3, a1, a2);
                const float target = rew_s[s0][lane] + gamma * select_out<J>(qn, nja);   // ia2c.py:110 (Q8)
                const float delta = target - q_cur_jt;
                q_cur_jt = select_out<J>(qn, jt_next);
                if (target_p) {
                    if (agent) *target_p = target;
                    target_p += E;
                }
                if (agent) loss = fmaf(delta, delta, loss);
                // output gradients of row t: dL/dQ(obs_t)[jt] and dL/dQ(next_obs_t)[nja] (residual gradient)
                dy_s[t & 3][lane] = make_float4(__int_as_float(jt), -2.f * delta * inv_b, __int_as_float(nja),
                                                2.f * gamma * delta * inv_b);
            }
            const int tb = it - 6;           // observation whose dz1 the backprop warp published last iteration
            if (tb >= 0 && tb <= T) {
                float xb[F];
                float2 dz1[3];
                obs_from_cls(cls_s[tb & (kRing - 1)][lane], xb);
#pragma unroll
                for (int k = 0; k < 3; ++k) dz1[k] = dz1_s[tb & 1][k][lane];
                accumulate_w1(xb, dz1, gB);
            }
            STAGE_SYNC();
        }
        KCLOCK(sc_loop_end);
        // hand the lane's partial sums to the block-wide reduction at the end of the kernel
#pragma unroll
        for (int k = 0; k < 21; ++k) { red_s[2 * k][lane] = gB[k].x; red_s[2 * k + 1][lane] = gB[k].y; }
        red_s[P][lane] = loss;
        if (lane < N && blockIdx.x == 0 && !(d.flags & IA2C_FLAG_SKIP_ADAM)) d.critic_step[net0 + lane] += 1;
        STAGE_CLOCK_EXIT("Cf");
    } else {
    // ==================================================================== Cb: critic backward, observation t = it - 5
    // ONE backward per observation with both output-gradient contributions it receives (from row t as
    // Q(obs_t)[jt_t], from row t-1 as the bootstrap Q(next_obs_{t-1})[nja_{t-1}]); 147 gradient accumulators
    // stay in registers for the whole episode.
    constexpr int GA = GN - 21;          // float2 accumulators for flat entries [42, 148): W2 | b2 | W3 | b3 (| loss slot)
    RegBack<J> back;
    load_regback<J>(back, d.critic_params + (int64_t)(net0 + i) * kCriticP);
    float2 gA[GA];
#pragma unroll
    for (int k = 0; k < GA; ++k) gA[k] = make_float2(0.f, 0.f);
    draw_belief_init();
    STAGE_CLOCK_INIT;
    for (int it = 0; it < n_iter; ++it) {
        draw_belief(it);             // stage R's belief half shares this warp
        const int t = it - 5;
        if (t >= 0 && t <= T) {
            int jt = -1, nja_prev = -1;
            float gq = 0.f, gqn_prev = 0.f;
            if (t < T) {
                const float4 v = dy_s[t & 3][lane];
                jt = __float_as_int(v.x);
                gq = v.y;
            }
            if (t > 0) {
                const float4 v = dy_s[(t - 1) & 3][lane];
                nja_prev = __float_as_int(v.z);
                gqn_prev = v.w;
            }
            float2 h1[3], h2[3], dz1[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) { h1[k] = hst_s[t & 3][k][lane]; h2[k] = hst_s[t & 3][3 + k][lane]; }
            bwd_regback<J>(back, h1, h2, [&](int o) { return (o == jt ? gq : 0.f) + (o == nja_prev ? gqn_prev : 0.f); }, gA, dz1);
#pragma unroll
            for (int k = 0; k < 3; ++k) dz1_s[t & 1][k][lane] = dz1[k];
        }
        STAGE_SYNC();
    }
    KCLOCK(sc_loop_end);
#pragma unroll
    for (int k = 0; k < GA; ++k) {
        if (42 + 2 * k < P) red_s[42 + 2 * k][lane] = gA[k].x;
        if (42 + 2 * k + 1 < P) red_s[42 + 2 * k + 1][lane] = gA[k].y;
    }
    STAGE_CLOCK_EXIT("R+Cb");
    }   // Cb
    }   // critic stages
    if (CRITIC) {
        // Block-wide reduction of the 147 gradient entries + the loss over the lanes that own the same agent (lane = env * G +
        // agent): every thread sums a few (entry, agent) items over the block's envs in ascending order and writes them to the
        // agent's partial row of this block.  (One shared-memory pass instead of log2(32 / G) shuffle rounds over 148 registers
        // in two warps: 1200 SHFL + FADD per block and ~2 us at the end of every rollout.)
        __syncthreads();
        constexpr int P1 = kCriticP + 1;
        for (int item = threadIdx.x; item < P1 * N; item += kBlock) {
            const int entry = item / N, a = item - entry * N;
            float sum = red_s[entry][a];
#pragma unroll
            for (int j = 1; j < EPW; ++j) sum += red_s[entry][a + G * j];
            partials[((int64_t)(net0 + a) * gridDim.x + blockIdx.x) * P1 + entry] = sum;
        }
    }
}

template <int N, int M>
int launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, const EnvPartners* p, cudaStream_t s) {
    constexpr int G = N <= 2 ? 2 : (N <= 4 ? 4 : 8);
    const int64_t blocks = (d->E + (32 / G) - 1) / (32 / G);   // one block = 4 stage warps over 32/G envs
    if (p) {
        if (runs)
            return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, true, true, true>,
                              dim3((unsigned)blocks, (unsigned)runs->runs), dim3(kBlock), 0, s, *d, d->partials, *runs, *p);
        if (d->flags & IA2C_FLAG_FUSED_CRITIC)
            return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, true, false, true>, dim3((unsigned)blocks), dim3(kBlock),
                              0, s, *d, d->partials, NoRuns{}, *p);
        return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, false, false, true>, dim3((unsigned)blocks), dim3(kBlock), 0,
                          s, *d, nullptr, NoRuns{}, *p);
    }
    if (runs)   // every run with its own row of blocks, partitioned as a standalone run of E envs
        return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, true, true>, dim3((unsigned)blocks, (unsigned)runs->runs),
                          dim3(kBlock), 0, s, *d, d->partials, *runs, NoPartners{});
    if (d->flags & IA2C_FLAG_FUSED_CRITIC)
        return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, true, false>, dim3((unsigned)blocks), dim3(kBlock), 0, s, *d,
                          d->partials, NoRuns{}, NoPartners{});
    return launch_pdl("rollout_fused_kernel", rollout_fused_kernel<N, M, false, false>, dim3((unsigned)blocks), dim3(kBlock), 0, s, *d,
                      nullptr, NoRuns{}, NoPartners{});
}

}  // namespace

// Returns 1 if (N, M) has a fused instantiation.
int rollout_fused_supported(int N, int M) { return (M == 5 && N >= 2 && N <= 8) || (M == 3 && N == 2); }

// Number of partial rows per agent the fused critic stage writes (= rollout grid size).
int64_t rollout_fused_blocks(int64_t E, int N) {
    const int G = N <= 2 ? 2 : (N <= 4 ? 4 : 8);
    return (E + (32 / G) - 1) / (32 / G);
}

// runs != nullptr: all runs of a batch (ia2c_train_episode_runs), always with the critic-gradient stage.
// p != nullptr: the PARTNERS instantiation (frozen partners per env).
int rollout_fused_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, const EnvPartners* p, cudaStream_t s) {
    if (d->M == 3 && d->N == 2) return launch<2, 3>(d, runs, p, s);
    switch (d->N) {
        case 2: return launch<2, 5>(d, runs, p, s);
        case 3: return launch<3, 5>(d, runs, p, s);
        case 4: return launch<4, 5>(d, runs, p, s);
        case 5: return launch<5, 5>(d, runs, p, s);
        case 6: return launch<6, 5>(d, runs, p, s);
        case 7: return launch<7, 5>(d, runs, p, s);
        case 8: return launch<8, 5>(d, runs, p, s);
    }
    set_error("rollout_fused: no instantiation for N=%d M=%d", d->N, d->M);
    return IA2C_ERR_UNSUPPORTED;
}

}  // namespace ia2c
