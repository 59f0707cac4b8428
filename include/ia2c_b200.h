/* ia2c_b200.h — C ABI of libia2c_b200.so: the B200 (sm_100a) implementation of IA2C's
 * rollout-and-update hot path.
 *
 * Conventions (SURVEY.md §8 b2)
 *   - every pointer is a DEVICE pointer unless its name starts with host_;
 *   - the library never allocates or frees caller-visible memory: all buffers, including
 *     workspaces, are passed in (the Python host passes torch CUDA tensors' data_ptr());
 *   - kernels are enqueued on `stream` (a cudaStream_t passed as void*); no entry point
 *     synchronises the host, except the *_host entry points which say so;
 *   - return 0 on success, a negative ia2c_status otherwise; ia2c_last_error() describes the
 *     last failure on the calling thread.  No C++ exception crosses this boundary.
 *   - network parameters are one flat fp32 vector per net in nn.Linear state_dict order:
 *       l1.weight[H,F] l1.bias[H] l2.weight[H,H] l2.bias[H] l3.weight[O,H] l3.bias[O]
 *     with H = IA2C_HIDDEN = 6 (reference: ac_nets.py:24,26-33).
 *
 * Each entry point names the reference interface it replaces (file:line in thinclab/IA2C).
 */
#ifndef IA2C_B200_H
#define IA2C_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IA2C_ABI_VERSION 6
#define IA2C_HIDDEN 6          /* ac_nets.py:24 */
#define IA2C_OBS_FEATURES 6    /* Org observation: [onehot3(prev class), onehot3(class)]  Org.py:37,112-114 */
#define IA2C_AGENT_ACTIONS 3   /* ia2c.py:44 */
#define IA2C_JOINT_ACTIONS 9   /* ia2c.py:45 */
#define IA2C_BELIEF_RECORD 8   /* bytes per packed (agent, modelled other) belief record */
#define IA2C_MAX_MODELS 6      /* packed record holds up to 6 model beliefs (reference: 5, ia2c.py:46) */

typedef enum {
    IA2C_OK = 0,
    IA2C_ERR_INVALID = -1,     /* bad dimension / null pointer / unsupported shape */
    IA2C_ERR_CUDA = -2,        /* CUDA runtime error at launch */
    IA2C_ERR_UNSUPPORTED = -3
} ia2c_status;

const char* ia2c_last_error(void);
int ia2c_abi_version(void);
/* Number of kernels launched by this library since load (the bench's gpu_launches count). */
uint64_t ia2c_launch_count(void);

/* ------------------------------------------------------------------ (1) Org environment ---- */
/* Env state is structure-of-arrays over E independent envs:
 *   state  int32[E]   financial-health state 0..4           (Org.state,   Org.py:23)
 *   hist   double[E]  reward history r (fp64 recurrence)    (Org.reward,  Org.py:25,55)
 *   cls    uint8[E,2] observation classes {previous, current} (Org.observation, Org.py:37,112-114)
 *   elapsed int32[E]  steps since reset (gymnasium TimeLimit, ia2c.py:37)
 */

/* Org.reset (Org.py:128-148) for all E envs; obs_out float[E,6] may be NULL. */
int ia2c_org_reset(int32_t* state, double* hist, uint8_t* cls, int32_t* elapsed, float* obs_out,
                   int64_t E, void* stream);

/* Org.step (Org.py:51-126) with the reference's joint action code per env (0..8; any other code
 * leaves state and reward untouched but shifts the observation memory).  max_episode_steps > 0
 * adds TimeLimit truncation with same-step autoreset (gym.make_vec, ia2c.py:34-42): obs_out is then
 * the reset observation, reward_out the real pre-reset reward.
 *   joint int32[E]; obs_out float[E,6]; reward_out double[E]; reward_f32_out float[E] (may be NULL);
 *   state_trace int32[E] (state right after the step, before any autoreset; may be NULL);
 *   truncated_out uint8[E] (may be NULL). */
int ia2c_org_step_joint(int32_t* state, double* hist, uint8_t* cls, int32_t* elapsed,
                        const int32_t* joint, float* obs_out, double* reward_out, float* reward_f32_out,
                        int32_t* state_trace, uint8_t* truncated_out,
                        int64_t E, int32_t max_episode_steps, void* stream);

/* Org-N step (builder-defined generalisation, DESIGN.md): actions uint8[E,N] in {0,1,2}; N=2 is
 * exactly ia2c_org_step_joint with joint = a0*3+a1 (ia2c.py:84). */
int ia2c_org_step_agents(int32_t* state, double* hist, uint8_t* cls, int32_t* elapsed,
                         const uint8_t* actions, float* obs_out, double* reward_out, float* reward_f32_out,
                         int32_t* state_trace, uint8_t* truncated_out,
                         int64_t E, int32_t N, int32_t max_episode_steps, void* stream);

/* ------------------------------------------------------------------ (2) belief filter ------- */
/* BeliefFilter.update (belief_filter_deprecated.py:45-59), dense reference layout, fp64:
 *   filter_action double[M,A]; lik double[R,A] (any likelihood rows); prev double[R,M]; u double[R]
 *   -> ap int64[R], bprime double[R,M] (rounded to 2 decimals), prediction double[R,A] (may be NULL).
 * M, A <= 8. */
int ia2c_belief_update_dense(const double* filter_action, const double* lik, const double* prev,
                             const double* u, int64_t* ap, double* bprime, double* prediction,
                             int64_t R, int32_t M, int32_t A, void* stream);

/* Pairwise packed form used by the trainer: one 8-byte record per (env, agent i, modelled other jj):
 * bytes 0..M-1 = posterior in hundredths (lossless: posteriors are rounded to 2 decimals,
 * belief_filter_deprecated.py:58), byte 6 = predicted action.  The likelihood 0.8/0.1 of
 * ia2c.py:53-58 is synthesised from the other agent's action (never materialised).
 *   records uint8[E,N,K,8] in/out (K = N-1 modelled others, ascending agent order, skipping i);
 *   filter_action double[N,M,3]; actions uint8[E,N];
 *   u_injected double[E,N,K] or NULL -> Philox(seed, episode, t, global pair index);
 *   pred_out uint8[E,N,K] (may be NULL); belief_out uint8[E,N,K,M] (may be NULL; debugging/parity);
 *   pred_partner_out uint8[E,N] = mode over modelled others of the predicted action, ties -> lowest;
 *   reset_prior != 0: ignore stored records and start from the uniform prior round(1/M,2)
 *   (ia2c.py:79; belief_filter_deprecated.py:29). env_offset = global index of env 0 (multi-GPU). */
int ia2c_belief_update_pairs(uint8_t* records, const double* filter_action, const uint8_t* actions,
                             const double* u_injected, uint8_t* pred_out, uint8_t* belief_out,
                             uint8_t* pred_partner_out, int64_t E, int32_t N, int32_t M, int32_t reset_prior,
                             uint64_t seed, uint32_t episode, uint32_t t, int64_t env_offset, void* stream);

/* The same update carried through a WHOLE episode in one launch (the trainer's rollout for many modelled others): the record
 * lives in registers from the uniform prior of step 0 (ia2c.py:79) to step T1-1 and is written once; the per-step inputs
 * and outputs are the trajectory arrays.  Bit-identical to T1 calls of ia2c_belief_update_pairs (reset_prior at the first).
 *   act uint8[T1,E,N]; u_injected double[T1,E,N,K] or NULL -> Philox(seed, episode, t, ...);
 *   pred_dump uint8[T1,E,N,K], belief_dump uint8[T1,E,N,K,M] (may be NULL); partner_pred uint8[T1,E,N] out;
 *   records uint8[E,N,K,8] out.  Requires ia2c_belief_supports_episode(N, M): 9 <= N <= 512. */
int ia2c_belief_supports_episode(int32_t N, int32_t M);
int ia2c_belief_update_pairs_episode(uint8_t* records, const double* filter_action, const uint8_t* act, const double* u_injected,
                                     uint8_t* pred_dump, uint8_t* belief_dump, uint8_t* partner_pred, int64_t E, int32_t N,
                                     int32_t M, int32_t T1, uint64_t seed, uint32_t episode, int64_t env_offset, void* stream);

/* Diagnostic: q_seq[i] = the library's branch-free fp64 division sequence (csrc/common.cuh: ddiv_seq),
 * q_ieee[i] = IEEE a/b (__ddiv_rn).  Used by the tests to prove the two agree bit for bit on the
 * operand ranges the belief filter and the reward recurrence produce. */
int ia2c_debug_divide(const double* a, const double* b, double* q_seq, double* q_ieee, int64_t n, void* stream);

/* Diagnostic: the FP32 fma-pipe issue peak of this GPU — independent register-resident fma chains at full occupancy,
 * packed != 0 with fma.rn.f32x2 (FFMA2, what csrc/mlp_f2.cuh is written in), 0 with scalar fma.rn.f32.  The measured
 * denominator for the MLP-bound kernels (hidden_size = 6 rules tensor cores out).  out float[1] (never written in
 * practice); host_flops_out receives the FLOPs of one launch; time it with CUDA events on `stream`. */
int ia2c_debug_fp32_peak(float* out, int32_t iters, int32_t packed, int32_t blocks_per_sm, double* host_flops_out, void* stream);

/* ------------------------------------------------------------------ (3) actor / critic MLPs -- */
/* NeuralNet.forward (ac_nets.py:34-41) for `nets` independent networks over the same rows:
 *   params float[nets,P]; x float[rows,F] (shared by all nets) -> y float[nets,rows,O];
 *   softmax != 0 applies the actor's softmax.  F arbitrary, O <= 32.
 *   h1_out float[rows,6] (may be NULL; nets == 1 only): the post-ReLU layer-1 activations, kept so that the
 *   backward pass does not have to read x again to recompute them. */
int ia2c_mlp_forward(const float* params, const float* x, float* y, float* h1_out, int64_t rows, int32_t F, int32_t O,
                     int32_t nets, int32_t softmax, void* stream);

/* Backward of the above for ONE net: given dy float[rows,O] = dL/d(output) (for softmax nets dL/dprobs),
 * accumulates dL/dparams into grad float[P] (grad += if accumulate != 0, else overwritten) and, if dx
 * is not NULL, writes dL/dx float[rows,F].  Replaces autograd through ac_nets.py:34-41.
 *   h1_saved float[rows,6] (may be NULL): ia2c_mlp_forward's h1_out for the same x and params;
 *   workspace float[ia2c_mlp_backward_workspace(rows,F,O)] */
size_t ia2c_mlp_backward_workspace(int64_t rows, int32_t F, int32_t O);
int ia2c_mlp_backward(const float* params, const float* x, const float* dy, const float* h1_saved, float* grad, float* dx,
                      float* workspace, int64_t rows, int32_t F, int32_t O, int32_t softmax,
                      int32_t accumulate, void* stream);

/* Index-input forms (SURVEY.md 8 f2; a2c_test.py:57,67 feeds one_hot(state, F)): idx int64[rows] in [0, F) stands for the row
 * one_hot(idx, F).  Same results, bit for bit, as the dense entry points on the materialised one-hot rows, without reading or
 * building a [rows, F] tensor.  ia2c_mlp_backward_index needs the h1 written by ia2c_mlp_forward_index; workspace as for
 * ia2c_mlp_backward (ia2c_mlp_backward_workspace).  Indices have no gradient. */
int ia2c_mlp_forward_index(const float* params, const int64_t* idx, float* y, float* h1_out, int64_t rows, int32_t F,
                           int32_t O, int32_t softmax, void* stream);
int ia2c_mlp_backward_index(const float* params, const int64_t* idx, const float* dy, const float* h1_saved, float* grad,
                            float* workspace, int64_t rows, int32_t F, int32_t O, int32_t softmax, int32_t accumulate,
                            void* stream);
int ia2c_actor_sample_index(const float* params, const int64_t* idx, const float* u, int64_t* actions_out, float* probs_out,
                            int64_t rows, int32_t F, int32_t O, uint64_t seed, uint64_t counter, void* stream);

/* ActorNetwork.sample_action (ac_nets.py:94-102): forward + Categorical(probs).sample().
 *   u float[rows] uniforms in [0,1) (injected) or NULL -> Philox(seed, counter); the sampler is
 *   inverse-CDF over q = p/sum(p) (statistically, not stream-, equivalent to torch.multinomial).
 *   actions_out int64[rows]; probs_out float[rows,O] may be NULL. */
int ia2c_actor_sample(const float* params, const float* x, const float* u, int64_t* actions_out,
                      float* probs_out, int64_t rows, int32_t F, int32_t O, uint64_t seed, uint64_t counter,
                      void* stream);

/* ------------------------------------------------------------------ (4) losses ---------------- */
/* CriticNetwork.batch_update loss (ac_nets.py:64-70): loss = mean((target - Q[act])^2) over B rows.
 *   Q float[B,O], act int32[B], target float[B] -> loss_out float[1], dQ float[B,O], dtarget float[B]
 *   (dtarget may be NULL; it is what autograd sends into a target that carries a graph, ia2c.py:108-113). */
int ia2c_critic_loss(const float* Q, const int32_t* act, const float* target, float* loss_out, float* dQ,
                     float* dtarget, float* workspace, int64_t B, int32_t O, void* stream);

/* ActorNetwork.batch_update loss (ac_nets.py:113-117) with torch.distributions.Categorical(probs=p)
 * semantics: q = p/sum(p), logit = log(clamp(q, eps, 1-eps)), loss = mean(adv*(-logit[a]) - beta*H).
 *   probs float[B,O], act int32[B], adv float[B] -> loss_out float[1], dprobs float[B,O],
 *   dadv float[B] (may be NULL; gradient into a differentiable advantage, a2c_org_test.py:86-91).
 *   status_out int32[1]: set to 1 if any row is not a valid simplex (the reference raises ValueError). */
int ia2c_actor_loss(const float* probs, const int32_t* act, const float* adv, float beta, float* loss_out,
                    float* dprobs, float* dadv, int32_t* status_out, float* workspace, int64_t B, int32_t O,
                    void* stream);
size_t ia2c_loss_workspace(int64_t B);

/* Adam step (torch.optim.Adam defaults, single-tensor path; ac_nets.py:50,72,89,119) over `nets` flat
 * parameter vectors of length P.  step_count int32[nets] lives on the device and is incremented by the
 * kernel (CUDA-graph friendly); bias corrections are computed in fp64 on the device.
 *   grad_accum: if not NULL, grad_accum += grad first and Adam uses grad_accum — the reference's actor
 *   never zeroes its gradients (ac_nets.py:112-119 has no zero_grad). */
int ia2c_adam_step(float* params, const float* grad, float* grad_accum, float* exp_avg, float* exp_avg_sq,
                   int32_t* step_count, double lr, double beta1, double beta2, double eps,
                   int32_t nets, int32_t P, void* stream);

/* CriticNetwork.batch_update (kind 0; ac_nets.py:62-72) / ActorNetwork.batch_update (kind 1; ac_nets.py:112-119) in ONE
 * call for a target / advantage that carries no autograd graph: forward, loss (ia2c_critic_loss / ia2c_actor_loss
 * semantics), backward, Adam step (torch defaults: betas 0.9 / 0.999, eps 1e-8).
 *   params / exp_avg / exp_avg_sq float[P], step_count int32[1] (device, incremented): as ia2c_adam_step;
 *   grad float[P]: kind 0 -> overwritten with this update's gradient (the critic calls zero_grad first);
 *                  kind 1 -> grad += gradient, and Adam steps on the running sum (the actor never zeroes it, Q2);
 *   exactly one of x float[rows,F] (dense rows) and idx int64[rows] (class indices standing for one_hot rows);
 *   act int32[rows]; signal float[rows] = target (kind 0) or advantage (kind 1); beta = entropy weight (kind 1);
 *   loss_out float[1] (device); status_out int32[1] (zeroed by the caller; required for kind 1, optional for kind 0): bit 0 is set
 *   if a probability row is not a simplex (kind 1), bit 1 if an idx value lies outside [0, F) (such rows are clamped, never read
 *   out of bounds — the caller decides what to do with the update);
 *   workspace float[ia2c_net_update_workspace(rows,F,O)].
 * Wide dense inputs (the a2c_test.py shape) take a single-pass kernel that reads x ONCE (bulk async copies into shared
 * memory, both the layer-1 products and the layer-1 weight gradient computed from the staged tile). */
size_t ia2c_net_update_workspace(int64_t rows, int32_t F, int32_t O);
int ia2c_net_update(int32_t kind, float* params, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_count,
                    const float* x, const int64_t* idx, const int32_t* act, const float* signal, float beta, double lr,
                    float* loss_out, int32_t* status_out, float* workspace, int64_t rows, int32_t F, int32_t O, void* stream);

/* ------------------------------------------------------------------ fused IA2C trainer -------- */
/* One descriptor for the whole episode of ia2c.py:62-129, generalised to N agents (DESIGN.md "Org-N").
 * Trajectory layout in HBM (time-major, env-minor, structure of arrays):
 *   obs      float[T+1,E,6]   obs[t]; next_obs[t] is obs[t+1] (obs[T] is the post-autoreset observation)
 *   reward   float[T,E]       float32(r) as stored by ia2c.py:99
 *   act      uint8[T+1,E,N]   sampled own actions (act[t+1] = "next action")
 *   partner_true uint8[T+1,E,N]  mode of the other agents' true actions
 *   partner_pred uint8[T+1,E,N]  mode of the belief-predicted actions of the modelled others
 */
typedef struct ia2c_episode_desc {
    int64_t E;                 /* envs on this rank */
    int64_t E_total;           /* envs over all ranks (mean denominators) */
    int64_t env_offset;        /* global index of local env 0 (RNG counters) */
    int32_t N, T, M;           /* agents, steps per episode, models */
    int32_t max_episode_steps; /* TimeLimit (ia2c.py:37) */
    float gamma, beta;
    double lr_actor, lr_critic;
    uint64_t seed;
    uint32_t episode;
    int32_t flags;             /* IA2C_FLAG_* */
    /* networks: params/adam state float[N,105] (actor) and float[N,147] (critic).
     * Gradient buffers carry the phase's loss in one extra trailing slot per net, so that one
     * all-reduce moves both: actor_grad float[N,106], critic_grad float[N,148]. */
    float *actor_params, *actor_grad, *actor_grad_accum, *actor_m, *actor_v;
    float *critic_params, *critic_grad, *critic_m, *critic_v;
    int32_t *actor_step, *critic_step;     /* int32[N] Adam step counters (device) */
    float *loss_out;                       /* float[2,N]: critic losses then actor losses */
    const double* filter_action;           /* double[N,M,3] */
    /* env state */
    int32_t* env_state; double* env_hist; uint8_t* env_cls; int32_t* env_elapsed;
    double* ep_return;                     /* double[E] sum of fp64 rewards (ia2c.py:102) */
    /* trajectory */
    float *obs, *reward; uint8_t *act, *partner_true, *partner_pred;
    uint8_t* belief_records;               /* uint8[E,N,K,8] */
    /* replay / injected randomness (any may be NULL) */
    const uint8_t* inj_actions;            /* uint8[T+1,E,N]: replayed action samples */
    const float* inj_u_action;             /* float[T+1,E,N]: uniforms for the inverse-CDF sampler */
    const double* inj_u_belief;            /* double[T+1,E,N,K] */
    /* optional parity dumps (may be NULL) */
    int32_t* state_trace;                  /* int32[T,E] */
    double* reward_f64;                    /* double[T,E] */
    uint8_t* pred_dump;                    /* uint8[T+1,E,N,K] */
    uint8_t* belief_dump;                  /* uint8[T+1,E,N,K,M] */
    float* adv_dump;                       /* float[N,T,E] */
    float* target_dump;                    /* float[N,T,E] */
    /* workspace */
    float* partials; size_t partials_floats;  /* per-block gradient partials */
} ia2c_episode_desc;

#define IA2C_FLAG_FUSED_ROLLOUT 1   /* use the persistent one-launch rollout kernel (N <= 8) */
#define IA2C_FLAG_FUSED_CRITIC  4   /* with FUSED_ROLLOUT: the rollout kernel also accumulates the critic gradient
                                       (ia2c_critic_phase then only reduces the partials and applies Adam) */
#define IA2C_FLAG_GRAD_ONLY     8   /* critic/actor phase stop after the gradient kernel (per-block partials only);
                                       ia2c_allreduce_adam then reduces, exchanges and steps */
#define IA2C_FLAG_ACTOR_COLUMNS 16  /* actor phase: use the time-chunk column kernel instead of the pipelined one (A/B, parity tests) */
#define IA2C_FLAG_SKIP_ADAM     2   /* stop after writing gradients (multi-GPU: all-reduce, then ia2c_adam_step) */
#define IA2C_FLAG_ROLLOUT_PER_STEP 64 /* rollout (N > 8): one env_step + one actor_step kernel per step instead of the persistent
                                      * rollout_many_kernel (9 <= N <= 256 with the whole-episode belief kernel) — A/B and parity tests */
#define IA2C_FLAG_BELIEF_PER_STEP 32 /* rollout (N > 8): one belief kernel per step (ia2c_belief_update_pairs) instead of the
                                      * whole-episode kernel (ia2c_belief_update_pairs_episode) — A/B and parity tests */

size_t ia2c_episode_partials_floats(const ia2c_episode_desc* d);

/* 1 if IA2C_FLAG_FUSED_ROLLOUT has an instantiation for N agents and M models (N <= 8 with M = 5; N = 2 with M = 3). */
int ia2c_rollout_fused_supported(int32_t N, int32_t M);

/* Rollout only: ia2c.py:72-102 for all E envs (T+1 actor/belief evaluations, T env steps). */
int ia2c_rollout(const ia2c_episode_desc* d, void* stream);
/* Critic phase (ia2c.py:104-114): fused forward(obs) + forward(next_obs) + MSE + backward through
 * both passes -> critic_grad float[N,148], loss_out[0,:]; then Adam unless IA2C_FLAG_SKIP_ADAM. */
int ia2c_critic_phase(const ia2c_episode_desc* d, void* stream);
/* Actor phase (ia2c.py:116-129): advantage from the UPDATED critic, policy-gradient + entropy loss,
 * backward -> actor_grad float[N,106], loss_out[1,:]; then accumulate + Adam unless SKIP_ADAM. */
int ia2c_actor_phase(const ia2c_episode_desc* d, void* stream);
/* Adam from the gradient buffers (after a multi-GPU all-reduce): which = 0 critics, 1 actors. */
int ia2c_apply_adam(const ia2c_episode_desc* d, int32_t which, void* stream);
#define IA2C_MAX_RANKS 8   /* one node: NVLink peers of an 8-GPU box */
/* Multi-GPU: fused gradient all-reduce + Adam over NVLink peer memory, ONE kernel per optimiser phase instead of
 * reduce -> NCCL all-reduce -> Adam.  Run it after the phase's gradient kernel (ia2c_rollout with
 * IA2C_FLAG_FUSED_CRITIC, or ia2c_critic_phase / ia2c_actor_phase with IA2C_FLAG_GRAD_ONLY).
 * inbox[p] is rank p's symmetric buffer mapped into this process (ia2c_peer_inbox_bytes bytes, 8-byte aligned,
 * zero-initialised): every gradient entry travels as ONE naturally aligned 64-bit word {epoch << 32 | float bits}
 * written with a single st.relaxed.sys.u64, so a message carries its own flag and cannot tear.  mc_inbox, if not
 * NULL, is the NVSwitch multicast mapping of the same buffers: one multimem.st then reaches every rank's inbox
 * instead of `world` unicast stores.  epoch starts at 1 and increases by one per call on every rank (same value
 * on all ranks); a rank can be at most one exchange ahead of a peer, so the inbox is double-buffered by epoch
 * parity.  adam_step is the Adam step number of this update.  Every rank must launch it.
 * Failure: if a peer's words do not arrive within timeout_us (0 -> 2 s) the kernel applies NOTHING for the
 * affected entries, stops, and raises error[p] on EVERY rank (error[] are the ranks' symmetric int32 error
 * words); once a rank's error word is set every later ia2c_allreduce_adam on it is a no-op.  The host must
 * poll its own error word (trainer.py: check_comm) before trusting or checkpointing parameters. */
typedef struct ia2c_peer_desc {
    int32_t rank, world;       /* world <= 8 (one NVSwitch domain) */
    uint64_t* inbox[IA2C_MAX_RANKS];
    uint64_t* mc_inbox;        /* multicast (NVLS) mapping of the inboxes, or NULL */
    int32_t* error[IA2C_MAX_RANKS];         /* every rank's error word; error[rank] is this rank's own */
    uint32_t timeout_us;       /* poll budget per entry in microseconds (0 -> 2 000 000) */
    uint32_t reserved;
} ia2c_peer_desc;
size_t ia2c_peer_inbox_bytes(const ia2c_episode_desc* d, int32_t world);
int ia2c_allreduce_adam(const ia2c_episode_desc* d, int32_t which, const ia2c_peer_desc* peers, uint32_t epoch,
                        int32_t adam_step, void* stream);
/* One whole episode of a multi-GPU run in one call per rank: ia2c_rollout, critic gradient, ia2c_allreduce_adam
 * (epoch0 + 1), actor gradient, ia2c_allreduce_adam (epoch0 + 2); Adam step number = desc.episode + 1.
 * desc.flags must carry SKIP_ADAM | GRAD_ONLY.  The caller advances its epoch counter by 2. */
int ia2c_train_episode_p2p(const ia2c_episode_desc* d, const ia2c_peer_desc* peers, uint32_t epoch0, void* stream);


/* rollout + critic phase + actor phase on one stream. */
int ia2c_train_episode(const ia2c_episode_desc* d, void* stream);
/* Same, with HOST buffers: copies the injected uniforms host->device, runs the episode, copies
 * loss_out and ep_return device->host and synchronises the stream.  host_u_action float[T+1,E,N],
 * host_u_belief double[T+1,E,N,K] (pinned memory recommended); the desc's inj_u_* must point at
 * device staging buffers of the same size. */
int ia2c_train_episode_host(const ia2c_episode_desc* d, const float* host_u_action,
                            const double* host_u_belief, float* host_loss_out, double* host_ep_return,
                            void* stream);

/* Profiling form of ia2c_train_episode: CUDA events between the kernel launch groups on `stream`, one sync at
 * the end.  host_ms_out float[5] = {rollout, critic gradient, critic reduce+Adam, actor gradient, actor
 * reduce+Adam} in milliseconds. */
int ia2c_train_episode_timed(const ia2c_episode_desc* d, float* host_ms_out, void* stream);

/* Pipelined form of the above for n_episodes consecutive episodes, ONE copy per direction per episode:
 *   host_tapes[k]  (pinned) = [u_action float[T+1,E,N] | pad to 8 B | u_belief double[T+1,E,N,K]], ia2c_host_tape_bytes;
 *   host_results   (pinned) = n_episodes x [loss float[2,N] | pad to 8 B | ep_return double[E]], ia2c_host_result_bytes.
 * On the device the two tapes share one staging region (desc.inj_u_belief must follow desc.inj_u_action at the padded
 * offset; stage_b is a second region of the same size) and desc.ep_return follows desc.loss_out the same way.  The H2D
 * copy of episode k+1 overlaps the compute of episode k on an internal copy stream; with result_b (a second device result
 * region of ia2c_host_result_bytes, may be NULL) the D2H of episode k also runs on its own stream under episode k+1, and the
 * last episode's results are left in desc.loss_out / desc.ep_return; one host sync at the end.
 * Episode numbers are desc.episode .. desc.episode + n_episodes - 1. */
size_t ia2c_host_tape_bytes(const ia2c_episode_desc* d);
size_t ia2c_host_result_bytes(const ia2c_episode_desc* d);
/* The pipeline's two internal streams (H2D copy, D2H download) and its events live in a caller-owned handle, created on
 * the current device; the library keeps no hidden per-thread state.  Destroy drains and frees them. */
typedef struct ia2c_host_pipe ia2c_host_pipe;
int ia2c_host_pipe_create(ia2c_host_pipe** out);
int ia2c_host_pipe_destroy(ia2c_host_pipe* pipe);
/* Depth of the device staging ring (default 2, up to 8): desc.inj_u_action is region 0, stage_b holds `stages - 1` consecutive
 * regions of ia2c_host_stage_stride(desc) bytes.  A deeper ring lets the H2D copies run further ahead of the kernels (on a
 * multi-GPU box the kernels wait for the slowest rank twice per episode; with two regions the copy engine waits with them). */
int ia2c_host_pipe_set_stages(ia2c_host_pipe* pipe, int32_t stages);
size_t ia2c_host_stage_stride(const ia2c_episode_desc* d);
/* On any error the call still drains everything it enqueued before returning (no copy is left in flight). */
int ia2c_train_episodes_host(const ia2c_episode_desc* d, ia2c_host_pipe* pipe, void* stage_b, void* result_b,
                             int32_t n_episodes, const void* const* host_tapes, void* host_results, void* stream);
/* The same pipeline on every rank of a multi-GPU run (one process per GPU): after each gradient phase the fused NVLink
 * all-reduce + Adam (ia2c_allreduce_adam) with epochs epoch0+1 .. epoch0+2*n_episodes; desc.flags = SKIP_ADAM | GRAD_ONLY.
 * Every rank must call it with the same n_episodes. */
int ia2c_train_episodes_host_p2p(const ia2c_episode_desc* d, ia2c_host_pipe* pipe, const ia2c_peer_desc* peers,
                                 uint32_t epoch0, void* stage_b, void* result_b, int32_t n_episodes,
                                 const void* const* host_tapes, void* host_results, void* stream);

/* ------------------------------------------------------------------ batches of independent runs -- */
/* R independent IA2C training runs (seeds, hyper-parameter sweeps) advanced together, one episode number for all, in the
 * launches of ONE episode.  All runs share N, M, T, max_episode_steps and E = envs per run; run r has its own Philox key
 * seed[r], its own parameters, belief models and Adam state, and its own lr_actor / lr_critic / gamma / beta.
 *
 * Contract: run r computes byte for byte what ia2c_train_episode computes for a standalone run of E envs with
 * desc.seed = seed[r], flags FUSED_ROLLOUT | FUSED_CRITIC | ACTOR_COLUMNS and the run's hyper-parameters — trajectory,
 * beliefs, returns, losses, gradients, Adam moments, step counters, actor grad_accum and parameters.  Philox counters use
 * the env's index WITHIN its run, the means divide by T * E, and every run's gradient partial rows are partitioned as a
 * standalone run of E envs partitions them, so every fixed-order sum is the same sum.
 *
 * `d` describes ONE run's shape (E = E_total = envs per run, env_offset = 0; desc.seed is not used); its pointers hold all
 * R runs stacked:
 *   per-net buffers  (params, grads, Adam m / v, step counters, actor_grad_accum, filter_action): R*N rows, run r at rows
 *                    [r*N, (r+1)*N);
 *   per-env buffers  (env state, ep_return, belief_records, and the trajectory obs[T+1, R*E, 6], reward[T, R*E],
 *                    act / partner_true / partner_pred [T+1, R*E, N]): the env axis has length R*E, run r at [r*E, (r+1)*E);
 *   loss_out         float[2, R*N] (critic losses of all nets, then actor losses);
 *   partials         ia2c_runs_partials_floats(d, R) floats.
 * Supported: the fused path only (ia2c_rollout_fused_supported(N, M): N <= 8), one GPU, Philox sampling; batches of
 * 9 <= N <= 256 agents have their own entry point, ia2c_train_episode_runs_many (below).  desc.flags may
 * carry only FUSED_ROLLOUT, FUSED_CRITIC and ACTOR_COLUMNS (the path is always that one).  Refused with
 * IA2C_ERR_UNSUPPORTED: other (N, M), a non-zero env_offset or E_total != E (multi-GPU), injected replay tapes, parity
 * dumps, other flags.  Refused with IA2C_ERR_INVALID: runs < 1, runs * N > IA2C_MAX_RUN_NETS (the actor-gradient grid
 * has one block row per net), a NULL seed array, missing buffers.  Every check runs before the first CUDA call.
 * The host-tape pipelines have no batched form. */
#define IA2C_MAX_RUN_NETS 65535
typedef struct ia2c_runs_desc {
    int32_t runs;              /* R >= 1, R * N <= IA2C_MAX_RUN_NETS */
    int32_t reserved;
    const uint64_t* seed;      /* device uint64[R]: Philox key of run r (desc.seed is not used) */
    const double* lr_actor;    /* device double[R], or NULL -> desc.lr_actor for every run */
    const double* lr_critic;   /* device double[R], or NULL -> desc.lr_critic */
    const float* gamma;        /* device float[R],  or NULL -> desc.gamma */
    const float* beta;         /* device float[R],  or NULL -> desc.beta */
} ia2c_runs_desc;
size_t ia2c_runs_partials_floats(const ia2c_episode_desc* d, int32_t runs);
/* One episode of every run: fused rollout + critic gradient, critic reduce + Adam, actor gradient, actor reduce + Adam —
 * the four launches of a standalone episode, each covering all R runs. */
int ia2c_train_episode_runs(const ia2c_episode_desc* d, const ia2c_runs_desc* r, void* stream);

/* A batch of R independent Org-N runs with 9 <= N <= 256 agents, in SIX launches per episode whatever R is.  Same descriptors
 * and the same stacked layout as ia2c_train_episode_runs (above): per-net rows R*N, env axis R*E, loss_out float[2, R*N],
 * partials ia2c_runs_partials_floats(d, R) floats; desc.flags = IA2C_FLAG_ACTOR_COLUMNS.
 *
 * Contract: run r computes byte for byte what ia2c_train_episode computes for a standalone run of E envs with desc.seed =
 * seed[r], flags = ACTOR_COLUMNS (the whole-episode rollout and belief kernels, then the column actor kernel) and the run's
 * lr_actor / lr_critic / gamma / beta — trajectory, belief records, partner_pred, returns, losses, gradients, Adam moments, step
 * counters, actor grad_accum and parameters.  (Above N = 64 a standalone trainer defaults to the pipelined actor kernel, whose
 * sums are ordered differently: the contract is with the column kernel.)  Philox counters use the env's index within its run.
 *
 * Launches (grid x, y; each run partitioned exactly as a standalone run of E envs, so every fixed-order sum is the same sum):
 *   1. rollout_many_kernel          (ceil(E / c), R): c envs per block, chosen once for the batch (waves over R * ceil(E / c)
 *                                   blocks x c); one block's envs lie in one run;
 *   2. belief_pairs_episode_kernel  (env blocks of one run, R*N): blockIdx.y = run*N + agent is the filter row;
 *   3. critic_grad_kernel           (grad_blocks(E), R*N);
 *   4. reduce_adam_kernel (critics) (R*N, ceil(148 / 32));
 *   5. actor_grad_kernel            (grad_blocks(E), R*N), the column kernel;
 *   6. reduce_adam_kernel (actors)  (R*N, ceil(106 / 32)).
 * Refused with IA2C_ERR_UNSUPPORTED: N <= 8 (use ia2c_train_episode_runs), N > 256, a non-zero env_offset or E_total != E,
 * injected replay tapes, parity dumps, flags other than exactly IA2C_FLAG_ACTOR_COLUMNS.  Refused with IA2C_ERR_INVALID:
 * runs < 1, runs * N > IA2C_MAX_RUN_NETS, a NULL seed array, M outside 2..6, missing buffers, a workspace smaller than
 * ia2c_runs_partials_floats(d, R).  Every check runs before the first CUDA call. */
int ia2c_train_episode_runs_many(const ia2c_episode_desc* d, const ia2c_runs_desc* r, void* stream);

/* ------------------------------------------------------------------ native A2C trainer (a2c_org_test.py) -- */
/* One update of a2c_org_test.py:43-92 for R independent runs x E envs: a single joint agent with 9 actions, actor and
 * critic both 6 -> 6 -> 6 -> 9 MLPs (147 parameters each, the actor ending in a softmax), Org envs that are never reset
 * after ia2c_org_reset and have no TimeLimit (SURVEY.md Q6).  Per env and update: T steps of Org.step(pending action)
 * followed by a sample of the next action from the post-step observation; the stored pair is (post-step obs, action
 * taken) (Q4).  Critic: target = reward (masks = 0, Q5), L = mean((r - Q(S)[a])^2), Adam.  Actor: Q from the UPDATED
 * critic, V = sum(Q * pi), adv = Q[a] - V with gradient through pi (Q7), policy gradient + beta * entropy, Adam on the
 * never-zeroed running sum of the gradients (Q2).  One row per env (the reference's two buffer rows are copies of one
 * env); the means divide by T * E.  gamma is absent on purpose: with masks = 0 it multiplies zero.
 *
 * Sampling: inj_actions == NULL -> Philox stream 3, key = seed[r], counter = (env index within its run,
 * slot | 3 << 16, update), the 24-bit uniform of the inverse-CDF sampler; slot 0 is update 0's first draw from the reset
 * observation, slot t + 1 the draw after step t.  inj_actions uint8[T+1, R*E] replays actions (codes 0..8) in the same
 * slot order; slot 0 is read at update 0 only.
 *
 * Layout (stacked like ia2c_runs_desc): per-net buffers have R rows (params / Adam m, v / grad_accum float[R,147],
 * grads float[R,148] with this update's loss in the trailing slot, step counters int32[R]); per-env buffers have an
 * env axis of length R*E, run r at [r*E, (r+1)*E): env_state int32, env_hist double, env_cls uint8[.,2], env_elapsed
 * int32 (steps since reset), pending_action uint8, ep_return double (fp64 sum of the update's T rewards); trajectory
 * obs float[T, R*E, 6], act uint8[T, R*E], reward float[T, R*E]; loss_out float[2, R] (critic losses, then actor).
 *
 * Contract: run r computes byte for byte what a call with R = 1, seed[0] = seed[r] and run r's hyper-parameters computes
 * on run r's slices.  One update is FOUR launches: rollout + critic gradient, critic reduce + Adam, actor gradient, actor
 * reduce + Adam.  Every check (ranges, NULL seed or buffers, workspace size) runs before the first CUDA call. */
#define IA2C_A2C_MAX_RUNS 65535           /* R: one grid row per run */
#define IA2C_A2C_MAX_ENVS 1073741824      /* E and R * E */
#define IA2C_A2C_MAX_STEPS 65534          /* T: the slot field of the Philox counter is 16 bits */
typedef struct ia2c_a2c_desc {
    int64_t E;                 /* envs per run */
    int32_t R, T;              /* runs, steps per update */
    uint32_t update;           /* update number (Philox counter; update 0 draws the first action) */
    float beta;                /* entropy weight when beta_run is NULL */
    double lr_actor, lr_critic;            /* learning rates when the per-run arrays are NULL */
    const uint64_t* seed;                  /* uint64[R]: Philox key of run r */
    const double* lr_actor_run;            /* double[R] or NULL */
    const double* lr_critic_run;           /* double[R] or NULL */
    const float* beta_run;                 /* float[R] or NULL */
    float *actor_params, *actor_grad, *actor_grad_accum, *actor_m, *actor_v;
    float *critic_params, *critic_grad, *critic_m, *critic_v;
    int32_t *actor_step, *critic_step;
    int32_t* env_state; double* env_hist; uint8_t* env_cls; int32_t* env_elapsed;
    uint8_t* pending_action;
    double* ep_return;
    float* obs; uint8_t* act; float* reward;
    float* loss_out;
    const uint8_t* inj_actions;            /* uint8[T+1, R*E] or NULL */
    float* partials; size_t partials_floats;  /* ia2c_a2c_partials_floats(desc) */
} ia2c_a2c_desc;
size_t ia2c_a2c_partials_floats(const ia2c_a2c_desc* d);
int ia2c_a2c_train_update(const ia2c_a2c_desc* d, void* stream);

/* ------------------------------------------------------------------ frozen-policy evaluation of IA2C actors -- */
/* Plays `episodes` episodes of T Org-N steps in each of E envs of each of R runs with the runs' actors frozen: no belief
 * filter, no critic, no update (the IA2C actor reads only the observation).  Every item (episode k, env e) starts from
 * the reset state, steps with the same-step autoreset at max_episode_steps (0: no limit) and sums its fp64 rewards in step
 * order.  Actions are sampled by the inverse CDF at a uniform or, with greedy != 0, are the argmax of the distribution
 * (ties to the lowest action, as torch.argmax).
 *
 * Layout: actor_params f32[R*N, 105], run r at rows [r*N, (r+1)*N) (as ia2c_runs_desc stacks them);
 *   policy        out f32[R*N, 9, 3]: each actor's softmax at observation class c = 3 * prev_cls + cur_cls (the one-hot
 *                 [onehot3(prev_cls), onehot3(cur_cls)]), bit-identical to the probabilities the training samplers draw from;
 *   returns       out f64[R, episodes, E] (greedy: f64[R]);
 *   action_counts out u64[R*N, 3], overwritten: how often each agent took each action over all items and steps;
 *   inj_u_action  f32[episodes, T, R*E, N] or NULL: the uniforms, instead of Philox (parity and tests; not with greedy).
 * Sampling without a tape: Philox stream 4, key = seed (the same for every run), counter = (index, t | 4 << 16,
 * episode0 + k) with index = e * ceil(N/4) + agent / 4 for env e within its run; agent i takes word i mod 4 and converts it
 * as the training sampler converts its word: (w >> 8) * 2^-24.  All runs and all evaluations with the same seed / episode0
 * thus see the same numbers: comparisons between runs are paired.
 *
 * Two launches: the policy table (which also zeroes action_counts), then the episodes.
 * Contract: run r computes byte for byte what an R = 1 call with run r's actor rows computes.  For fixed actor parameters
 * and an injected tape, returns and action counts are byte-identical to the env part of ia2c_rollout (ep_return, and the
 * counts of act[0..T-1]) fed U[t] = inj_u_action[0, t] with one episode.  Nothing outside policy, returns and
 * action_counts is written.
 * Every check runs before the first CUDA call: a NULL descriptor or output pointer, R, N, E, episodes or T out of range,
 * R * N above IA2C_MAX_RUN_NETS, E * episodes beyond one grid, episode0 + episodes above 2^32, greedy with
 * E * episodes != 1 (Org is deterministic: every greedy episode of a run is the same) or with a tape, and a policy
 * workspace smaller than ia2c_eval_policy_floats(desc). */
#define IA2C_EVAL_MAX_RUNS 65535     /* R: one grid row per run */
#define IA2C_EVAL_MAX_AGENTS 1023    /* a step's action counts are packed in 10-bit fields */
#define IA2C_EVAL_MAX_STEPS 65535    /* T: the t field of the Philox counter is 16 bits */
typedef struct ia2c_eval_desc {
    const float* actor_params;       /* f32[R*N, 105] */
    int32_t R, N;                    /* 1 <= R, 2 <= N <= 1023, R * N <= IA2C_MAX_RUN_NETS */
    int64_t E;                       /* envs per run */
    int32_t episodes, T, max_episode_steps, greedy;
    uint64_t seed;                   /* Philox key (stream 4) */
    uint32_t episode0;               /* Philox episode of item k is episode0 + k; episode0 + episodes <= 2^32 */
    const float* inj_u_action;       /* f32[episodes, T, R*E, N] or NULL */
    float* policy; size_t policy_floats;   /* out and workspace: f32[R*N, 9, 3], ia2c_eval_policy_floats(desc) */
    double* returns;                 /* out: f64[R, episodes, E] (greedy: f64[R]) */
    unsigned long long* action_counts;     /* out: u64[R*N, 3] */
} ia2c_eval_desc;
size_t ia2c_eval_policy_floats(const ia2c_eval_desc* d);
int ia2c_evaluate(const ia2c_eval_desc* d, void* stream);

/* ------------------------------------------------------------------ cross-play: lineups of actors from a pool -- */
/* Evaluates P lineups whose seats are filled from a pool of actors (the rows of one batch, or of several sources
 * concatenated), so that separately trained runs can be played against each other: the cross-play matrix of a sweep.
 *
 * Definitions: the pool is actor_params f32[nets, 105]; lineup p seats pool row lineups[p * N + i] in seat i (rows may
 * repeat within a lineup, and a row may sit in a seat other than the one it was trained in).  Lineup p plays `episodes`
 * (K) episodes of T steps in each of E envs exactly as ia2c_evaluate plays one run: same reset state, same-step autoreset at
 * max_episode_steps, fp64 step-order return, Philox stream 4 with the same counters (e = the env within the lineup), or
 * the argmax with greedy != 0 (E = K = 1).
 * Contract: lineup p computes, byte for byte, the returns and action counts that an R = 1 ia2c_evaluate call computes when
 * its actor rows are pool[lineups[p, 0..N-1]], with the same seed, episode0, E, K, T, max_episode_steps and greedy.  So the
 * lineup of run r's own agents reproduces run r's evaluation, and all lineups see the same random numbers: the cells of a
 * cross-play matrix are paired samples.
 *
 * Layout:
 *   lineups       i32[P, N], pool rows;
 *   policy        out and workspace f32[nets, 9, 3]: the pool's table, as ia2c_evaluate tabulates it (>= nets * 27 floats);
 *   returns       out f64[P, episodes, E];
 *   action_counts out u64[P * N, 3], overwritten: per lineup and seat;
 *   return_sum    out f64[P]: lineup p's n = K * E returns, items x[j] = returns[p] in row-major order, summed in a fixed order:
 *                 lane j of 256 adds x[j], x[j + 256], x[j + 512], ... in increasing order from +0.0, then a halving tree
 *                 combines the lanes (s[j] += s[j + w] for j < w, w = 128, 64, ..., 1) and the sum is s[0] (the order of
 *                 ia2c_record_episode's return_sum); every addition is one IEEE fp64 add, round to nearest;
 *   return_m2     out f64[P]: with mean = return_sum / n (one IEEE divide), the sum of (x[j] - mean)^2 (one subtract and one
 *                 multiply each, never fused) in the same order.  Both are the same bytes from run to run;
 *   inj_u_action  f32[episodes, T, P*E, N] or NULL: the uniforms instead of Philox (the evaluation tape with P in place of R).
 * Guarded entries: lineups live on the device and are not checked before the launches.  A lineup with an entry outside
 * [0, nets) reads nothing of the table; its returns, return_sum and return_m2 are NaN and its counts 0.  Other lineups are
 * unaffected.
 *
 * Three launches, all with programmatic dependent launch (table, lineups and returns read after the wait through L2):
 *   lineup_policy_kernel           the pool's table (ia2c_evaluate's per-row forward and softmax), and action_counts zeroed;
 *   lineup_episodes_kernel<WIDE>   ia2c_evaluate's episode kernel with the block's table gathered from the lineup's pool rows;
 *                                  grid (item blocks, y, z) with lineup p = blockIdx.z * gridDim.y + blockIdx.y, so that P
 *                                  may exceed 65535;
 *   lineup_stats_kernel            one warp per lineup: return_sum and return_m2.
 * Nothing outside policy, returns, action_counts, return_sum and return_m2 is written.
 * Every check runs before the first CUDA call: a NULL descriptor or pointer, N outside 2..1023, nets < 1, P outside
 * 1..IA2C_EVAL_MAX_LINEUPS, E, episodes, T, max_episode_steps, episode0 and greedy as ia2c_evaluate checks them, and a
 * policy workspace smaller than nets * 27 floats. */
#define IA2C_EVAL_MAX_LINEUPS 1048576   /* P: the full matrix of 1024 runs */
typedef struct ia2c_lineup_desc {
    const float* actor_params;       /* f32[nets, 105]: the pool */
    int32_t nets, N;                 /* pool rows >= 1; seats 2 <= N <= 1023 */
    int32_t P, reserved;             /* lineups, 1 <= P <= IA2C_EVAL_MAX_LINEUPS */
    const int32_t* lineups;          /* i32[P, N] */
    int64_t E;                       /* envs per lineup */
    int32_t episodes, T, max_episode_steps, greedy;
    uint64_t seed;                   /* Philox key (stream 4) */
    uint32_t episode0;               /* Philox episode of item k is episode0 + k; episode0 + episodes <= 2^32 */
    const float* inj_u_action;       /* f32[episodes, T, P*E, N] or NULL */
    float* policy; size_t policy_floats;   /* out and workspace: f32[nets, 9, 3] */
    double* returns;                 /* out: f64[P, episodes, E] */
    unsigned long long* action_counts;     /* out: u64[P*N, 3] */
    double* return_sum;              /* out: f64[P] */
    double* return_m2;               /* out: f64[P] */
} ia2c_lineup_desc;
int ia2c_evaluate_lineups(const ia2c_lineup_desc* d, void* stream);

/* ------------------------------------------------------------------ learning curves: per-episode statistics on the device -- */
/* Reduces the trajectory an episode just left into slot `slot` of a caller-owned ring, in ONE launch, so that learning curves
 * are read back in bulk instead of with a stream synchronisation per episode.  `d` is the descriptor the episode ran with: a
 * standalone trainer's (runs = 1) or a batch's stacked one (ia2c_runs_desc layout, E = envs per run, runs = R).  Read:
 * act, partner_true, partner_pred u8[T+1, R*E, N], ep_return f64[R*E], loss_out f32[2, R*N]; any path that fills them
 * (fused, whole-episode, per-step, injected tapes) is covered.  Nothing else of `d` is read and nothing of it is written.
 *
 * Definitions, for run r, agent i (net n = r*N + i) and all steps 0 <= t < T (the T steps the env took) and envs 0 <= e < E:
 *   action_counts[slot, n, a] = #{ act[t, r*E+e, i] == a }                                   (a = 0, 1, 2)
 *   partner_hits[slot, n]     = #{ partner_pred[t, r*E+e, i] == partner_true[t, r*E+e, i] }  (the belief filter's hit count)
 *   loss[slot]                = loss_out, byte for byte (critic row, then actor row)
 *   return_sum[slot, r]       = the run's E returns summed in a fixed order: lane j of 256 adds ep_return[r*E + j],
 *                               [r*E + j + 256], [r*E + j + 512], ... in increasing order from +0.0, then a halving tree
 *                               combines the lanes (s[j] += s[j + w] for j < w, w = 128, 64, ..., 1) and the sum is s[0];
 *                               every addition is one IEEE fp64 add, round to nearest.  The same bytes from run to run.
 *
 * The ring (device, allocated zeroed by the caller): capacity >= 2 slots of each array.  The call writes return_sum and
 * loss of slot s, ADDS the counts and hits of this episode into slot s with integer atomics, and zeroes the counts and hits
 * of slot (s + 1) mod capacity for the next call; it writes nothing else.  So slot s must hold zero counts when the call
 * runs (a zeroed ring, or the previous call on slot s - 1), and slot (s + 1) mod capacity must have been read before the call
 * on slot s is enqueued: the ring holds at most capacity - 1 episodes that have not been read.
 * Launched with programmatic dependent launch; the trajectory is read after the wait through L2.
 * Every check runs before the first CUDA call: a NULL descriptor or pointer, runs < 1, N, T or E < 1, runs * N above
 * IA2C_MAX_RUN_NETS, capacity < 2 and a slot outside [0, capacity) (IA2C_ERR_INVALID); env_offset != 0 or E_total != E
 * (a multi-GPU shard; IA2C_ERR_UNSUPPORTED); T * E >= 2^32 (u32 counts; IA2C_ERR_INVALID). */
typedef struct ia2c_history_desc {
    int32_t capacity;                 /* episodes the ring holds, >= 2 */
    double* return_sum;               /* out f64[capacity, R]: sum of ep_return over the run's E envs */
    float* loss;                      /* out f32[capacity, 2, R*N]: copy of loss_out (critic row, actor row) */
    uint32_t* action_counts;          /* out u32[capacity, R*N, 3] */
    uint32_t* partner_hits;           /* out u32[capacity, R*N] */
} ia2c_history_desc;
int ia2c_record_episode(const ia2c_episode_desc* d, int32_t runs, const ia2c_history_desc* h, int32_t slot, void* stream);

/* ------------------------------------------------------------------ population-based training of a batch of runs -- */
/* One generation of population-based training (PBT) on a batch of R runs (ia2c_runs_desc layout, `d` the batch's episode
 * descriptor, `h` its history ring as ia2c_record_episode fills it), entirely on the device: rank the runs by their recent
 * training returns, overwrite the worst q with copies of runs drawn from the best q, and perturb the copies'
 * hyper-parameters.  Called between episodes; nothing is read back to the host.
 *
 * Definitions (R runs of N agents, w = p->window, s = p->slot the ring slot of the newest record, C = h->capacity):
 *   fitness[r]  = the fp64 sum of return_sum[(s - w + 1 + k) mod C, r] for k = 0 .. w - 1, oldest first, added in that
 *                 order from +0.0 with one IEEE fp64 add each (round to nearest).  The same bytes from run to run.
 *   order       the runs sorted by fitness, higher first; a NaN fitness ranks below every non-NaN one; ties (equal
 *                 fitness, both NaN included; -0.0 == +0.0) go to the lower run index.  A total order: rank[r] is r's
 *                 position in it, order[rank[r]] = r.
 *   recipients  the bottom q runs, order[R - q + j] for j = 0 .. q - 1; donors are drawn from the top q, order[0 .. q-1].
 *                 2q <= R, so the two sets are disjoint.
 *   donor       recipient v draws ONE Philox block, stream 5: key = p->seed, counter = (v, 0, 0 | 5 << 16,
 *                 p->generation) (the layout of the other streams: index v, t = 0, episode = generation) -> words
 *                 (x, y, z, w); donor = order[((x >> 8) * q) >> 24], in unsigned 64-bit integer arithmetic.
 *   copy        every byte of the recipient's rows [v*N, (v+1)*N) of actor_params, critic_params, actor_m, actor_v,
 *                 critic_m, critic_v, actor_step, critic_step, actor_grad_accum and filter_action becomes the byte of the
 *                 donor's rows as it was before the call.  Nothing else of `d` is written: not the env state, trajectory,
 *                 ep_return, belief_records, loss_out, actor_grad or critic_grad, and no row of a run that is not a
 *                 recipient.  The recipient keeps its seed.
 *   explore     the recipient takes the donor's lr_actor, lr_critic, gamma and beta; then, for each set bit of
 *                 p->perturb, f = p->factor_hi if the top bit of the word is set, else p->factor_lo, and
 *                   lr_actor  = __dmul_rn(lr_actor, f)                       (bit 0, IA2C_PBT_LR_ACTOR, word y)
 *                   lr_critic = __dmul_rn(lr_critic, f)                      (bit 1, IA2C_PBT_LR_CRITIC, word z)
 *                   beta      = __double2float_rn(__dmul_rn((double)beta, f)) (bit 2, IA2C_PBT_BETA, word w)
 *                 gamma is inherited, never perturbed.  Other runs' hyper-parameters are unchanged.
 * The hyper-parameters live in the four device arrays of `p` (read and written), which must be the arrays the batch's
 * ia2c_runs_desc points at for its next episode to train with them.
 *
 * Log (device, written for every run r): log_fitness[r], log_rank[r], log_donor[r] (-1: not a recipient) and the four
 * hyper-parameters of run r after the step.  workspace: ia2c_pbt_workspace_bytes(R) bytes, int32 order[R].
 *
 * Two launches, both with programmatic dependent launch (ring rows, parameters and hyper-parameters are read after the wait
 * through L2): pbt_rank_kernel (ceil(R / 256) blocks of 256 threads, one thread per run, O(R^2) compares over fitness tiles
 * staged in shared memory) and pbt_apply_kernel (q x ceil(N / agents per block) blocks: the draw, the log row and the
 * hyper-parameters of recipient j in block (j, 0), the row copies in 16-byte words where donor and recipient rows share
 * their 16-byte alignment, else 4-byte words).  q = 0 launches both kernels, logs, and changes no training byte.
 * Every check runs before the first CUDA call: a NULL descriptor or pointer (the ten buffers above, h->return_sum, the
 * four hyper-parameter arrays, the seven log arrays, the workspace), R < 1, N < 1, R * N above IA2C_MAX_RUN_NETS, capacity
 * < 2, window outside [1, capacity - 1], a slot outside [0, capacity), q < 0 or 2q > R, perturb bits other than the three
 * above, a factor that is not finite and > 0, a workspace smaller than ia2c_pbt_workspace_bytes(R) (IA2C_ERR_INVALID);
 * env_offset != 0 or E_total != E (a multi-GPU shard; IA2C_ERR_UNSUPPORTED). */
#define IA2C_PBT_LR_ACTOR 1
#define IA2C_PBT_LR_CRITIC 2
#define IA2C_PBT_BETA 4
typedef struct ia2c_pbt_desc {
    int32_t window;                   /* episodes summed into the fitness, 1 <= window <= capacity - 1 */
    int32_t slot;                     /* ring slot of the newest record */
    int32_t q;                        /* recipients (and donor candidates), 0 <= 2q <= R */
    uint32_t perturb;                 /* IA2C_PBT_* bits */
    double factor_lo, factor_hi;      /* multipliers for a clear / set top bit, finite and > 0 */
    uint64_t seed;                    /* Philox key (stream 5) */
    uint32_t generation;              /* Philox counter word 3 */
    int32_t reserved;
    double* lr_actor;                 /* in/out device double[R] */
    double* lr_critic;                /* in/out device double[R] */
    float* gamma;                     /* in/out device float[R] */
    float* beta;                      /* in/out device float[R] */
    double* log_fitness;              /* out f64[R] */
    int32_t* log_rank;                /* out i32[R] */
    int32_t* log_donor;               /* out i32[R], -1 for a run that kept its own state */
    double* log_lr_actor;             /* out f64[R], after the step */
    double* log_lr_critic;            /* out f64[R] */
    float* log_gamma;                 /* out f32[R] */
    float* log_beta;                  /* out f32[R] */
    void* workspace; size_t workspace_bytes;
} ia2c_pbt_desc;
size_t ia2c_pbt_workspace_bytes(int32_t runs);
int ia2c_pbt_step(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_history_desc* h, const ia2c_pbt_desc* p,
                  void* stream);

/* ------------------------------------------------------------------ frozen partners: train against a pool of actors -- */
/* Seats frozen actors from a pool in each run's partner seats before an episode, so that the learning seats train against
 * partners drawn from a population (fictitious co-play, population play) instead of against one co-learning partner.  Called
 * before the episode's entry point (ia2c_train_episode, ia2c_rollout, ia2c_train_episode_runs, ia2c_train_episode_runs_many),
 * which then runs unchanged.  Nothing is read back to the host.
 *
 * Definitions (R runs of N agents: `r` NULL is one standalone run, R = 1, keyed by d->seed; else the batch's stacked layout):
 *   pool    rows f32[P, 105], actor rows (any row may sit in any seat: the IA2C actor reads only the shared observation);
 *           seats i32[S], the partner seats, distinct, in [0, N), 1 <= S <= N - 1 (at least one seat keeps learning);
 *           teams i32[Q, S]: team t seats pool row teams[t, j] in seat seats[j].
 *   draw    before episode k run r draws ONE Philox block, stream 6: key = the run's training seed (r->seed[run], or d->seed),
 *           counter = (0, 0, 0 | 6 << 16, k) (the layout of the other streams: index 0, t = 0, episode = k = p->episode)
 *           -> words (x, y, z, w); team = (x * Q) >> 32 in unsigned 64-bit arithmetic.  A run of a batch and a standalone
 *           trainer with the same seed draw the same teams.
 *   seat    for each j < S, the 420 bytes of actor_params row r*N + seats[j] become pool row teams[team, j].  Nothing else of
 *           `d` is written: the partner seats' critic, Adam moments and steps, actor_grad_accum, belief records and models stay
 *           as they are, and the episode then runs and updates every seat as it always does.  The partner seats' updates are
 *           discarded by the next call; the row a partner seat holds after an episode is its partner plus one update.
 * Contract: a run trained with ia2c_seat_partners before each episode computes, byte for byte, what the same entry point
 * computes when the caller writes the drawn team's rows into the seat rows itself before each episode.
 * Guarded entries: seats and teams live on the device and are not checked before the launch.  A run whose drawn team has an
 * entry outside [0, P), or whose seats have one outside [0, N), writes none of its seats and logs -1; other runs are unaffected.
 * Log: log_team[run] = the drawn team, or -1 (out i32[R]).
 *
 * One launch with programmatic dependent launch: partner_seat_kernel, grid (R, ceil(S / seats per block)); every block redraws
 * its run's Philox block and checks the run's S entries, one thread copies each 4-byte word of a row.  It waits before its
 * first store (the previous episode's reduce + Adam and ia2c_pbt_step write the rows it overwrites), reads seats, teams and the
 * seeds after the wait through L2, and releases its successor first thing: every first kernel of an episode reads actor_params
 * only after its own wait.
 * Every check runs before the first CUDA call: a NULL descriptor or pointer (d->actor_params, rows, seats, teams, log_team,
 * r->seed), runs < 1, runs * N above IA2C_MAX_RUN_NETS, S outside 1..N-1, P < 1, Q outside 1..IA2C_PARTNER_MAX_TEAMS
 * (IA2C_ERR_INVALID); env_offset != 0 or E_total != E (a multi-GPU shard; IA2C_ERR_UNSUPPORTED). */
#define IA2C_PARTNER_MAX_TEAMS 1048576   /* Q */
typedef struct ia2c_partner_desc {
    const float* rows;                /* f32[P, 105]: the pool */
    int32_t P;                        /* pool rows >= 1 */
    const int32_t* seats;             /* i32[S] */
    int32_t S;                        /* 1 <= S <= N - 1 */
    const int32_t* teams;             /* i32[Q, S] */
    int32_t Q;                        /* 1 <= Q <= IA2C_PARTNER_MAX_TEAMS */
    uint32_t episode;                 /* Philox counter word 3: the episode about to run */
    int32_t* log_team;                /* out i32[R] */
} ia2c_partner_desc;
int ia2c_seat_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_partner_desc* p, void* stream);

/* ------------------------------------------------------------------ frozen partners per env -- */
/* A second partner mode: instead of one team per run and episode (ia2c_seat_partners), every ENV draws its own team before
 * every episode, and the rollout kernels play it in that env.  A learner of E envs then meets up to E partners per episode,
 * so each actor update averages over the pool instead of following one partner's convention (population play).
 *
 * Definitions (R runs of N agents, E envs per run; `r` NULL is one standalone run, R = 1, keyed by d->seed):
 *   pool    rows, P, seats, S, teams, Q as in ia2c_partner_desc; policy f32[P, 9, 3], row p's softmax at observation class
 *           c = 3 * prev + cur, as ia2c_partner_policy writes it (it is what the training samplers compute from row p).
 *   draw    before episode k = d->episode, env e of run r (e counted within its run) draws ONE Philox block, stream 7:
 *           key = the run's training seed (r->seed[run], or d->seed), counter = (e, 0, 0 | 7 << 16, k) -> words (x, y, z, w);
 *           team = (x * Q) >> 32 in unsigned 64-bit arithmetic.  A run of a batch and a standalone trainer with the same seed
 *           draw the same teams.
 *   play    in env e the agent in seat seats[j] acts with pool row teams[team, j]: the same observation, action uniform and
 *           inverse-CDF sampler as with its own row (if a seat repeats, the lowest j wins).  Nothing of the run's own state is
 *           read or written for this: the partner seats' own actor rows are never used to act while the mode is on, yet they
 *           receive the episode's updates as every seat does (their critics, beliefs and Adam state are trained on the
 *           partners' actions).  A run that leaves the mode continues self-play from those rows.  To keep them as they are,
 *           train with the partner seats frozen (ia2c_train_episode_frozen, below).
 *   guard   an env whose drawn team has a row outside [0, P), or whose seats have one outside [0, N), plays the run's own rows
 *           in every seat and logs -1; other envs are unaffected.
 *   log     log_env_team[r * E + e] = the drawn team, or -1 (out i32[R, E], written by the rollout kernel).
 * Contract: the trajectory is byte-equal to what the same kernel path produces if env e's partner seats held team t_e's rows;
 * with Q = 1 the mode equals ia2c_seat_partners before each episode, byte for byte, in everything the partner seats' actor rows
 * do not feed.  Everything after the rollout (critic, belief filter, actor gradient of every seat) is unchanged.
 *
 * Kernels: the PARTNERS instantiations of rollout_fused_kernel (N <= 8, every (N, M) it has, standalone and batched: every
 * env's lane group draws its team once before the step loop, a partner lane loads its pool row into registers, the group's
 * leader logs) and rollout_many_kernel (9 <= N <= 256: the block's owner threads draw the chunk's teams into shared memory and
 * log them, a partner-seat thread samples from policy[teams[team, j]] at the env's class).  Pool, seats, teams and table are
 * read after griddepcontrol.wait.  An episode makes exactly the launches of the unpartnered entry point.
 *
 * ia2c_partner_policy: one launch (programmatic dependent launch) writing policy f32[P, 9, 3] from rows f32[P, 105] with the
 * forward and softmax of ia2c_evaluate's table; build it once per pool (needed for N > 8; the N <= 8 kernels read the rows).
 * ia2c_rollout_env_partners: what ia2c_rollout does, standalone.  ia2c_train_episode_env_partners: r NULL is
 * ia2c_train_episode; otherwise ia2c_train_episode_runs (N <= 8) or ia2c_train_episode_runs_many (9 <= N <= 256), with the
 * same descriptors and checks.
 * Refusals, all before the first CUDA call.  IA2C_ERR_INVALID: a NULL descriptor or pointer (rows, seats, teams, log_env_team,
 * r->seed; policy when N > 8), runs < 1, N < 2, runs * N above IA2C_MAX_RUN_NETS, S outside 1..N-1, P < 1, Q outside
 * 1..IA2C_PARTNER_MAX_TEAMS, and whatever the unpartnered entry point refuses as invalid.  IA2C_ERR_UNSUPPORTED: every path
 * without a PARTNERS instantiation (standalone N <= 8 without IA2C_FLAG_FUSED_ROLLOUT, an (N, M) without a fused
 * instantiation, N > 256, IA2C_FLAG_ROLLOUT_PER_STEP or IA2C_FLAG_BELIEF_PER_STEP, no whole-episode belief kernel), injected
 * actions (inj_actions), and a multi-GPU shard (env_offset != 0 or E_total != E). */
typedef struct ia2c_env_partner_desc {
    const float* rows;                /* f32[P, 105]: the pool */
    int32_t P;                        /* pool rows >= 1 */
    const float* policy;              /* f32[P, 9, 3] from ia2c_partner_policy; may be NULL for N <= 8 */
    const int32_t* seats;             /* i32[S] */
    int32_t S;                        /* 1 <= S <= N - 1 */
    const int32_t* teams;             /* i32[Q, S] */
    int32_t Q;                        /* 1 <= Q <= IA2C_PARTNER_MAX_TEAMS */
    int32_t* log_env_team;            /* out i32[R, E] */
} ia2c_env_partner_desc;
int ia2c_partner_policy(const float* rows, int32_t P, float* policy, void* stream);
int ia2c_rollout_env_partners(const ia2c_episode_desc* d, const ia2c_env_partner_desc* p, void* stream);
int ia2c_train_episode_env_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p,
                                    void* stream);

/* ------------------------------------------------------------------ prioritized partners per env -- */
/* The per-env mode above draws every team with probability 1/Q, so a learner spends most of its samples on partners it
 * already plays well with.  Prioritized draws (prioritized fictitious self-play) weight each team by how badly the run does
 * with it, from statistics the device records after every episode: no host round trip.  Only the per-env mode has them.
 *
 * Definitions (R runs, E envs per run, Q teams; a standalone run is R = 1):
 *   statistics  count i64[R, Q] and sum i64[R, Q].  ia2c_record_partner_returns, after a prioritized episode, adds for every
 *               env e of run r with logged team t = env_team[r * E + e]:  count[r, t] += 1,
 *               sum[r, t] += llrint(ep_return[r * E + e] * 2^20) (round half to even: fixed point with 20 fraction bits).
 *               An env is skipped where t lies outside [0, Q) (a logged -1), where its return is not finite, or where
 *               |return| * 2^20 >= 2^62.  Integer adds give the same bytes in any order (64-bit atomics); sums wrap.
 *   weights     ia2c_prioritize_partners(power p in 0..16, floor f in [0, 1]), per run, in fp64 with correctly rounded
 *               operations and no contraction:  for every played team (count > 0) m_q = ((double)sum_q * 2^-20) / (double)count_q;
 *               hi, lo = the largest and smallest m_q.  No team played, or hi == lo: W_q = 2^24 for every q.  Otherwise
 *               x_q = (hi - m_q) / (hi - lo) and w_q = f + (1 - f) * x_q^p for a played team (x^p multiplied left to right from
 *               x^0 = 1), w_q = 1 (the worst played team's weight: untried partners are tried) for an unplayed one, and
 *               W_q = min(2^24, floor(w_q * 2^24)).
 *   table       u64[R, Q + 1]: C_0 = 0, C_{q+1} = C_q + W_q.  Equal weights (C_q = q * 2^24) until the first
 *               ia2c_prioritize_partners; the caller initialises it so.  `reset` zeroes the run's statistics in the same launch.
 *   draw        env e of run r takes the stream-7 word x of ia2c_env_partner_desc's draw; y = floor(x * C_Q / 2^32) (a 128-bit
 *               product) and the team is the q with C_q <= y < C_{q+1}: teams of weight 0 are never drawn.  With equal
 *               weights this is (x * Q) >> 32 exactly, so a prioritized run equals a uniform per-env run byte for byte until
 *               its first ia2c_prioritize_partners.  C_Q = 0 logs -1 (the env plays its own rows); the guard of the per-env
 *               mode is unchanged.
 *
 * ia2c_rollout_env_partners_prioritized / ia2c_train_episode_env_partners_prioritized: ia2c_rollout_env_partners /
 * ia2c_train_episode_env_partners drawing from w->table (the PARTNERS instantiations of the rollout kernels: same launches).
 * ia2c_record_partner_returns: one launch (partner_returns_kernel, one thread per (run, env)) after the episode's kernels,
 * reading d->ep_return (R * E entries) and the episode's env-team log.  ia2c_prioritize_partners: one launch
 * (partner_priority_kernel, one block per run: min / max, weights, prefix scan, optional reset).  All programmatic dependent
 * launches that read nothing before griddepcontrol.wait.
 * Refusals, all before the first CUDA call.  IA2C_ERR_INVALID: a NULL descriptor or pointer (count, sum, table; env_team,
 * d->ep_return), R < 1, Q outside 1..IA2C_PARTNER_MAX_TEAMS, R * Q above IA2C_PARTNER_PRIORITY_MAX_CELLS, E < 1, p outside
 * 0..16, f outside [0, 1], and for the twins R != runs or Q != the pool's Q, with everything the uniform entry points refuse
 * (with their status).  IA2C_ERR_UNSUPPORTED: ia2c_record_partner_returns on a multi-GPU shard (env_offset != 0 or
 * E_total != E). */
#define IA2C_PARTNER_PRIORITY_MAX_CELLS 16777216   /* R * Q: 16 B of statistics per cell */
typedef struct ia2c_partner_priority_desc {
    int64_t* count;                   /* i64[R, Q] */
    int64_t* sum;                     /* i64[R, Q]: returns in fixed point, 2^-20 */
    uint64_t* table;                  /* u64[R, Q + 1]: prefix sums of the weights */
    int32_t R;                        /* runs >= 1 */
    int32_t Q;                        /* teams, the pool's Q */
} ia2c_partner_priority_desc;
int ia2c_rollout_env_partners_prioritized(const ia2c_episode_desc* d, const ia2c_env_partner_desc* p,
                                          const ia2c_partner_priority_desc* w, void* stream);
int ia2c_train_episode_env_partners_prioritized(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p,
                                                const ia2c_partner_priority_desc* w, void* stream);
int ia2c_record_partner_returns(const ia2c_episode_desc* d, const int32_t* env_team, const ia2c_partner_priority_desc* w,
                                void* stream);
int ia2c_prioritize_partners(const ia2c_partner_priority_desc* w, int32_t power, double floor_weight, int32_t reset, void* stream);

/* ------------------------------------------------------------------ frozen seats -- */
/* Trains an episode with some seats frozen: a frozen seat acts (with its own actor row, a row seated by ia2c_seat_partners
 * before the call, or its env's pool row), but nothing of it is updated and the update kernels skip it.  With the partner
 * seats frozen this is training against truly frozen partners; with no pool it trains a best response to fixed co-players.
 *
 * Definitions (R runs of N agents, the same mask for every run; `r` NULL is one standalone run):
 *   mask        bit n of mask[n >> 6] set: seat n is frozen.  No bit at or above N; at least one seat frozen and one trained.
 *   trained     every byte of every buffer of a trained seat, and the trajectory, ep_return, env state and partner logs, are
 *               what the same entry point computes with nothing frozen: a seat's critic, actor gradient and beliefs read only
 *               the trajectory and that seat's own rows.
 *   frozen      net n = run * N + seat of a frozen seat: actor_params, critic_params, actor_grad, critic_grad, actor_m / v,
 *               critic_m / v, actor_step, critic_step and actor_grad_accum are byte-unchanged (ia2c_seat_partners, before the
 *               call, writes actor rows as it always does); loss_out[0, n] and loss_out[1, n] are NaN.
 *   beliefs     N <= 8: the fused rollout runs every seat's filter as before, so a frozen seat's belief records and
 *               partner_pred are what they are with nothing frozen.  9 <= N <= 256: the whole-episode belief kernel skips
 *               frozen rows: their records are untouched and their partner_pred entries (all T + 1 steps) are 0xFF, "no
 *               prediction"; a standalone episode with parity dumps writes no pred_dump / belief_dump entry of theirs either
 *               (those slots keep what they held).
 * Paths: those with whole-episode kernels.  Standalone: N <= 8 with IA2C_FLAG_FUSED_ROLLOUT (with or without
 * IA2C_FLAG_FUSED_CRITIC), 9 <= N <= 256 with the whole-episode rollout and belief kernels; both with IA2C_FLAG_ACTOR_COLUMNS.
 * Batches: ia2c_train_episode_runs (N <= 8) and ia2c_train_episode_runs_many (9 <= N <= 256).  p (the per-env pool) and w
 * (prioritized draws; needs p) may be NULL, as for ia2c_train_episode_env_partners(_prioritized).  The launches are those of
 * the unfrozen entry point (4 at N <= 8, 6 at 9..256); ia2c_seat_partners before and ia2c_record_partner_returns after the
 * call stay the caller's.  Kernels: instantiations of the gradient, reduce and whole-episode belief kernels over the trained
 * seats, whose list the entry point builds from the mask and passes by value; each trained net keeps the partition and the
 * partial rows of the unfrozen episode, so its fixed-order sums are the same sums.
 * Refusals, all before the first CUDA call.  IA2C_ERR_INVALID: a NULL mask, a bit at or above N, no seat frozen or none
 * trained, and whatever the unfrozen entry point refuses.  IA2C_ERR_UNSUPPORTED: IA2C_FLAG_SKIP_ADAM or IA2C_FLAG_GRAD_ONLY,
 * a multi-GPU shard (env_offset != 0 or E_total != E), IA2C_FLAG_ROLLOUT_PER_STEP or IA2C_FLAG_BELIEF_PER_STEP, N <= 8
 * without IA2C_FLAG_FUSED_ROLLOUT or a fused instantiation, N > 256 or no whole-episode belief kernel, the pipelined actor
 * kernel (no IA2C_FLAG_ACTOR_COLUMNS), and injected tapes in a batch. */
typedef struct ia2c_frozen_seats {
    uint64_t mask[4];                 /* host memory: bit n set, seat n frozen (N <= 256) */
} ia2c_frozen_seats;
int ia2c_train_episode_frozen(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p,
                              const ia2c_partner_priority_desc* w, const ia2c_frozen_seats* f, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IA2C_B200_H */
