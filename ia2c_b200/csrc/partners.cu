// partners.cu — seat frozen partners from a pool in each run's partner seats before an episode (ia2c_seat_partners), and the
// pool's policy table and refusals of the per-env mode (ia2c_partner_policy, ia2c_train_episode_env_partners; its kernels are
// the PARTNERS instantiations of the rollout kernels in rollout_fused.cu and trainer.cu).
//
// ONE launch, partner_seat_kernel, grid (R, ceil(S / kSeatsPerBlock)), block (128, kSeatsPerBlock): row y of block (r, b)
// serves seat slot j = b * kSeatsPerBlock + y of run r, thread x < 105 copies word x of the 105-float row.  Every block
// redraws its run's stream-6 Philox block (10 rounds, cheaper than a second launch) and checks all S entries of the drawn team
// and all S seats, so that a run with a bad entry writes none of its seats whichever block finds it; block (r, 0) logs.
// Launched with launch_pdl: it releases its successor first thing (every first kernel of an episode loads actor_params only
// after its own griddepcontrol.wait: rollout_fused_kernel, rollout_many_kernel, env_step_kernel / actor_step_kernel) and
// waits before its first load and store (the previous episode's reduce_adam_kernel and pbt_apply_kernel write the rows).
#include <math_constants.h>

#include "common.cuh"
#include "mlp_f2.cuh"

namespace ia2c {
namespace {

constexpr uint32_t kStreamPartners = 6;
constexpr int kWordThreads = 128;    // >= kActorP words of a row
constexpr int kSeatsPerBlock = 4;

struct SeatArgs {
    float* actor_params;
    const uint64_t* seeds;           // device u64[R], or NULL: every run is keyed by `seed`
    uint64_t seed;
    const float* rows;
    const int32_t *seats, *teams;
    int32_t N, P, S, Q;
    uint32_t episode;
    int32_t* log_team;
};

__global__ void __launch_bounds__(kWordThreads * kSeatsPerBlock) partner_seat_kernel(const __grid_constant__ SeatArgs a) {
    pdl_prologue();
    const int run = blockIdx.x;
    const uint64_t key = a.seeds ? __ldcg(reinterpret_cast<const unsigned long long*>(a.seeds) + run) : a.seed;
    const uint32_t x = philox_draw(key, kStreamPartners, a.episode, 0u, 0ull).x;
    const int team = (int)(((uint64_t)x * (uint64_t)a.Q) >> 32);
    const int32_t* trow = a.teams + (int64_t)team * a.S;
    const int tid = threadIdx.y * kWordThreads + threadIdx.x;
    bool bad = false;
    for (int j = tid; j < a.S; j += kWordThreads * kSeatsPerBlock) {
        const int32_t row = __ldcg(trow + j), seat = __ldcg(a.seats + j);
        bad |= row < 0 || row >= a.P || seat < 0 || seat >= a.N;
    }
    bad = __syncthreads_or(bad);
    if (blockIdx.y == 0 && tid == 0) a.log_team[run] = bad ? -1 : team;
    const int j = blockIdx.y * kSeatsPerBlock + threadIdx.y;
    if (bad || j >= a.S || threadIdx.x >= kActorP) return;
    const int64_t src = (int64_t)__ldcg(trow + j) * kActorP, dst = ((int64_t)run * a.N + __ldcg(a.seats + j)) * kActorP;
    a.actor_params[dst + threadIdx.x] = __ldcg(a.rows + src + threadIdx.x);
}

int validate_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_partner_desc* p) {
    const char* who = "ia2c_seat_partners";
    IA2C_REQUIRE(d && p, "%s: null episode or partner descriptor", who);
    IA2C_REQUIRE(d->actor_params, "%s: null actor_params", who);
    IA2C_REQUIRE(p->rows && p->seats && p->teams && p->log_team, "%s: null rows, seats, teams or log_team", who);
    IA2C_REQUIRE(!r || r->seed, "%s: null seed array in the runs descriptor", who);
    const int32_t R = r ? r->runs : 1;
    IA2C_REQUIRE(R >= 1, "%s: runs=%d must be >= 1", who, R);
    IA2C_REQUIRE(d->N >= 2, "%s: N=%d must be >= 2 (a partner seat and a learning seat)", who, d->N);
    IA2C_REQUIRE((int64_t)R * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS (%d)", who,
                 (long long)R * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(p->S >= 1 && p->S <= d->N - 1, "%s: S=%d outside [1, N - 1 = %d]", who, p->S, d->N - 1);
    IA2C_REQUIRE(p->P >= 1, "%s: P=%d must be >= 1", who, p->P);
    IA2C_REQUIRE(p->Q >= 1 && p->Q <= IA2C_PARTNER_MAX_TEAMS, "%s: Q=%d outside [1, IA2C_PARTNER_MAX_TEAMS = %d]", who, p->Q,
                 IA2C_PARTNER_MAX_TEAMS);
    if (d->env_offset != 0 || d->E_total != d->E) {
        set_error("%s: env_offset=%lld, E_total=%lld, E=%lld: partners are seated on one GPU (env_offset 0, E_total = E)", who,
                  (long long)d->env_offset, (long long)d->E_total, (long long)d->E);
        return IA2C_ERR_UNSUPPORTED;
    }
    return 0;
}

constexpr int kPolicyThreads = 128;

// one thread per (pool row, observation class); the rows are read after the wait, through L2
__global__ void __launch_bounds__(kPolicyThreads) partner_policy_kernel(const float* rows, int32_t P, float* policy) {
    pdl_prologue();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < (int64_t)P * kObsClasses) policy_row(rows, policy, idx);
}

// ---------------------------------------------------------------- prioritized partners per env
constexpr int kReturnThreads = 256;
constexpr int kPriorityThreads = 256;
constexpr double kFix = 1048576.0;                     // 2^20: fixed-point scale of the return sums
constexpr double kFixLimit = 4611686018427387904.0;    // 2^62
constexpr unsigned long long kUnitWeight = 1ull << 24;

struct ReturnArgs {
    const double* ep_return;          // f64[R * E]
    const int32_t* team;              // i32[R * E]: the episode's env-team log
    unsigned long long *count, *sum;  // i64[R, Q], added to as u64 (two's complement)
    int64_t E, n;                     // envs per run, R * E
    int32_t Q;
};

// one thread per (run, env): integer atomics, so the sums are the same bytes in any order
__global__ void __launch_bounds__(kReturnThreads) partner_returns_kernel(const __grid_constant__ ReturnArgs a) {
    pdl_prologue();   // the log and the returns are written by the episode's rollout kernel
    const int64_t g = (int64_t)blockIdx.x * kReturnThreads + threadIdx.x;
    if (g >= a.n) return;
    const int32_t t = __ldcg(a.team + g);
    const double v = __dmul_rn(__ldcg(a.ep_return + g), kFix);
    if (t < 0 || t >= a.Q || !(fabs(v) < kFixLimit)) return;   // a logged -1, a non-finite or too large return
    const int64_t cell = (g / a.E) * a.Q + t;
    atomicAdd(a.count + cell, 1ull);
    atomicAdd(a.sum + cell, (unsigned long long)llrint(v));   // round half to even
}

struct PriorityArgs {
    long long *count, *sum;           // i64[R, Q]
    unsigned long long* table;        // u64[R, Q + 1]
    double floor_w;
    int32_t Q, power, reset;
};

__device__ __forceinline__ double team_mean(long long s, long long n) {
    return __ddiv_rn(__dmul_rn((double)s, 1.0 / kFix), (double)n);
}

// one block per run: the played teams' min / max mean, then tiles of kPriorityThreads teams: weight, block-wide inclusive scan
// (integers: exact) plus the carry of the tiles before, and the reset of the cells just read
__global__ void __launch_bounds__(kPriorityThreads) partner_priority_kernel(const __grid_constant__ PriorityArgs a) {
    __shared__ double hi_s[kPriorityThreads / 32], lo_s[kPriorityThreads / 32];
    __shared__ unsigned long long warp_s[kPriorityThreads / 32];
    pdl_prologue();   // the statistics are written by the episodes' partner_returns_kernel
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, Q = a.Q;
    long long* cnt = a.count + (int64_t)blockIdx.x * Q;
    long long* sum = a.sum + (int64_t)blockIdx.x * Q;
    unsigned long long* c = a.table + (int64_t)blockIdx.x * (Q + 1);
    double hi = -CUDART_INF, lo = CUDART_INF;
    for (int q = tid; q < Q; q += kPriorityThreads) {
        const long long n = __ldcg(cnt + q);
        if (n > 0) {
            const double m = team_mean(__ldcg(sum + q), n);
            hi = fmax(hi, m), lo = fmin(lo, m);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    }
    if (lane == 0) hi_s[warp] = hi, lo_s[warp] = lo;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kPriorityThreads / 32; ++w) hi = fmax(hi, hi_s[w]), lo = fmin(lo, lo_s[w]);
    const bool equal = !(hi > lo);   // no team played, or hi == lo
    const double span = equal ? 1.0 : __dadd_rn(hi, -lo), keep = __dadd_rn(1.0, -a.floor_w);
    if (tid == 0) c[0] = 0ull;
    unsigned long long carry = 0ull;
    for (int base = 0; base < Q; base += kPriorityThreads) {
        const int q = base + tid;
        unsigned long long W = 0ull;
        if (q < Q) {
            const long long n = __ldcg(cnt + q);
            W = kUnitWeight;   // equal weights, or an unplayed team: w = 1
            if (!equal && n > 0) {
                const double x = __ddiv_rn(__dadd_rn(hi, -team_mean(__ldcg(sum + q), n)), span);
                double xp = 1.0;
                for (int k = 0; k < a.power; ++k) xp = __dmul_rn(xp, x);
                const double w = __dadd_rn(a.floor_w, __dmul_rn(keep, xp));
                W = min(kUnitWeight, (unsigned long long)__dmul_rn(w, (double)kUnitWeight));
            }
            if (a.reset) cnt[q] = 0, sum[q] = 0;
        }
        unsigned long long s = W;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += v;
        }
        if (lane == 31) warp_s[warp] = s;
        __syncthreads();
        unsigned long long before = carry, total = 0ull;
#pragma unroll
        for (int w = 0; w < kPriorityThreads / 32; ++w) {
            if (w < warp) before += warp_s[w];
            total += warp_s[w];
        }
        if (q < Q) c[q + 1] = before + s;
        carry += total;
        __syncthreads();   // warp_s is rewritten by the next tile
    }
}

}  // namespace

// Every refusal of ia2c_rollout_env_partners / ia2c_train_episode_env_partners that concerns the pool or the path; the episode
// descriptor's own buffers are checked by the entry points' existing checks after this.  No CUDA call.
int validate_env_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_env_partner_desc* p, const char* who) {
    IA2C_REQUIRE(d && p, "%s: null episode or partner descriptor", who);
    IA2C_REQUIRE(p->rows && p->seats && p->teams && p->log_env_team, "%s: null rows, seats, teams or log_env_team", who);
    IA2C_REQUIRE(!r || r->seed, "%s: null seed array in the runs descriptor", who);
    const int32_t R = r ? r->runs : 1;
    IA2C_REQUIRE(R >= 1, "%s: runs=%d must be >= 1", who, R);
    IA2C_REQUIRE(d->N >= 2, "%s: N=%d must be >= 2 (a partner seat and a learning seat)", who, d->N);
    IA2C_REQUIRE((int64_t)R * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS (%d)", who,
                 (long long)R * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(p->S >= 1 && p->S <= d->N - 1, "%s: S=%d outside [1, N - 1 = %d]", who, p->S, d->N - 1);
    IA2C_REQUIRE(p->P >= 1, "%s: P=%d must be >= 1", who, p->P);
    IA2C_REQUIRE(p->Q >= 1 && p->Q <= IA2C_PARTNER_MAX_TEAMS, "%s: Q=%d outside [1, IA2C_PARTNER_MAX_TEAMS = %d]", who, p->Q,
                 IA2C_PARTNER_MAX_TEAMS);
    IA2C_REQUIRE(d->N <= 8 || p->policy, "%s: null policy table (N=%d > 8 samples partner seats from it: ia2c_partner_policy)", who, d->N);
    auto unsupported = [&](const char* what) {
        set_error("%s: %s", who, what);
        return IA2C_ERR_UNSUPPORTED;
    };
    if (d->env_offset != 0 || d->E_total != d->E)
        return unsupported("partners per env are played on one GPU (env_offset 0, E_total = E)");
    if (d->inj_actions) return unsupported("injected actions replace the partners' samples (inj_actions must be NULL)");
    if (d->N > 256) return unsupported("N above 256 runs the per-step rollout, which has no partner instantiation");
    if (d->N <= 8) {
        if (!ia2c_rollout_fused_supported(d->N, d->M))
            return unsupported("this (N, M) has no fused rollout instantiation (N <= 8 needs M = 5, or N = 2 with M = 3)");
        if (!r && !(d->flags & IA2C_FLAG_FUSED_ROLLOUT))
            return unsupported("N <= 8 without IA2C_FLAG_FUSED_ROLLOUT runs the per-step rollout, which has no partner instantiation");
    } else if (!r && ((d->flags & (IA2C_FLAG_ROLLOUT_PER_STEP | IA2C_FLAG_BELIEF_PER_STEP)) || !ia2c_belief_supports_episode(d->N, d->M))) {
        return unsupported("the per-step rollout (ROLLOUT_PER_STEP, BELIEF_PER_STEP, or no whole-episode belief kernel) has no partner instantiation");
    }
    return 0;
}

EnvPartners env_partners_arg(const ia2c_env_partner_desc* p) {
    EnvPartners a;
    a.rows = p->rows, a.policy = p->policy, a.seats = p->seats, a.teams = p->teams;
    a.P = p->P, a.S = p->S, a.Q = p->Q, a.log = p->log_env_team;
    a.table = nullptr;
    return a;
}

// The checks of a prioritized partners descriptor that every entry point makes.  No CUDA call.
int validate_partner_priority(const ia2c_partner_priority_desc* w, const char* who) {
    IA2C_REQUIRE(w, "%s: null priority descriptor", who);
    IA2C_REQUIRE(w->count && w->sum && w->table, "%s: null count, sum or table", who);
    IA2C_REQUIRE(w->R >= 1, "%s: R=%d must be >= 1", who, w->R);
    IA2C_REQUIRE(w->Q >= 1 && w->Q <= IA2C_PARTNER_MAX_TEAMS, "%s: Q=%d outside [1, IA2C_PARTNER_MAX_TEAMS = %d]", who, w->Q,
                 IA2C_PARTNER_MAX_TEAMS);
    IA2C_REQUIRE((int64_t)w->R * w->Q <= IA2C_PARTNER_PRIORITY_MAX_CELLS,
                 "%s: R * Q = %lld above IA2C_PARTNER_PRIORITY_MAX_CELLS (%d)", who, (long long)w->R * w->Q,
                 IA2C_PARTNER_PRIORITY_MAX_CELLS);
    return 0;
}

}  // namespace ia2c

using namespace ia2c;

extern "C" int ia2c_partner_policy(const float* rows, int32_t P, float* policy, void* stream) {
    IA2C_REQUIRE(rows && policy, "ia2c_partner_policy: null rows or policy");
    IA2C_REQUIRE(P >= 1, "ia2c_partner_policy: P=%d must be >= 1", P);
    const int64_t items = (int64_t)P * kObsClasses;
    return launch_pdl("partner_policy_kernel", partner_policy_kernel, dim3((unsigned)ceil_div(items, kPolicyThreads)), dim3(kPolicyThreads), 0,
                      as_stream(stream), rows, P, policy);
}

extern "C" int ia2c_record_partner_returns(const ia2c_episode_desc* d, const int32_t* env_team, const ia2c_partner_priority_desc* w,
                                           void* stream) {
    const char* who = "ia2c_record_partner_returns";
    IA2C_REQUIRE(d, "%s: null episode descriptor", who);
    IA2C_REQUIRE(d->ep_return && env_team, "%s: null ep_return or env_team", who);
    if (int rc = validate_partner_priority(w, who)) return rc;
    IA2C_REQUIRE(d->E >= 1, "%s: E=%lld must be >= 1", who, (long long)d->E);
    if (d->env_offset != 0 || d->E_total != d->E) {
        set_error("%s: env_offset=%lld, E_total=%lld, E=%lld: partner returns are recorded on one GPU (env_offset 0, E_total = E)",
                  who, (long long)d->env_offset, (long long)d->E_total, (long long)d->E);
        return IA2C_ERR_UNSUPPORTED;
    }
    ReturnArgs a;
    a.ep_return = d->ep_return, a.team = env_team;
    a.count = reinterpret_cast<unsigned long long*>(w->count), a.sum = reinterpret_cast<unsigned long long*>(w->sum);
    a.E = d->E, a.n = (int64_t)w->R * d->E, a.Q = w->Q;
    return launch_pdl("partner_returns_kernel", partner_returns_kernel, dim3((unsigned)ceil_div(a.n, kReturnThreads)),
                      dim3(kReturnThreads), 0, as_stream(stream), a);
}

extern "C" int ia2c_prioritize_partners(const ia2c_partner_priority_desc* w, int32_t power, double floor_weight, int32_t reset,
                                        void* stream) {
    const char* who = "ia2c_prioritize_partners";
    if (int rc = validate_partner_priority(w, who)) return rc;
    IA2C_REQUIRE(power >= 0 && power <= 16, "%s: power=%d outside [0, 16]", who, power);
    IA2C_REQUIRE(floor_weight >= 0.0 && floor_weight <= 1.0, "%s: floor=%g outside [0, 1]", who, floor_weight);
    PriorityArgs a;
    a.count = reinterpret_cast<long long*>(w->count), a.sum = reinterpret_cast<long long*>(w->sum);
    a.table = reinterpret_cast<unsigned long long*>(w->table);
    a.floor_w = floor_weight, a.Q = w->Q, a.power = power, a.reset = reset != 0;
    return launch_pdl("partner_priority_kernel", partner_priority_kernel, dim3((unsigned)w->R), dim3(kPriorityThreads), 0,
                      as_stream(stream), a);
}

extern "C" int ia2c_seat_partners(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_partner_desc* p, void* stream) {
    if (int rc = validate_partners(d, r, p)) return rc;
    SeatArgs a;
    a.actor_params = d->actor_params;
    a.seeds = r ? r->seed : nullptr, a.seed = d->seed;
    a.rows = p->rows, a.seats = p->seats, a.teams = p->teams;
    a.N = d->N, a.P = p->P, a.S = p->S, a.Q = p->Q;
    a.episode = p->episode, a.log_team = p->log_team;
    const dim3 grid((unsigned)(r ? r->runs : 1), (unsigned)ceil_div(p->S, kSeatsPerBlock));
    return launch_pdl("partner_seat_kernel", partner_seat_kernel, grid, dim3(kWordThreads, kSeatsPerBlock), 0, as_stream(stream), a);
}
