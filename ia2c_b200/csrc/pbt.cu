// pbt.cu — population-based training of a batch of runs: rank, copy and perturb runs on the device between episodes.
//
// ia2c_pbt_step runs one PBT generation (include/ia2c_b200.h states the definitions) in TWO launches and reads nothing back:
//   pbt_rank_kernel    grid ceil(R / 256), 256 threads, one thread per run.  Thread r sums run r's fitness from the history
//                      ring (window rows, oldest first), then counts the runs that beat it: each block walks the runs in
//                      tiles of 256 whose fitness its threads compute into shared memory (every block recomputes the sums,
//                      window loads per run and tile, instead of a second launch).  The count is r's rank; the thread
//                      writes order[rank] = r to the workspace and run r's log row (fitness, rank, donor -1, the
//                      hyper-parameters as they are).  O(R^2) compares: ~10^9 at the largest legal batch, spread over the chip.
//   pbt_apply_kernel   grid (q, ceil(N / kAgentsPerBlock)), 256 threads.  Block (j, y) serves recipient v = order[R - q + j]:
//                      it draws v's stream-5 Philox block, resolves the donor through order, and copies the agents
//                      [y * kAgentsPerBlock, ...) of the donor's ten per-net buffers onto v's rows; block (j, 0) also writes
//                      v's inherited and perturbed hyper-parameters and its log row.  Donors and recipients are disjoint
//                      (2q <= R), so no block reads a row another block writes.
// Both are launched with launch_pdl; every producer-written byte (ring rows, order, parameters, hyper-parameters) is read
// after griddepcontrol.wait through L2 (ld.global.cg).  pbt_rank_kernel releases its successor first thing, as the episode's
// kernels do; pbt_apply_kernel does NOT: it writes filter_action, which the next episode's first kernels read before their
// wait (DESIGN.md §6, launch gaps), so their launch must wait for its completion.
#include <cmath>

#include "common.cuh"

namespace ia2c {
namespace {

constexpr uint32_t kStreamPbt = 5;
constexpr int kRankThreads = 256;
constexpr int kCopyThreads = 256;
constexpr int kAgentsPerBlock = 8;   // ~29 KB of rows per block (3.6 KB per agent at M = 5)
constexpr int kBuffers = 10;

struct RankArgs {
    const double* ring;                   // return_sum f64[capacity, R]
    int32_t capacity, slot, window, R;
    const double *lr_actor, *lr_critic;
    const float *gamma, *beta;
    int32_t* order;                       // workspace i32[R]
    double* log_fitness;
    int32_t *log_rank, *log_donor;
    double *log_lr_actor, *log_lr_critic;
    float *log_gamma, *log_beta;
};

// The fixed-order fitness of run r: window ring rows, oldest first, one fp64 add each from +0.0.
__device__ __forceinline__ double run_fitness(const RankArgs& a, int r) {
    int s = a.slot - a.window + 1;
    if (s < 0) s += a.capacity;
    double f = 0.0;
    for (int k = 0; k < a.window; ++k) {
        f = __dadd_rn(f, __ldcg(a.ring + (int64_t)s * a.R + r));
        if (++s == a.capacity) s = 0;
    }
    return f;
}

// Does (fa, ia) come before (fb, ib)?  Higher fitness first, NaN last, ties to the lower run index.
__device__ __forceinline__ bool ranks_before(double fa, int ia, double fb, int ib) {
    const bool na = isnan(fa), nb = isnan(fb);
    if (na != nb) return nb;
    if (!na && fa != fb) return fa > fb;
    return ia < ib;
}

__global__ void __launch_bounds__(kRankThreads) pbt_rank_kernel(const __grid_constant__ RankArgs a) {
    __shared__ double tile[kRankThreads];
    pdl_prologue();
    const int tid = threadIdx.x, base = blockIdx.x * kRankThreads, r = base + tid;
    const double f = r < a.R ? run_fitness(a, r) : 0.0;
    int before = 0;   // runs that rank before r
    for (int t0 = 0; t0 < a.R; t0 += kRankThreads) {
        const int j = t0 + tid;
        tile[tid] = t0 == base ? f : (j < a.R ? run_fitness(a, j) : 0.0);
        __syncthreads();
        const int n = min(kRankThreads, a.R - t0);
        if (r < a.R)
            for (int k = 0; k < n; ++k) before += ranks_before(tile[k], t0 + k, f, r);
        __syncthreads();
    }
    if (r >= a.R) return;
    a.order[before] = r;
    a.log_fitness[r] = f;
    a.log_rank[r] = before;
    a.log_donor[r] = -1;
    a.log_lr_actor[r] = __ldcg(a.lr_actor + r);
    a.log_lr_critic[r] = __ldcg(a.lr_critic + r);
    a.log_gamma[r] = __ldcg(a.gamma + r);
    a.log_beta[r] = __ldcg(a.beta + r);
}

struct ApplyArgs {
    uint32_t* buf[kBuffers];              // the ten per-net buffers, R*N rows each
    int32_t row_words[kBuffers];          // 4-byte words per row
    const int32_t* order;
    int32_t R, N, q;
    uint32_t perturb, generation;
    double factor_lo, factor_hi;
    uint64_t seed;
    double *lr_actor, *lr_critic;
    float *gamma, *beta;
    int32_t* log_donor;
    double *log_lr_actor, *log_lr_critic;
    float *log_gamma, *log_beta;
};

// n words from src to dst by the block: 16-byte loads and stores where both share their alignment mod 16, else 4-byte words.
__device__ __forceinline__ void copy_words(const uint32_t* src, uint32_t* dst, int64_t n) {
    const int tid = threadIdx.x;
    int64_t head = n;
    if (((reinterpret_cast<uintptr_t>(src) ^ reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
        head = min(n, (int64_t)(((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15) >> 2));
        const int64_t vecs = (n - head) >> 2;
        const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
        uint4* d4 = reinterpret_cast<uint4*>(dst + head);
        for (int64_t i = tid; i < vecs; i += kCopyThreads) d4[i] = __ldcg(s4 + i);
        for (int64_t i = head + (vecs << 2) + tid; i < n; i += kCopyThreads) dst[i] = __ldcg(src + i);
    }
    for (int64_t i = tid; i < head; i += kCopyThreads) dst[i] = __ldcg(src + i);
}

__global__ void __launch_bounds__(kCopyThreads) pbt_apply_kernel(const __grid_constant__ ApplyArgs a) {
    // No early release: the next episode's kernels stage the agents' models (filter_action) before their griddepcontrol.wait,
    // and this kernel writes them.  Without launch_dependents the successor starts only once every copy has completed.
    pdl_wait();
    if ((int)blockIdx.x >= a.q) return;   // q = 0: the one block of the launch has no recipient
    const int v = __ldcg(a.order + a.R - a.q + blockIdx.x);
    const uint4 w = philox_draw(a.seed, kStreamPbt, a.generation, 0u, (uint64_t)v);
    const int donor = __ldcg(a.order + (int)(((uint64_t)(w.x >> 8) * (uint64_t)a.q) >> 24));
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        double lra = __ldcg(a.lr_actor + donor), lrc = __ldcg(a.lr_critic + donor);
        float beta = __ldcg(a.beta + donor);
        const float gamma = __ldcg(a.gamma + donor);
        if (a.perturb & IA2C_PBT_LR_ACTOR) lra = __dmul_rn(lra, (w.y >> 31) ? a.factor_hi : a.factor_lo);
        if (a.perturb & IA2C_PBT_LR_CRITIC) lrc = __dmul_rn(lrc, (w.z >> 31) ? a.factor_hi : a.factor_lo);
        if (a.perturb & IA2C_PBT_BETA) beta = __double2float_rn(__dmul_rn((double)beta, (w.w >> 31) ? a.factor_hi : a.factor_lo));
        a.lr_actor[v] = lra, a.lr_critic[v] = lrc, a.gamma[v] = gamma, a.beta[v] = beta;
        a.log_donor[v] = donor;
        a.log_lr_actor[v] = lra, a.log_lr_critic[v] = lrc, a.log_gamma[v] = gamma, a.log_beta[v] = beta;
    }
    const int a0 = blockIdx.y * kAgentsPerBlock, na = min(kAgentsPerBlock, a.N - a0);
#pragma unroll 1
    for (int b = 0; b < kBuffers; ++b) {
        const int64_t rw = a.row_words[b];
        copy_words(a.buf[b] + ((int64_t)donor * a.N + a0) * rw, a.buf[b] + ((int64_t)v * a.N + a0) * rw, na * rw);
    }
}

bool positive_finite(double x) { return std::isfinite(x) && x > 0.0; }

int validate_pbt(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_history_desc* h, const ia2c_pbt_desc* p) {
    const char* who = "ia2c_pbt_step";
    IA2C_REQUIRE(d && r && h && p, "%s: null episode, runs, history or pbt descriptor", who);
    IA2C_REQUIRE(d->actor_params && d->critic_params && d->actor_m && d->actor_v && d->critic_m && d->critic_v && d->actor_step &&
                     d->critic_step && d->actor_grad_accum && d->filter_action,
                 "%s: null per-net buffer (actor_params, critic_params, Adam moments and steps, actor_grad_accum, filter_action)",
                 who);
    IA2C_REQUIRE(h->return_sum, "%s: null return_sum ring", who);
    IA2C_REQUIRE(p->lr_actor && p->lr_critic && p->gamma && p->beta, "%s: null hyper-parameter array (all four are required)", who);
    IA2C_REQUIRE(p->log_fitness && p->log_rank && p->log_donor && p->log_lr_actor && p->log_lr_critic && p->log_gamma && p->log_beta,
                 "%s: null log array", who);
    IA2C_REQUIRE(p->workspace, "%s: null workspace", who);
    const int32_t R = r->runs;
    IA2C_REQUIRE(R >= 1, "%s: runs=%d must be >= 1", who, R);
    IA2C_REQUIRE(d->N >= 1 && d->M >= 1, "%s: N=%d and M=%d must be >= 1", who, d->N, d->M);
    IA2C_REQUIRE((int64_t)R * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS (%d)", who,
                 (long long)R * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(h->capacity >= 2, "%s: capacity=%d must be >= 2", who, h->capacity);
    IA2C_REQUIRE(p->window >= 1 && p->window <= h->capacity - 1, "%s: window=%d outside [1, capacity - 1 = %d]", who, p->window,
                 h->capacity - 1);
    IA2C_REQUIRE(p->slot >= 0 && p->slot < h->capacity, "%s: slot=%d outside [0, capacity=%d)", who, p->slot, h->capacity);
    IA2C_REQUIRE(p->q >= 0 && 2 * (int64_t)p->q <= R, "%s: q=%d must satisfy 0 <= 2q <= runs=%d", who, p->q, R);
    IA2C_REQUIRE((p->perturb & ~(uint32_t)(IA2C_PBT_LR_ACTOR | IA2C_PBT_LR_CRITIC | IA2C_PBT_BETA)) == 0,
                 "%s: perturb=0x%x has bits other than lr_actor, lr_critic and beta", who, p->perturb);
    IA2C_REQUIRE(positive_finite(p->factor_lo) && positive_finite(p->factor_hi), "%s: factors (%g, %g) must be finite and > 0",
                 who, p->factor_lo, p->factor_hi);
    IA2C_REQUIRE(p->workspace_bytes >= ia2c_pbt_workspace_bytes(R), "%s: workspace of %zu bytes below ia2c_pbt_workspace_bytes = %zu",
                 who, p->workspace_bytes, ia2c_pbt_workspace_bytes(R));
    if (d->env_offset != 0 || d->E_total != d->E) {
        set_error("%s: env_offset=%lld, E_total=%lld, E=%lld: PBT runs on one GPU (env_offset 0, E_total = E)", who,
                  (long long)d->env_offset, (long long)d->E_total, (long long)d->E);
        return IA2C_ERR_UNSUPPORTED;
    }
    return 0;
}

}  // namespace
}  // namespace ia2c

using namespace ia2c;

extern "C" size_t ia2c_pbt_workspace_bytes(int32_t runs) { return runs > 0 ? (size_t)runs * sizeof(int32_t) : 0; }

extern "C" int ia2c_pbt_step(const ia2c_episode_desc* d, const ia2c_runs_desc* r, const ia2c_history_desc* h,
                             const ia2c_pbt_desc* p, void* stream) {
    if (int rc = validate_pbt(d, r, h, p)) return rc;
    const cudaStream_t s = as_stream(stream);
    const int32_t R = r->runs, N = d->N;
    int32_t* order = static_cast<int32_t*>(p->workspace);

    RankArgs ra;
    ra.ring = h->return_sum, ra.capacity = h->capacity, ra.slot = p->slot, ra.window = p->window, ra.R = R;
    ra.lr_actor = p->lr_actor, ra.lr_critic = p->lr_critic, ra.gamma = p->gamma, ra.beta = p->beta;
    ra.order = order;
    ra.log_fitness = p->log_fitness, ra.log_rank = p->log_rank, ra.log_donor = p->log_donor;
    ra.log_lr_actor = p->log_lr_actor, ra.log_lr_critic = p->log_lr_critic, ra.log_gamma = p->log_gamma, ra.log_beta = p->log_beta;
    if (int rc = launch_pdl("pbt_rank_kernel", pbt_rank_kernel, dim3((unsigned)ceil_div(R, kRankThreads)), dim3(kRankThreads), 0, s,
                            ra))
        return rc;

    ApplyArgs aa;
    const void* const bufs[kBuffers] = {d->actor_params, d->critic_params, d->actor_m,     d->actor_v,          d->critic_m,
                                        d->critic_v,     d->actor_step,    d->critic_step, d->actor_grad_accum, d->filter_action};
    const int32_t words[kBuffers] = {kActorP, kCriticP, kActorP, kActorP, kCriticP, kCriticP, 1, 1, kActorP,
                                     d->M * IA2C_AGENT_ACTIONS * 2};   // filter_action: f64[M, 3] per net
    for (int b = 0; b < kBuffers; ++b) aa.buf[b] = static_cast<uint32_t*>(const_cast<void*>(bufs[b])), aa.row_words[b] = words[b];
    aa.order = order, aa.R = R, aa.N = N, aa.q = p->q;
    aa.perturb = p->perturb, aa.generation = p->generation, aa.factor_lo = p->factor_lo, aa.factor_hi = p->factor_hi;
    aa.seed = p->seed;
    aa.lr_actor = p->lr_actor, aa.lr_critic = p->lr_critic, aa.gamma = p->gamma, aa.beta = p->beta;
    aa.log_donor = p->log_donor;
    aa.log_lr_actor = p->log_lr_actor, aa.log_lr_critic = p->log_lr_critic, aa.log_gamma = p->log_gamma, aa.log_beta = p->log_beta;
    // q = 0 still launches (one block that returns): two launches per generation whatever q is
    const dim3 grid((unsigned)(p->q > 0 ? p->q : 1), (unsigned)(p->q > 0 ? ceil_div(N, kAgentsPerBlock) : 1));
    return launch_pdl("pbt_apply_kernel", pbt_apply_kernel, grid, dim3(kCopyThreads), 0, s, aa);
}
