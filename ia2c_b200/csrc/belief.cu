// belief.cu — Bayesian belief filter over the other agents' candidate models.
//
// Replaces BeliefFilter.update (belief_filter_deprecated.py:45-59) and noisy_private_obs
// (ia2c.py:53-58).  All arithmetic is fp64 with explicit round-to-nearest intrinsics so that ptxas
// cannot contract mul+add: the posterior is rounded to 2 decimals before it becomes the next prior
// (belief_filter_deprecated.py:58), so a single flipped rounding is a 0.01 error (SURVEY.md §7.3).
// Operation order per row (SURVEY.md Appendix A.2):
//   t[a][m] = Fm[m][a]*prev[m];  bp[m] = (lik0*t0 + lik1*t1) + lik2*t2 ...;  S = ((bp0+bp1)+bp2)+...
//   b[m] = bp[m]/S;  pred[a] = sum_m b[m]*Fm[m][a];  ap = first a with u < cumsum(pred), none -> 0
//   out[m] = rint(b[m]*100)/100
//
// Two layouts:
//   dense  — the reference's fp64 [R,M]/[R,A] arrays (class API, 88 B per update at M=5,A=3);
//   pairs  — the trainer's packed records: posteriors are k/100 with integer k, stored as uint8
//            (lossless), 8 B per (env, agent, modelled other); likelihood synthesised from the other
//            agent's action; stages the models, actions and a k/100 table in shared memory and
//            reduces the predicted actions per agent (mode) with shared-memory counters.
#include <algorithm>

#include "common.cuh"

namespace ia2c {
int belief_pairs_episode_runs_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, cudaStream_t s);   // trainer.cu
int belief_pairs_episode_seats_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, const TrainedSeats& f, cudaStream_t s);
namespace {

constexpr int kThreads = 256;
constexpr int kMaxDense = 8;

// Core update with compile-time M, A.  fa is [M][A] (row = model).
template <int M, int A>
__device__ __forceinline__ int belief_core(const double* __restrict__ fa, const double (&lik)[A],
                                           const double (&prev)[M], double u, double (&b)[M], double (&pred)[A]) {
    double bp[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        double acc = __dmul_rn(lik[0], __dmul_rn(fa[m * A + 0], prev[m]));
#pragma unroll
        for (int a = 1; a < A; ++a) acc = __dadd_rn(acc, __dmul_rn(lik[a], __dmul_rn(fa[m * A + a], prev[m])));
        bp[m] = acc;
    }
    double S = bp[0];
#pragma unroll
    for (int m = 1; m < M; ++m) S = __dadd_rn(S, bp[m]);
    const double rS = drcp_seq(S);   // one refined reciprocal shared by the M divisions (common.cuh)
#pragma unroll
    for (int m = 0; m < M; ++m) b[m] = ddiv_with(bp[m], S, rS);
#pragma unroll
    for (int a = 0; a < A; ++a) {
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < M; ++m) acc = __dadd_rn(acc, __dmul_rn(b[m], fa[m * A + a]));
        pred[a] = acc;
    }
    double c = pred[0];
    int ap = 0;
    bool found = u < c;
#pragma unroll
    for (int a = 1; a < A; ++a) {
        c = __dadd_rn(c, pred[a]);
        if (!found && u < c) {
            ap = a;
            found = true;
        }
    }
    return ap;  // falls through to 0 when u >= cumsum[-1] (SURVEY.md Q11)
}

template <int M, int A>
__global__ void __launch_bounds__(kThreads)
belief_dense_kernel(const double* __restrict__ filter_action, const double* __restrict__ lik_in,
                    const double* __restrict__ prev_in, const double* __restrict__ u_in, int64_t* __restrict__ ap_out,
                    double* __restrict__ bprime_out, double* __restrict__ pred_out, int64_t R) {
    __shared__ double fa[M * A];
    for (int i = threadIdx.x; i < M * A; i += blockDim.x) fa[i] = filter_action[i];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (r >= R) return;
    double lik[A], prev[M], b[M], pred[A];
#pragma unroll
    for (int a = 0; a < A; ++a) lik[a] = lik_in[r * A + a];
#pragma unroll
    for (int m = 0; m < M; ++m) prev[m] = prev_in[r * M + m];
    const int ap = belief_core<M, A>(fa, lik, prev, u_in[r], b, pred);
    ap_out[r] = ap;
#pragma unroll
    for (int m = 0; m < M; ++m) bprime_out[r * M + m] = ddiv_seq(rint(__dmul_rn(b[m], 100.0)), 100.0);
    if (pred_out) {
#pragma unroll
        for (int a = 0; a < A; ++a) pred_out[r * A + a] = pred[a];
    }
}

#ifndef IA2C_BELIEF_SEATS   // the non-template kernels: in belief.cu only
// Runtime-dimension fallback (M, A <= 8), same operation order.
__global__ void __launch_bounds__(kThreads)
belief_dense_generic_kernel(const double* __restrict__ filter_action, const double* __restrict__ lik_in,
                            const double* __restrict__ prev_in, const double* __restrict__ u_in,
                            int64_t* __restrict__ ap_out, double* __restrict__ bprime_out,
                            double* __restrict__ pred_out, int64_t R, int M, int A) {
    __shared__ double fa[kMaxDense * kMaxDense];
    for (int i = threadIdx.x; i < M * A; i += blockDim.x) fa[i] = filter_action[i];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (r >= R) return;
    double bp[kMaxDense], b[kMaxDense];
    double S = 0.0;
    for (int m = 0; m < M; ++m) {
        const double p = prev_in[r * M + m];
        double acc = __dmul_rn(lik_in[r * A], __dmul_rn(fa[m * A], p));
        for (int a = 1; a < A; ++a) acc = __dadd_rn(acc, __dmul_rn(lik_in[r * A + a], __dmul_rn(fa[m * A + a], p)));
        bp[m] = acc;
        S = (m == 0) ? acc : __dadd_rn(S, acc);
    }
    for (int m = 0; m < M; ++m) {
        b[m] = ddiv_seq(bp[m], S);
        bprime_out[r * M + m] = ddiv_seq(rint(__dmul_rn(b[m], 100.0)), 100.0);
    }
    const double u = u_in[r];
    double c = 0.0;
    int ap = 0;
    bool found = false;
    for (int a = 0; a < A; ++a) {
        double acc = 0.0;
        for (int m = 0; m < M; ++m) acc = __dadd_rn(acc, __dmul_rn(b[m], fa[m * A + a]));
        if (pred_out) pred_out[r * A + a] = acc;
        c = (a == 0) ? acc : __dadd_rn(c, acc);
        if (!found && u < c) {
            ap = a;
            found = true;
        }
    }
    ap_out[r] = ap;
}
#endif

// ------------------------------------------------------------------------------------------------
// Packed pairwise update.  A block owns `n_envs` whole envs (small N*K) or one env's agent chunk
// [i0, i1) (large N*K); within the block consecutive threads take consecutive records (coalesced
// 8-byte loads/stores).
struct PairsArgs {
    uint8_t* records;
    const double* filter_action;   // [N,M,3]
    const uint8_t* actions;        // [E,N]
    const double* u_injected;      // [E,N,K] or null
    uint8_t* pred_out;             // [E,N,K] or null
    uint8_t* belief_out;           // [E,N,K,M] or null
    uint8_t* pred_partner_out;     // [E,N] or null
    int64_t E, env_offset;
    int N, K, envs_per_block, agents_per_block, chunks_per_env, reset_prior;
    uint64_t seed;
    uint32_t episode, t;
    uint32_t stage_offset;         // byte offset of the cp.async staging ring in dynamic shared memory (table kernel)
    uint32_t rk[20];               // Philox round keys (k0_r, k1_r), r = 0..9 — derived from seed on the host so that the
                                   // rounds read them straight from the constant bank (table kernel)
};

template <int M>
__global__ void __launch_bounds__(kThreads) belief_pairs_kernel(PairsArgs P) {
    constexpr int A = IA2C_AGENT_ACTIONS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = P.N, K = P.K;
    const int64_t e0 = (int64_t)(blockIdx.x / P.chunks_per_env) * P.envs_per_block;
    const int chunk = blockIdx.x % P.chunks_per_env;
    const int i0 = chunk * P.agents_per_block;
    const int i1 = min(N, i0 + P.agents_per_block);
    const int n_agents = i1 - i0;
    const int n_envs = (int)min((int64_t)P.envs_per_block, P.E - e0);

    pdl_prologue();
    double* tab = reinterpret_cast<double*>(smem_raw);             // [101] k/100
    double* fa = tab + 104;                                        // [n_agents][M*A]
    int* counts = reinterpret_cast<int*>(fa + P.agents_per_block * M * A);   // [envs_per_block][agents_per_block][A]
    uint8_t* act = reinterpret_cast<uint8_t*>(counts + P.envs_per_block * P.agents_per_block * A);  // [envs_per_block][N]

    for (int k = threadIdx.x; k <= 100; k += blockDim.x) tab[k] = __ddiv_rn((double)k, 100.0);
    for (int i = threadIdx.x; i < n_agents * M * A; i += blockDim.x) fa[i] = P.filter_action[(int64_t)i0 * M * A + i];
    for (int i = threadIdx.x; i < n_envs * n_agents * A; i += blockDim.x) counts[i] = 0;
    for (int i = threadIdx.x; i < n_envs * N; i += blockDim.x) act[i] = P.actions[e0 * N + i];
    __syncthreads();

    const int prior_k = (int)rint(100.0 * (rint(100.0 / M) / 100.0));  // round(1/M, 2) in hundredths
    const int per_env = n_agents * K;
    const int total = n_envs * per_env;
    for (int q = threadIdx.x; q < total; q += blockDim.x) {
        const int el = q / per_env;
        const int rem = q - el * per_env;
        const int il = rem / K;          // local agent
        const int jj = rem - il * K;     // modelled-other slot
        const int i = i0 + il;
        const int j = jj + (jj >= i);    // others in ascending order, skipping i
        const int64_t e = e0 + el;
        const int64_t rec = ((e * N + i) * (int64_t)K + jj);
        uint2 raw = make_uint2(0u, 0u);
        if (!P.reset_prior) raw = *reinterpret_cast<const uint2*>(P.records + rec * IA2C_BELIEF_RECORD);
        double prev[M];
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const uint32_t word = m < 4 ? raw.x : raw.y;
            const int k = P.reset_prior ? prior_k : (int)((word >> (8 * (m & 3))) & 0xFFu);
            prev[m] = tab[k];
        }
        const int seen = act[el * N + j];
        double lik[A];
#pragma unroll
        for (int a = 0; a < A; ++a) lik[a] = (a == seen) ? 0.8 : 0.1;   // ia2c.py:53-58
        const double u = P.u_injected ? P.u_injected[rec]
                                      : philox_belief_uniform(P.seed, P.episode, P.t, (uint64_t)((P.env_offset + e) * N + i), K, jj);
        double b[M], pred[A];
        const int ap = belief_core<M, A>(fa + il * M * A, lik, prev, u, b, pred);
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const uint32_t k = (uint32_t)__double2int_rn(__dmul_rn(b[m], 100.0));  // rint, half-to-even
            if (m < 4) lo |= k << (8 * m); else hi |= k << (8 * (m - 4));
            if (P.belief_out) P.belief_out[rec * M + m] = (uint8_t)k;
        }
        hi |= (uint32_t)ap << 16;  // byte 6
        *reinterpret_cast<uint2*>(P.records + rec * IA2C_BELIEF_RECORD) = make_uint2(lo, hi);
        if (P.pred_out) P.pred_out[rec] = (uint8_t)ap;
        if (P.pred_partner_out) atomicAdd(&counts[(el * n_agents + il) * A + ap], 1);
    }
    if (P.pred_partner_out) {
        __syncthreads();
        for (int x = threadIdx.x; x < n_envs * n_agents; x += blockDim.x) {
            const int el = x / n_agents, il = x - el * n_agents;
            const int* c = counts + x * A;
            int best = 0;
#pragma unroll
            for (int a = 1; a < A; ++a) best = c[a] > c[best] ? a : best;   // ties -> lowest action
            P.pred_partner_out[(e0 + el) * N + i0 + il] = (uint8_t)best;
        }
    }
}

#ifndef IA2C_BELIEF_SEATS
__global__ void debug_divide_kernel(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ q_seq,
                                    double* __restrict__ q_ieee, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    q_seq[i] = ddiv_seq(a[i], b[i]);
    q_ieee[i] = __ddiv_rn(a[i], b[i]);
}
#endif

// ------------------------------------------------------------------------------------------------
// Table-driven pairwise update for many modelled others (K >= 32).
//
// belief_pairs_kernel costs ~100 fp64 instructions per record against 16 B of traffic.  This kernel keeps every
// output bit and spends ~1/3 of the instructions, none of them fp64 on the common path:
//  (1) the un-normalised posterior bp[m] = (l0*(F[m][0]*p) + l1*(F[m][1]*p)) + l2*(F[m][2]*p) depends only on the
//      agent's model m, the SEEN action (3 likelihood rows) and the prior, which is k/100 with integer k in 0..100.
//      A block that owns ONE agent tabulates all 3*M*101 values once in fp64 (same operations, same order as
//      belief_core) and keeps an fp32 copy of the table;
//  (2) the stored posterior is rint(100 * bp[m]/S) and the predicted action is a comparison of u with the cumulative
//      mixture — both are DECISIONS, so they are first taken in fp32 (table lookups, one MUFU.RCP, FFMA) together with
//      a rigorous distance-to-the-boundary test: the fp32 quotient 100*bp/S is within 6e-5 of the fp64 value
//      (10 roundings of 2^-24 relative on a value <= 100), so a rounding is accepted only when it is more than 1e-4
//      away from a half-integer; the inverse-CDF comparison u*S < sum_m bp[m]*Fcum[m][a] is accepted only when the
//      two sides differ by more than 1e-5*S (their fp32 errors are below 1e-6*S each);
//  (3) a record that fails either test (~0.1 % of them) is recomputed with the exact fp64 sequence of belief_core on
//      the fp64 table (same operands, same order, IEEE division) — bit-identical to belief_pairs_kernel and to the
//      oracle by construction, and checked against both by tests/test_gpu_belief.py.
// Thread = the FOUR modelled-other slots 4s..4s+3 of one (env, agent): they share one Philox block (common.cuh:
// philox_belief_quad) and give the scheduler four independent chains; the agent's K records of one env are 8*K
// contiguous bytes.  The per-agent predicted-action counts are packed 3 x 10 bits and reduced with one warp REDUX +
// one shared-memory atomic per (warp, env) instead of one atomic per record.
// FAST = the steady-state call of the rollout (device Philox, no dumps, priors from the records): the optional
// pointers are compiled out instead of costing a predicated-off instruction each per record.
constexpr float kRoundMagic = 12582912.f;       // 1.5 * 2^23: x + magic has rint(x) in its low mantissa bits
// Rounding screen: x32 = bp32 * (rcp.approx(S32) * 100) differs from the real 100*bp/S by at most 10 * 2^-24 relative (table entry
// 1, M - 1 <= five fp32 adds + their inputs 6, rcp.approx 2, the *100 1 — units of 2^-24), i.e. 6.0e-5 at x = 100; the window is 1.7 x that.
constexpr float kHalfWindow = 0.5f - 1.0e-4f;    // |100*b - rint(100*b)| above this -> exact path
constexpr float kCdfWindow = 1e-5f;              // |u*S - cumulative| below this * S -> exact path

template <int M>
struct TableView {
    const double* bpt;     // [A][M][101] fp64 un-normalised posteriors
    const float* bpt32;    // the same in fp32
    const double* fa;      // [M][A]
};

// exact fp64 sequence (belief_core on the table): -> the packed record {posterior hundredths, predicted action in byte 6}
template <int M>
__device__ __noinline__ uint2 belief_exact_record(const double* __restrict__ row, const double* __restrict__ fa, uint2 raw, int prior_k,
                                                  double u) {
    constexpr int A = IA2C_AGENT_ACTIONS;
    double bp[M], b[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const uint32_t word = m < 4 ? raw.x : raw.y;
        const int k = prior_k >= 0 ? prior_k : (int)((word >> (8 * (m & 3))) & 0xFFu);
        bp[m] = row[m * 101 + k];
    }
    double S = bp[0];
#pragma unroll
    for (int m = 1; m < M; ++m) S = __dadd_rn(S, bp[m]);
    const double rS = drcp_seq(S);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        b[m] = ddiv_with(bp[m], S, rS);
        const uint32_t k = (uint32_t)__double2int_rn(__dmul_rn(b[m], 100.0));
        if (m < 4) lo |= k << (8 * m); else hi |= k << (8 * (m - 4));
    }
    double c = 0.0;
    int ap = 0;
    bool found = false;
#pragma unroll
    for (int a = 0; a < A; ++a) {
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < M; ++m) acc = __dadd_rn(acc, __dmul_rn(b[m], fa[m * A + a]));
        c = (a == 0) ? acc : __dadd_rn(c, acc);
        if (!found && u < c) { ap = a; found = true; }
    }
    return make_uint2(lo, hi | ((uint32_t)ap << 16));
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

// Second-level rounding screen of ONE record, run by the rare lanes whose first-level test (constant window kHalfWindow)
// fired: the same fp32 quantities, but every value is tested against its OWN error bound — x32 is within 10 * 2^-24 * x of the
// real quotient, so a rounding is safe when |x32 - rint(x32)| < 0.5 - 1e-6 * (rint(x32) + 1) (1.7 x the bound).  Cuts the
// records that reach the fp64 sequence by ~5x.  -> true when the record still needs the exact path.
template <int M>
__device__ __noinline__ bool belief_refine_rounding(uint32_t row_s, uint2 raw) {
    float bp[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const uint32_t k = ((m < 4 ? raw.x : raw.y) >> (8 * (m & 3))) & 0xFFu;
        bp[m] = lds_f32(row_s + 4u * k + (uint32_t)(m * 101 * 4));
    }
    float S = bp[0];
#pragma unroll
    for (int m = 1; m < M; ++m) S = __fadd_rn(S, bp[m]);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(S));
    const float r100 = __fmul_rn(r, 100.f);
    bool exact = false;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const float kf = __fmaf_rn(bp[m], r100, kRoundMagic);
        const float nk = __fsub_rn(kRoundMagic, kf);                  // -rint(x32)
        const float d = __fmaf_rn(bp[m], r100, nk);
        exact |= fabsf(d) > __fmaf_rn(nk, 1e-6f, 0.5f - 1e-6f);      // 0.5 - 1e-6 * (rint + 1)
    }
    return exact;
}

// Philox4x32-10 with precomputed round keys (identical to philox4x32_10: key_r = key_0 + r * W)
__device__ __forceinline__ uint4 philox4x32_10_rk(uint4 c, const uint32_t (&rk)[20]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ rk[2 * r], lo1, hi0 ^ c.w ^ rk[2 * r + 1], lo0);
    }
    return c;
}

constexpr int kExactQueue = 1024;   // deferred exact-path records per block (expected ~0.25 % of <= 32640; overflow -> inline)

template <int M, bool FAST>
__global__ void __launch_bounds__(kThreads, 2) belief_pairs_table_kernel(const __grid_constant__ PairsArgs P) {
    constexpr int A = IA2C_AGENT_ACTIONS;
    const bool reset_prior = !FAST && P.reset_prior;
    const double* const u_injected = FAST ? nullptr : P.u_injected;
    uint8_t* const belief_out = FAST ? nullptr : P.belief_out;
    uint8_t* const pred_out = FAST ? nullptr : P.pred_out;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int queue_n;
    const int N = P.N, K = P.K, i = blockIdx.y;
    const int KQ = (K + 3) >> 2;                                     // quads per (env, agent); K padded to whole quads
    const int EC = P.envs_per_block;
    const int64_t e0 = (int64_t)blockIdx.x * EC;
    const int n_envs = (int)min((int64_t)EC, P.E - e0);
    double* tab = reinterpret_cast<double*>(smem_raw);               // [104]   k/100
    double* bpt = tab + 104;                                         // [A][M][101]
    double* fa = bpt + A * M * 101;                                  // [M][A]
    float* bpt32 = reinterpret_cast<float*>(fa + M * A);             // [A][M][101]
    float* fcum = bpt32 + ((A * M * 101 + 3) & ~3);                  // [2][M]: F[m][0], F[m][0]+F[m][1]
    uint32_t* counts = reinterpret_cast<uint32_t*>(fcum + ((2 * M + 3) & ~3));   // [EC] packed 3 x 10 bits
    uint16_t* queue = reinterpret_cast<uint16_t*>(counts + EC);      // [kExactQueue] deferred records: 4 * quad + slot
    uint32_t* seen4 = reinterpret_cast<uint32_t*>(queue + kExactQueue);   // [EC][KQ]: the OTHERS' actions, 4 slots per word
    unsigned char* stage = smem_raw + P.stage_offset;               // [kStages][kThreads][32 B] cp.async ring (16-byte aligned)
    pdl_release();
    // the table depends only on the agent's models: it is built while the kernel that samples this step's actions
    // may still be running (programmatic dependent launch); pdl_wait() below orders the reads of its output
    for (int k = threadIdx.x; k <= 100; k += blockDim.x) tab[k] = __ddiv_rn((double)k, 100.0);
    for (int k = threadIdx.x; k < M * A; k += blockDim.x) fa[k] = P.filter_action[(int64_t)i * M * A + k];
    for (int k = threadIdx.x; k < n_envs; k += blockDim.x) counts[k] = 0u;
    if (threadIdx.x == 0) queue_n = 0;
    __syncthreads();
    for (int x = threadIdx.x; x < A * M * 101; x += blockDim.x) {
        const int seen = x / (M * 101), m = (x / 101) % M, k = x % 101;
        const double p = tab[k];
        double acc = __dmul_rn(seen == 0 ? 0.8 : 0.1, __dmul_rn(fa[m * A + 0], p));
#pragma unroll
        for (int a = 1; a < A; ++a) acc = __dadd_rn(acc, __dmul_rn(seen == a ? 0.8 : 0.1, __dmul_rn(fa[m * A + a], p)));
        bpt[x] = acc;
        bpt32[x] = (float)acc;
    }
    if (threadIdx.x < M) {
        fcum[threadIdx.x] = (float)fa[threadIdx.x * A];
        fcum[M + threadIdx.x] = (float)__dadd_rn(fa[threadIdx.x * A], fa[threadIdx.x * A + 1]);
    }
    pdl_wait();
    // the others' actions of every env of the block, own action skipped, padded to whole quads: slot jj of env el is
    // byte jj of word el*KQ + jj/4, so a thread's four slots are ONE 32-bit shared load.  Word w of a row is the source
    // word w (slots below i), the source bytes 4w+1..4w+4 (slots above i), or a mix (the word that contains i).
    if ((N & 3) == 0) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(P.actions + e0 * N);   // rows are 4-byte aligned (N % 4 == 0)
        const int NW = N >> 2, iw = i >> 2;
        const uint32_t sel_mix = (i & 3) == 0 ? 0x4321u : ((i & 3) == 1 ? 0x4320u : ((i & 3) == 2 ? 0x4310u : 0x4210u));
        const int words = n_envs * KQ;
        // (env, word) of the thread's next item, advanced without divisions; eight items' loads in flight at a time
        const int s_el = (int)blockDim.x / KQ, s_w = (int)blockDim.x % KQ;
        int el = (int)threadIdx.x / KQ, w = (int)threadIdx.x % KQ;
        constexpr int kBatch = 8;
        for (int x0 = threadIdx.x; x0 < words; x0 += kBatch * blockDim.x) {
            uint32_t lo[kBatch], hi[kBatch];
            int ww[kBatch];
#pragma unroll
            for (int b = 0; b < kBatch; ++b) {
                const bool ok = x0 + b * (int)blockDim.x < words;
                ww[b] = w;
                lo[b] = ok ? __ldcg(src + el * NW + w) : 0u;
                hi[b] = (ok && w + 1 < NW) ? __ldcg(src + el * NW + w + 1) : 0u;
                el += s_el; w += s_w;
                if (w >= KQ) { w -= KQ; ++el; }
            }
#pragma unroll
            for (int b = 0; b < kBatch; ++b) {
                const int x = x0 + b * (int)blockDim.x;
                if (x < words) {
                    uint32_t v = __byte_perm(lo[b], hi[b], ww[b] < iw ? 0x3210u : (ww[b] > iw ? 0x4321u : sel_mix));
                    if (4 * ww[b] + 3 >= K) v &= 0xFFFFFFFFu >> (8 * (4 * ww[b] + 4 - K));      // zero the padding slots
                    seen4[x] = v;
                }
            }
        }
    } else {
        uint8_t* seen_b = reinterpret_cast<uint8_t*>(seen4);
        const int KP = 4 * KQ;
        for (int x = threadIdx.x; x < n_envs * KP; x += blockDim.x) {
            const int el = x / KP, jj = x - el * KP;
            seen_b[x] = jj < K ? P.actions[(e0 + el) * N + jj + (jj >= i)] : (uint8_t)0;
        }
    }
    __syncthreads();
    const int prior_k = reset_prior ? (int)rint(100.0 / M) : -1;
    float f0[M], f01[M];
#pragma unroll
    for (int m = 0; m < M; ++m) { f0[m] = fcum[m]; f01[m] = fcum[M + m]; }
    const uint32_t bpt32_s = (uint32_t)__cvta_generic_to_shared(bpt32);   // explicit shared-window addresses for the lookups

    // fp32 screen of TWO records at once (packed f32x2 arithmetic: one issue slot per pair of FMAs) -> the packed records
    // {posterior hundredths, predicted action in byte 6}; bit w of the result is set when record w's rounding or its
    // inverse-CDF decision is too close to call in fp32
    const float2 magic2 = make_float2(kRoundMagic, kRoundMagic), minus1 = make_float2(-1.f, -1.f);
    auto screen_pair = [&](uint32_t seenA, uint32_t seenB, float ufA, float ufB, uint2 rawA, uint2 rawB, uint2& outA, uint2& outB) -> uint32_t {
        const uint32_t rowA = bpt32_s + seenA * (M * 101 * 4), rowB = bpt32_s + seenB * (M * 101 * 4);
        float2 bp[M];
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const uint32_t sel = 0x4440u | (uint32_t)(m & 3);
            const uint32_t kA = reset_prior ? (uint32_t)prior_k : __byte_perm(m < 4 ? rawA.x : rawA.y, 0u, sel);
            const uint32_t kB = reset_prior ? (uint32_t)prior_k : __byte_perm(m < 4 ? rawB.x : rawB.y, 0u, sel);
            bp[m] = make_float2(lds_f32(rowA + 4u * kA + (uint32_t)(m * 101 * 4)), lds_f32(rowB + 4u * kB + (uint32_t)(m * 101 * 4)));
        }
        float2 S = bp[0];
#pragma unroll
        for (int m = 1; m < M; ++m) S = __fadd2_rn(S, bp[m]);
        float rA, rB;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rA) : "f"(S.x));
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rB) : "f"(S.y));
        const float2 r100 = __fmul2_rn(make_float2(rA, rB), make_float2(100.f, 100.f));
        float2 kf[M];
        float dmaxA = 0.f, dmaxB = 0.f;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            kf[m] = __ffma2_rn(bp[m], r100, magic2);                       // low mantissa bits = rint(100*bp/S)
            const float2 nk = __ffma2_rn(kf[m], minus1, magic2);           // magic - kf, exact
            const float2 d = __ffma2_rn(bp[m], r100, nk);                  // distance to that integer
            dmaxA = fmaxf(dmaxA, fabsf(d.x));
            dmaxB = fmaxf(dmaxB, fabsf(d.y));
        }
        float2 c0 = __fmul2_rn(bp[0], make_float2(f0[0], f0[0])), c1 = __fmul2_rn(bp[0], make_float2(f01[0], f01[0]));
#pragma unroll
        for (int m = 1; m < M; ++m) {
            c0 = __ffma2_rn(bp[m], make_float2(f0[m], f0[m]), c0);
            c1 = __ffma2_rn(bp[m], make_float2(f01[m], f01[m]), c1);
        }
        const float2 uS = __fmul2_rn(make_float2(ufA, ufB), S);
        const float2 win = __fmul2_rn(S, make_float2(kCdfWindow, kCdfWindow));
        const float2 g0 = __ffma2_rn(c0, minus1, uS), g1 = __ffma2_rn(c1, minus1, uS);   // uS - c0, uS - c1
        const uint32_t apA = uS.x < c0.x ? 0u : (uS.x < c1.x ? 1u : 2u), apB = uS.y < c0.y ? 0u : (uS.y < c1.y ? 1u : 2u);
        const bool exA = (dmaxA > kHalfWindow) | (fminf(fabsf(g0.x), fabsf(g1.x)) < win.x) | (ufA > 1.f - 2e-5f);
        const bool exB = (dmaxB > kHalfWindow) | (fminf(fabsf(g0.y), fabsf(g1.y)) < win.y) | (ufB > 1.f - 2e-5f);
        auto pack = [&](bool second, uint32_t ap) -> uint2 {
            uint32_t kb[M];
#pragma unroll
            for (int m = 0; m < M; ++m) kb[m] = __float_as_uint(second ? kf[m].y : kf[m].x);
            uint2 out;
            out.x = __byte_perm(__byte_perm(kb[0], kb[1 < M ? 1 : 0], 0x0040u), __byte_perm(kb[2 < M ? 2 : 0], kb[3 < M ? 3 : 0], 0x0040u), 0x5410u);
            if (M < 4) out.x &= (M == 2 ? 0xFFFFu : 0xFFFFFFu);
            // byte 0 = k4 (M > 4), byte 1 = k5 (M > 5), byte 2 = predicted action, byte 3 = 0 (ap < 256: its byte 1 is zero)
            out.y = M > 5 ? __byte_perm(__byte_perm(kb[M > 4 ? 4 : 0], kb[M > 5 ? 5 : 0], 0x0040u), ap, 0x5410u)
                          : (M > 4 ? __byte_perm(kb[M > 4 ? 4 : 0], ap, 0x5450u) : ap << 16);
            return out;
        };
        outA = pack(false, apA);
        outB = pack(true, apB);
        return (exA ? 1u : 0u) | (exB ? 2u : 0u);
    };
    auto dump = [&](int64_t rec, uint2 out) {
        if (belief_out) {
#pragma unroll
            for (int m = 0; m < M; ++m) belief_out[rec * M + m] = (uint8_t)(((m < 4 ? out.x : out.y) >> (8 * (m & 3))) & 0xFFu);
        }
        if (pred_out) pred_out[rec] = (uint8_t)(out.y >> 16);
    };

    const int total = n_envs * KQ;
    const bool warp_one_env = (KQ & 31) == 0;   // then total % 32 == 0 too: every warp is full and stays inside one env
    const int d_el = (int)blockDim.x / KQ, d_sq = (int)blockDim.x % KQ;
    int el = (int)threadIdx.x / KQ, sq = (int)threadIdx.x % KQ;
    uint8_t* const rec_base = P.records + ((e0 * N + i) * (int64_t)K) * IA2C_BELIEF_RECORD;   // record (e0, i, 0); block-local offsets fit 32 bits
    const uint32_t env_stride = (uint32_t)N * (uint32_t)K * IA2C_BELIEF_RECORD;
    const uint32_t d_off = (uint32_t)d_el * env_stride + (uint32_t)d_sq * (4 * IA2C_BELIEF_RECORD);
    const uint32_t wrap_off = env_stride - (uint32_t)KQ * (4 * IA2C_BELIEF_RECORD);
    uint32_t off = (uint32_t)el * env_stride + (uint32_t)sq * (4 * IA2C_BELIEF_RECORD);   // byte offset of the thread's quad
    // Philox counter of the thread's quad: (global belief row) * KQ + sq, as a block-uniform 64-bit base plus a local part
    const uint64_t ctr0 = (uint64_t)((P.env_offset + e0) * N + i) * (uint64_t)KQ;
    const uint32_t row_ctr = (uint32_t)N * (uint32_t)KQ;                                     // one env further
    uint32_t ctr = (uint32_t)el * row_ctr + (uint32_t)sq;
    const uint32_t d_ctr = (uint32_t)d_el * row_ctr + (uint32_t)d_sq, wrap_ctr = row_ctr - (uint32_t)KQ;
    const uint32_t c2 = (P.t & 0xFFFFu) | (kStreamBelief << 16);
    auto quad_words = [&](uint32_t ctr_) -> uint4 {
        const uint64_t index = ctr0 + ctr_;
        return philox4x32_10_rk(make_uint4((uint32_t)index, (uint32_t)(index >> 32), c2, P.episode), P.rk);
    };
    // The record stream is staged through shared memory with cp.async: every thread owns four 8-byte slots per stage
    // (laid out [slot][thread]: conflict-free) and copies its quad of iteration it + kStages - 1 while it computes on iteration it — kStages - 1 quads (up to 96 B) per
    // thread in flight without holding a register, and no barrier (a thread only reads what it copied itself).  A quad that
    // hangs over the end of the row (K not a multiple of 4) re-reads the row's last record and computes on it; only the
    // stores and the count leave it out.
    constexpr int kStages = 4;
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage) + threadIdx.x * 8u;   // [stage][slot w][thread]: conflict-free
    auto issue = [&](uint32_t off_, int sq_, int slot, bool live) {
        if (live && !reset_prior) {
            const uint8_t* rp = rec_base + off_;
            const uint32_t dst = stage_s + (uint32_t)slot * (kThreads * 32u);
            const int last = K - 1 - 4 * sq_;                               // >= 3 for a whole quad
#pragma unroll
            for (int w = 0; w < 4; ++w)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + (kThreads * 8u) * w), "l"(rp + 8 * min(w, last)) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // (el, sq, off, ctr) of the quad the thread will ISSUE next; the quad it COMPUTES on trails kStages - 1 iterations behind
    int el_i = el, sq_i = sq;
    uint32_t off_i = off;
    auto advance = [&](int& el_, int& sq_, uint32_t& off_, uint32_t* ctr_) {
        el_ += d_el; sq_ += d_sq; off_ += d_off;
        if (ctr_) *ctr_ += d_ctr;
        if (sq_ >= KQ) { sq_ -= KQ; ++el_; off_ += wrap_off; if (ctr_) *ctr_ += wrap_ctr; }
    };
    int q_i = threadIdx.x;
#pragma unroll
    for (int st = 0; st < kStages - 1; ++st) {
        issue(off_i, sq_i, st, q_i < total);
        advance(el_i, sq_i, off_i, nullptr);
        q_i += blockDim.x;
    }
    int slot = 0;
    for (int q = threadIdx.x; q < total; q += blockDim.x) {
        issue(off_i, sq_i, (slot + kStages - 1) % kStages, q_i < total);
        advance(el_i, sq_i, off_i, nullptr);
        q_i += blockDim.x;
        asm volatile("cp.async.wait_group %0;" ::"n"(kStages - 1) : "memory");
        uint2 raw[4];
        {
            const uint32_t src = stage_s + (uint32_t)slot * (kThreads * 32u);
#pragma unroll
            for (int w = 0; w < 4; ++w)
                asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(raw[w].x), "=r"(raw[w].y) : "r"(src + (kThreads * 8u) * w) : "memory");
            if (reset_prior) raw[0] = raw[1] = raw[2] = raw[3] = make_uint2(0u, 0u);
        }
        slot = (slot + 1) % kStages;
        const int jj0 = 4 * sq;
        const int n_valid = min(4, K - jj0);
        const int64_t rec0 = ((e0 + el) * N + i) * (int64_t)K + jj0;   // only the optional dumps / injected tapes index with it
        uint32_t words[4] = {0u, 0u, 0u, 0u};
        if (!u_injected) {
            const uint4 rnd = quad_words(ctr);
            words[0] = rnd.x; words[1] = rnd.y; words[2] = rnd.z; words[3] = rnd.w;
        }
        const uint32_t seen_w = seen4[q];
        uint2 out[4];
        float uf[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            if (u_injected) uf[w] = (float)u_injected[rec0 + min(w, n_valid - 1)];
            else uf[w] = __uint_as_float(0x3F800000u | (words[w] >> 9)) - 1.0f;   // floor(word / 2^9) * 2^-23: within 2^-23 of u
        }
        uint32_t need = screen_pair(__byte_perm(seen_w, 0u, 0x4440u), __byte_perm(seen_w, 0u, 0x4441u), uf[0], uf[1], raw[0], raw[1], out[0], out[1]);
        need |= screen_pair(__byte_perm(seen_w, 0u, 0x4442u), __byte_perm(seen_w, 0u, 0x4443u), uf[2], uf[3], raw[2], raw[3], out[2], out[3]) << 2;
        need &= (1u << n_valid) - 1u;
        if (need) {   // ~1 % of the quads: defer the flagged records to the exact pass below (their stored record stays untouched)
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                if (need & (1u << w)) {
                    const int pos = atomicAdd(&queue_n, 1);
                    if (pos < kExactQueue) {
                        queue[pos] = (uint16_t)(4 * q + w);
                    } else {   // queue full (never seen in practice): the exact sequence right here
                        const double u = u_injected ? u_injected[rec0 + w] : belief_word_to_unit_f64(words[w]);
                        const uint32_t seen = (seen_w >> (8 * w)) & 0xFFu;
                        out[w] = belief_exact_record<M>(bpt + seen * (M * 101), fa, raw[w], prior_k, u);
                        need &= ~(1u << w);
                    }
                }
            }
        }
        uint2* const wp = reinterpret_cast<uint2*>(rec_base + off);
        uint32_t packed = 0u;
        if (n_valid == 4 && !need) {
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                wp[w] = out[w];
                packed += 1u << (10u * (out[w].y >> 16));
            }
        } else {
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                if (w < n_valid && !(need & (1u << w))) {
                    wp[w] = out[w];
                    packed += 1u << (10u * (out[w].y >> 16));
                }
            }
        }
        if (belief_out || pred_out) {
#pragma unroll
            for (int w = 0; w < 4; ++w)
                if (w < n_valid && !(need & (1u << w))) dump(rec0 + w, out[w]);
        }
        if (FAST || P.pred_partner_out) {   // one REDUX + one shared atomic per group of lanes that share the env
            if (warp_one_env) {             // KQ % 32 == 0 and full warps: the whole warp works on one env
                const uint32_t sum = __reduce_add_sync(0xffffffffu, packed);
                if ((threadIdx.x & 31) == 0) atomicAdd(&counts[el], sum);
            } else {
                const unsigned peers = __match_any_sync(__activemask(), el);
                const uint32_t sum = __reduce_add_sync(peers, packed);
                if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&counts[el], sum);
            }
        }
        advance(el, sq, off, &ctr);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    // exact pass: the deferred records, one per thread, with the reference's fp64 sequence (dense: no lane waits for another's rare case)
    const int n_deferred = min(queue_n, kExactQueue);
    for (int x = threadIdx.x; x < n_deferred; x += blockDim.x) {
        const int code = queue[x], q = code >> 2, w = code & 3;
        const int el_ = q / KQ, sq_ = q - el_ * KQ;
        const int64_t rec = ((e0 + el_) * N + i) * (int64_t)K + 4 * sq_ + w;
        uint2* rp = reinterpret_cast<uint2*>(P.records + rec * IA2C_BELIEF_RECORD);
        const uint2 raw = reset_prior ? make_uint2(0u, 0u) : *rp;
        double u;
        if (u_injected) {
            u = u_injected[rec];
        } else {
            const uint4 rnd = quad_words((uint32_t)el_ * row_ctr + (uint32_t)sq_);
            u = belief_word_to_unit_f64(w == 0 ? rnd.x : (w == 1 ? rnd.y : (w == 2 ? rnd.z : rnd.w)));
        }
        const uint32_t seen = (seen4[q] >> (8 * w)) & 0xFFu;
        const uint2 out = belief_exact_record<M>(bpt + seen * (M * 101), fa, raw, prior_k, u);
        *rp = out;
        dump(rec, out);
        if (FAST || P.pred_partner_out) atomicAdd(&counts[el_], 1u << (10u * (out.y >> 16)));
    }
    if (P.pred_partner_out) {
        __syncthreads();
        for (int x = threadIdx.x; x < n_envs; x += blockDim.x) {
            const uint32_t c = counts[x];
            const int c0 = c & 1023, c1 = (c >> 10) & 1023, c2n = c >> 20;
            int best = 0, bc = c0;
            if (c1 > bc) { best = 1; bc = c1; }
            if (c2n > bc) best = 2;                                  // ties -> lowest action
            P.pred_partner_out[(e0 + x) * N + i] = (uint8_t)best;
        }
    }
}

template <int M>
int launch_pairs_table(PairsArgs& P, cudaStream_t stream) {
    P.envs_per_block = std::max(1, std::min(64, 16384 / P.K));   // amortise the table build and the staging of the others' actions
    const int64_t env_blocks = (P.E + P.envs_per_block - 1) / P.envs_per_block;
    size_t smem = (104 + 3 * M * 101 + M * 3) * sizeof(double) + (((3 * M * 101 + 3) & ~3) + ((2 * M + 3) & ~3)) * sizeof(float) +
                  (size_t)P.envs_per_block * sizeof(uint32_t) + kExactQueue * sizeof(uint16_t) +
                  (size_t)P.envs_per_block * (((size_t)P.K + 3) & ~size_t(3));
    smem = (smem + 15) & ~size_t(15);
    P.stage_offset = (uint32_t)smem;
    smem += (size_t)4 * kThreads * 32;   // kStages slots of 32 B per thread
    dim3 grid((unsigned)env_blocks, P.N);
    const bool fast = !P.reset_prior && !P.u_injected && !P.belief_out && !P.pred_out && P.pred_partner_out;
    if (fast) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(belief_pairs_table_kernel<M, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return launch_pdl("belief_pairs_table_kernel", belief_pairs_table_kernel<M, true>, grid, dim3(kThreads), smem, stream, P);
    } else {
        if (smem > 48 * 1024) cudaFuncSetAttribute(belief_pairs_table_kernel<M, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return launch_pdl("belief_pairs_table_kernel", belief_pairs_table_kernel<M, false>, grid, dim3(kThreads), smem, stream, P);
    }
}

// ------------------------------------------------------------------------------------------------
// Whole-episode pairwise update for many modelled others (9 <= N <= 512): the trainer's rollout.
//
// During a rollout nothing reads a belief before the update phase: the env and the actors depend on the sampled actions
// only (ia2c.py:72-102 — the filter's predicted action enters the critic's index at ia2c.py:104-121, after the episode).
// The rollout therefore runs its T+1 env / actor steps first and then updates every belief record through ALL T+1 steps in
// ONE kernel with the record resident on the SM (shared memory): the 16 bytes per update that belief_pairs_table_kernel streams per step
// (8-byte record read + written) shrink to one 8-byte store per EPISODE, and the byte unpack / pack, the address arithmetic,
// the cp.async ring and the table build are paid once per record-episode instead of once per update.  Same screen, same
// exact sequence, same Philox counters as the per-step kernel: bit-identical records, predictions and partner modes
// (tests/test_gpu_belief.py compares the two kernels and the oracle).
// Block = (agent, chunk of envs); every WARP owns whole envs (<= 4 quads = 16 records per lane) and runs the episode on its
// own: no block barrier inside the step loop.  Per step a warp stages the others' actions of the next step (registers ->
// its own shared-memory slots), screens its records, recomputes the flagged ones (~0.1 %) with the exact fp64 sequence —
// its own lanes, one record each, fixed in place before the next step reads them — reduces the predicted-action counts of
// its envs and writes partner_pred[t].  While one warp sits in an exact evaluation (a ~3000-cycle fp64 chain) the SM's
// other 15 warps keep screening: with the block-wide exact pass this kernel had first, 1.1 of every 5 cycles per issued
// instruction were barrier stalls (profiles/r02_ncu_summary.md §1b).
struct EpisodePairsArgs {
    uint8_t* records;              // [E,N,K,8] out: the posteriors after step T (+ predicted action of step T in byte 6)
    const double* filter_action;   // [N,M,3]
    const uint8_t* act;            // [T1,E,N] sampled actions of every step
    const double* u_injected;      // [T1,E,N,K] or null
    uint8_t* pred_dump;            // [T1,E,N,K] or null
    uint8_t* belief_dump;          // [T1,E,N,K,M] or null
    uint8_t* partner_pred;         // [T1,E,N]
    int64_t E, env_offset;
    int N, K, T1, envs_per_warp;
    uint32_t episode;
    uint32_t rk[20];
};
constexpr int kEpQuads = 4;                    // quads per lane
constexpr int kEpWarps = kThreads / 32;
constexpr int kEpWarpQuads = 32 * kEpQuads;    // quad slots of a warp: an env's KQ quads must fit (N <= 512)

// RUNS (FAST only): a batch of independent runs (ia2c_train_episode_runs_many), blockIdx.y = run * N + agent is the filter row; the
// run's envs are columns [run * E, (run + 1) * E) of an env axis of length R * E, `e0` stays the env's index within the run
// (Philox counters), and the Philox key is the run's seed, read after the wait.
// SEATS: frozen seats (ia2c_train_episode_frozen), grid y still R * N: y < R * L runs trained seat sa.seat[y % L] of run y / L;
// the blocks beyond it belong to the frozen rows, whose records stay untouched, and only write 0xFF ("no prediction") into
// their rows of partner_pred.
// (SEATS_Y: blockIdx.y, or in a SEATS instantiation the row of the full grid a trained row's block works as; trainer.cu has the same)
#define SEATS_Y (SEATS ? seats_y<RUNS>(N, sa) : blockIdx.y)
template <int M, bool FAST, bool RUNS, bool SEATS = false>
__global__ void __launch_bounds__(kThreads, 2) belief_pairs_episode_kernel(const __grid_constant__ EpisodePairsArgs P, RunsArg<RUNS> ra,
                                                                           const __grid_constant__ SeatsArg<SEATS> sa) {
    static_assert(FAST || !RUNS, "batches have no dumps or tapes");
    constexpr int A = IA2C_AGENT_ACTIONS;
    const double* const u_injected = FAST ? nullptr : P.u_injected;
    uint8_t* const belief_dump = FAST ? nullptr : P.belief_dump;
    uint8_t* const pred_dump = FAST ? nullptr : P.pred_dump;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int queue_n_w[kEpWarps];   // flagged records of the warp's current step
    const int N = P.N, K = P.K, i = RUNS ? (int)SEATS_Y % N : SEATS_Y;   // i: the agent
    const int run = RUNS ? (int)SEATS_Y / N : 0;
    if constexpr (SEATS) {
        const int n_runs = RUNS ? (int)gridDim.y / N : 1, L = sa.L;
        if ((int)blockIdx.y >= n_runs * L) {   // a frozen row: this block's envs, every step
            pdl_release();
            pdl_wait();
            const int y = (int)blockIdx.y - n_runs * L, nf = N - L, seat = sa.seat[L + y % nf];
            const int64_t col = (int64_t)(y / nf) * P.E, eb = (int64_t)blockIdx.x * kEpWarps * P.envs_per_warp;
            const int64_t ne = min((int64_t)kEpWarps * P.envs_per_warp, P.E - eb);
            for (int64_t k = threadIdx.x; k < (int64_t)P.T1 * ne; k += blockDim.x)
                P.partner_pred[((k / ne) * P.E * n_runs + col + eb + k % ne) * N + seat] = 0xFF;
            return;
        }
    }
    const int KQ = (K + 3) >> 2;
    const int EW = P.envs_per_warp, EWp = (EW + 3) & ~3;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t e0 = ((int64_t)blockIdx.x * kEpWarps + warp) * EW;                 // the warp's first env (within its run)
    // the env axis has n_runs * E columns, the run's start at col0 (both folded away in the standalone form, which thus reads P.E
    // where it always did)
    const int n_runs = RUNS ? (int)gridDim.y / N : 1;
    const int64_t col0 = RUNS ? (int64_t)run * P.E : 0;
    const int n_envs = (int)max((int64_t)0, min((int64_t)EW, P.E - e0));
    double* tab = reinterpret_cast<double*>(smem_raw);               // [104]   k/100
    double* bpt = tab + 104;                                         // [A][M][101]
    double* fa = bpt + A * M * 101;                                  // [M][A]
    float* bpt32 = reinterpret_cast<float*>(fa + M * A);             // [A][M][101]
    float* fcum = bpt32 + ((A * M * 101 + 3) & ~3);                  // [2][M]: F[m][0], F[m][0]+F[m][1]
    uint32_t* counts = reinterpret_cast<uint32_t*>(fcum + ((2 * M + 3) & ~3)) + warp * EWp;   // [warps][EWp] packed 3 x 10 bits
    uint2* st_mem = reinterpret_cast<uint2*>(counts - warp * EWp + kEpWarps * EWp);            // [4 * kEpQuads][kThreads] the records
    uint16_t* queue = reinterpret_cast<uint16_t*>(st_mem + 4 * kEpQuads * kThreads) + warp * (4 * kEpWarpQuads);   // [warps][records of a warp]
    uint32_t* seen4 = reinterpret_cast<uint32_t*>(queue - warp * (4 * kEpWarpQuads) + 4 * kEpQuads * kThreads);    // [kEpQuads][kThreads] the others' actions
    pdl_release();
    for (int k = threadIdx.x; k <= 100; k += blockDim.x) tab[k] = __ddiv_rn((double)k, 100.0);
    for (int k = threadIdx.x; k < M * A; k += blockDim.x) fa[k] = P.filter_action[(int64_t)(RUNS ? SEATS_Y : i) * M * A + k];
    if (threadIdx.x < kEpWarps) queue_n_w[threadIdx.x] = 0;
    for (int k = threadIdx.x; k < kEpWarps * EWp; k += blockDim.x) (counts - warp * EWp)[k] = 0u;
    __syncthreads();
    for (int x = threadIdx.x; x < A * M * 101; x += blockDim.x) {
        const int seen = x / (M * 101), m = (x / 101) % M, k = x % 101;
        const double p = tab[k];
        double acc = __dmul_rn(seen == 0 ? 0.8 : 0.1, __dmul_rn(fa[m * A + 0], p));
#pragma unroll
        for (int a = 1; a < A; ++a) acc = __dadd_rn(acc, __dmul_rn(seen == a ? 0.8 : 0.1, __dmul_rn(fa[m * A + a], p)));
        bpt[x] = acc;
        bpt32[x] = (float)acc;
    }
    if (threadIdx.x < M) {
        fcum[threadIdx.x] = (float)fa[threadIdx.x * A];
        fcum[M + threadIdx.x] = (float)__dadd_rn(fa[threadIdx.x * A], fa[threadIdx.x * A + 1]);
    }
    pdl_wait();
    __syncthreads();   // the last block-wide barrier: from here on the warps run independently
    if (n_envs == 0) return;
    // Philox with the round keys of P.rk or, in a batch, keyed by the run's seed: philox4x32_10 derives key_r = key_0 + r * W as
    // it goes, the formula the host fills P.rk with, so the numbers are the same
    uint2 run_key = make_uint2(0u, 0u);
    if constexpr (RUNS) {
        const uint64_t seed = ra.seed[run];
        run_key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    }
    auto philox = [&](uint4 c) -> uint4 {
        if constexpr (RUNS) return philox4x32_10(c, run_key);
        else return philox4x32_10_rk(c, P.rk);
    };
    float f0[M], f01[M];
#pragma unroll
    for (int m = 0; m < M; ++m) { f0[m] = fcum[m]; f01[m] = fcum[M + m]; }
    const uint32_t bpt32_s = (uint32_t)__cvta_generic_to_shared(bpt32);
    const float2 magic2 = make_float2(kRoundMagic, kRoundMagic), minus1 = make_float2(-1.f, -1.f);

    // fp32 screen of two records (see belief_pairs_table_kernel) -> packed records; bit w: record w's rounding is inside the
    // first-level window, bit 4 + w: its inverse-CDF comparison is too close to call
    auto screen_pair = [&](uint32_t seenA, uint32_t seenB, float ufA, float ufB, uint2 rawA, uint2 rawB, uint2& outA, uint2& outB) -> uint32_t {
        const uint32_t rowA = bpt32_s + seenA * (M * 101 * 4), rowB = bpt32_s + seenB * (M * 101 * 4);
        float2 bp[M];
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const uint32_t sel = 0x4440u | (uint32_t)(m & 3);
            const uint32_t kA = __byte_perm(m < 4 ? rawA.x : rawA.y, 0u, sel), kB = __byte_perm(m < 4 ? rawB.x : rawB.y, 0u, sel);
            bp[m] = make_float2(lds_f32(rowA + 4u * kA + (uint32_t)(m * 101 * 4)), lds_f32(rowB + 4u * kB + (uint32_t)(m * 101 * 4)));
        }
        float2 S = bp[0];
#pragma unroll
        for (int m = 1; m < M; ++m) S = __fadd2_rn(S, bp[m]);
        float rA, rB;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rA) : "f"(S.x));
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rB) : "f"(S.y));
        const float2 r100 = __fmul2_rn(make_float2(rA, rB), make_float2(100.f, 100.f));
        float2 kf[M];
        float dmaxA = 0.f, dmaxB = 0.f;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            kf[m] = __ffma2_rn(bp[m], r100, magic2);
            const float2 nk = __ffma2_rn(kf[m], minus1, magic2);
            const float2 d = __ffma2_rn(bp[m], r100, nk);
            dmaxA = fmaxf(dmaxA, fabsf(d.x));
            dmaxB = fmaxf(dmaxB, fabsf(d.y));
        }
        float2 c0 = __fmul2_rn(bp[0], make_float2(f0[0], f0[0])), c1 = __fmul2_rn(bp[0], make_float2(f01[0], f01[0]));
#pragma unroll
        for (int m = 1; m < M; ++m) {
            c0 = __ffma2_rn(bp[m], make_float2(f0[m], f0[m]), c0);
            c1 = __ffma2_rn(bp[m], make_float2(f01[m], f01[m]), c1);
        }
        const float2 uS = __fmul2_rn(make_float2(ufA, ufB), S);
        const float2 win = __fmul2_rn(S, make_float2(kCdfWindow, kCdfWindow));
        const float2 g0 = __ffma2_rn(c0, minus1, uS), g1 = __ffma2_rn(c1, minus1, uS);
        const uint32_t apA = uS.x < c0.x ? 0u : (uS.x < c1.x ? 1u : 2u), apB = uS.y < c0.y ? 0u : (uS.y < c1.y ? 1u : 2u);
        const bool rdA = dmaxA > kHalfWindow, rdB = dmaxB > kHalfWindow;          // rounding too close to call (first level)
        const bool cdA = (fminf(fabsf(g0.x), fabsf(g1.x)) < win.x) | (ufA > 1.f - 2e-5f);
        const bool cdB = (fminf(fabsf(g0.y), fabsf(g1.y)) < win.y) | (ufB > 1.f - 2e-5f);
        auto pack = [&](bool second, uint32_t ap) -> uint2 {
            uint32_t kb[M];
#pragma unroll
            for (int m = 0; m < M; ++m) kb[m] = __float_as_uint(second ? kf[m].y : kf[m].x);
            uint2 out;
            out.x = __byte_perm(__byte_perm(kb[0], kb[1 < M ? 1 : 0], 0x0040u), __byte_perm(kb[2 < M ? 2 : 0], kb[3 < M ? 3 : 0], 0x0040u), 0x5410u);
            if (M < 4) out.x &= (M == 2 ? 0xFFFFu : 0xFFFFFFu);
            out.y = M > 5 ? __byte_perm(__byte_perm(kb[M > 4 ? 4 : 0], kb[M > 5 ? 5 : 0], 0x0040u), ap, 0x5410u)
                          : (M > 4 ? __byte_perm(kb[M > 4 ? 4 : 0], ap, 0x5450u) : ap << 16);
            return out;
        };
        outA = pack(false, apA);
        outB = pack(true, apB);
        return (rdA ? 1u : 0u) | (rdB ? 2u : 0u) | (cdA ? 16u : 0u) | (cdB ? 32u : 0u);
    };

    // ---- the lane's quads (fixed for the whole episode): quad slot ql = lane + 32 s of the warp, s < kEpQuads; env = ql / KQ,
    // quad of the env = ql % KQ.  The records live in shared memory ([slot][thread] 8-byte words: conflict-free), so the quad
    // loop is a real loop (the step body stays inside the instruction cache) and a flagged record is fixed in place.
    const int total = n_envs * KQ;                               // quad slots of this warp in use (<= kEpWarpQuads)
    const bool warp_one_env = (KQ & 31) == 0;
    const int prior_k = (int)rint(100.0 / M);
    uint2 prior;
    prior.x = (uint32_t)prior_k * (M >= 4 ? 0x01010101u : (M == 3 ? 0x010101u : 0x0101u));
    prior.y = M > 4 ? (uint32_t)prior_k * (M > 5 ? 0x0101u : 0x01u) : 0u;
    const uint32_t st_s = (uint32_t)__cvta_generic_to_shared(st_mem) + threadIdx.x * 8u;   // + (4 s + w) * kThreads * 8
#pragma unroll
    for (int k = 0; k < 4 * kEpQuads; ++k) st_mem[k * kThreads + threadIdx.x] = prior;
    const int d_el = 32 / KQ, d_sq = 32 % KQ;
    const int el0 = lane / KQ, sq0 = lane % KQ;
    const uint64_t ctr0 = (uint64_t)((P.env_offset + e0) * N + i) * (uint64_t)KQ;
    const uint32_t row_ctr = (uint32_t)N * (uint32_t)KQ;
    // staging of the others' actions of one step (own action skipped, 4 slots per word).  N % 4 == 0: every env's row of actions
    // is word-aligned — one or two 32-bit loads per quad and a byte permutation that drops the own action; any other N: four
    // byte loads per quad.
    const bool aligned = (N & 3) == 0;
    const int NW = N >> 2, iw = i >> 2;
    const uint32_t sel_mix = (i & 3) == 0 ? 0x4321u : ((i & 3) == 1 ? 0x4320u : ((i & 3) == 2 ? 0x4310u : 0x4210u));
    // per quad, fixed for the episode — aligned: source word offset and byte selector; otherwise: byte offset of the env's row
    // and the quad's first slot.  Padding slots (jj >= K) keep whatever the selector picks / zero — they are computed on but
    // never stored or counted.
    uint32_t stage_lo[kEpQuads], stage_hi[kEpQuads], stage_src[kEpQuads], stage_sel[kEpQuads];
    {
        int el = el0, sq = sq0;
#pragma unroll
        for (int s_ = 0; s_ < kEpQuads; ++s_) {
            const bool ok = lane + 32 * s_ < total;
            if (aligned) {
                stage_src[s_] = ok ? (uint32_t)(el * NW + sq) : 0xFFFFFFFFu;
                stage_sel[s_] = (sq < iw ? 0x3210u : (sq > iw ? 0x4321u : sel_mix)) | (sq + 1 < NW ? 0u : 0x80000000u);   // bit 31: no next word
            } else {
                stage_src[s_] = ok ? (uint32_t)(el * N) : 0xFFFFFFFFu;
                stage_sel[s_] = (uint32_t)(4 * sq);
            }
            el += d_el; sq += d_sq;
            if (sq >= KQ) { sq -= KQ; ++el; }
        }
    }
    // the actions are written by the kernel before this one: coherent loads (an ld.global.nc may be hoisted above griddepcontrol.wait)
    auto stage_load = [&](int t) {
        const uint8_t* src8 = P.act + ((int64_t)t * P.E * n_runs + col0 + e0) * N;
        if (aligned) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(src8);
#pragma unroll
            for (int s_ = 0; s_ < kEpQuads; ++s_) {
                const bool ok = stage_src[s_] != 0xFFFFFFFFu;
                stage_lo[s_] = ok ? __ldcg(src + stage_src[s_]) : 0u;
                stage_hi[s_] = (ok && !(stage_sel[s_] >> 31)) ? __ldcg(src + stage_src[s_] + 1) : 0u;
            }
        } else {
#pragma unroll
            for (int s_ = 0; s_ < kEpQuads; ++s_) {
                uint32_t word = 0u;
                if (stage_src[s_] != 0xFFFFFFFFu) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int jj = (int)stage_sel[s_] + k;               // modelled-other slot -> agent index, skipping self
                        if (jj < K) word |= (uint32_t)__ldcg(src8 + stage_src[s_] + jj + (jj >= i ? 1 : 0)) << (8 * k);
                    }
                }
                stage_lo[s_] = word;
            }
        }
    };
    auto stage_store = [&]() {   // own slots only
#pragma unroll
        for (int s_ = 0; s_ < kEpQuads; ++s_)
            seen4[s_ * kThreads + threadIdx.x] = aligned ? __byte_perm(stage_lo[s_], stage_hi[s_], stage_sel[s_] & 0xFFFFu) : stage_lo[s_];
    };
    auto dump = [&](int64_t trec, uint2 out) {
        if (belief_dump) {
#pragma unroll
            for (int m = 0; m < M; ++m) belief_dump[trec * M + m] = (uint8_t)(((m < 4 ? out.x : out.y) >> (8 * (m & 3))) & 0xFFu);
        }
        if (pred_dump) pred_dump[trec] = (uint8_t)(out.y >> 16);
    };
    stage_load(0);
    stage_store();
    __syncwarp();

    for (int t = 0; t < P.T1; ++t) {
        if (t + 1 < P.T1) stage_load(t + 1);                       // next step's actions: in flight during this step's arithmetic
        const uint32_t c2 = ((uint32_t)t & 0xFFFFu) | (kStreamBelief << 16);
        const int64_t tbase = (int64_t)t * P.E * N * K;            // index of step t in the per-step tapes / dumps
        int el = el0, sq = sq0;
#pragma unroll 1
        for (int s_ = 0; s_ < kEpQuads; ++s_) {
            const int ql = lane + 32 * s_;
            if (32 * s_ >= total) break;                           // warp-uniform: whole warp past the end
            const bool live = ql < total;
            const int jj0 = 4 * sq;
            const int n_valid = live ? min(4, K - jj0) : 0;
            const int64_t trec0 = tbase + ((e0 + (live ? el : 0)) * N + i) * (int64_t)K + jj0;
            uint32_t words[4] = {0u, 0u, 0u, 0u};
            if (!u_injected) {
                const uint64_t index = ctr0 + (uint32_t)(live ? el : 0) * row_ctr + (uint32_t)sq;
                const uint4 rnd = philox(make_uint4((uint32_t)index, (uint32_t)(index >> 32), c2, P.episode));
                words[0] = rnd.x; words[1] = rnd.y; words[2] = rnd.z; words[3] = rnd.w;
            }
            const uint32_t seen_w = live ? seen4[s_ * kThreads + threadIdx.x] : 0u;
            const uint32_t sp = st_s + (uint32_t)(4 * s_) * (kThreads * 8u);
            uint2 raw[4];
#pragma unroll
            for (int w = 0; w < 4; ++w)
                asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(raw[w].x), "=r"(raw[w].y) : "r"(sp + (kThreads * 8u) * w) : "memory");
            float uf[4];
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                if (u_injected) uf[w] = n_valid ? (float)u_injected[trec0 + min(w, n_valid - 1)] : 0.f;
                else uf[w] = __uint_as_float(0x3F800000u | (words[w] >> 9)) - 1.0f;
            }
            uint2 out[4];
            uint32_t need = screen_pair(__byte_perm(seen_w, 0u, 0x4440u), __byte_perm(seen_w, 0u, 0x4441u), uf[0], uf[1], raw[0], raw[1], out[0], out[1]);
            need |= screen_pair(__byte_perm(seen_w, 0u, 0x4442u), __byte_perm(seen_w, 0u, 0x4443u), uf[2], uf[3], raw[2], raw[3], out[2], out[3]) << 2;
            need &= ((1u << n_valid) - 1u) * 0x11u;
            if (need) {   // ~0.4 % of the quads: second-level test of the rounding flags, value by value
                uint32_t still = need >> 4;
#pragma unroll
                for (int w = 0; w < 4; ++w)
                    if ((need & ~still) & (1u << w))
                        still |= belief_refine_rounding<M>(bpt32_s + ((seen_w >> (8 * w)) & 0xFFu) * (M * 101 * 4), raw[w]) ? (1u << w) : 0u;
                need = still;
            }
            uint32_t packed = 0u;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                if (w < n_valid && !(need & (1u << w))) {
                    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(sp + (kThreads * 8u) * w), "r"(out[w].x), "r"(out[w].y) : "memory");
                    packed += 1u << (10u * (out[w].y >> 16));
                    if (belief_dump || pred_dump) dump(trec0 + w, out[w]);
                }
            }
            if (need) {   // ~0.1 % of the quads: the flagged records go to the warp's exact pass below, which fixes them in place
                int pos = atomicAdd(&queue_n_w[warp], __popc(need));
#pragma unroll
                for (int w = 0; w < 4; ++w)
                    if (need & (1u << w)) queue[pos++] = (uint16_t)((ql << 2) | w);
            }
            if (warp_one_env) {
                const uint32_t sum = __reduce_add_sync(0xffffffffu, packed);
                if (lane == 0) atomicAdd(&counts[el], sum);
            } else {
                const unsigned peers = __match_any_sync(__activemask(), live ? el : -1);
                const uint32_t sum = __reduce_add_sync(peers, packed);
                if (lane == __ffs(peers) - 1 && live) atomicAdd(&counts[el], sum);
            }
            el += d_el; sq += d_sq;
            if (sq >= KQ) { sq -= KQ; ++el; }
        }
        __syncwarp();
        // ---- exact pass of the warp: its flagged records, one per lane, with the reference's fp64 sequence, fixed in place
        const int n_def = *reinterpret_cast<volatile int*>(&queue_n_w[warp]);
        for (int x = lane; x < n_def; x += 32) {
            const int code = queue[x], ql = code >> 2, w = code & 3;
            const int el_ = ql / KQ, sq_ = ql - el_ * KQ;
            uint2* rp = st_mem + (4 * (ql >> 5) + w) * kThreads + (warp << 5) + (ql & 31);
            const int64_t trec = tbase + ((e0 + el_) * N + i) * (int64_t)K + 4 * sq_ + w;
            double u;
            if (u_injected) {
                u = u_injected[trec];
            } else {
                const uint64_t index = ctr0 + (uint32_t)el_ * row_ctr + (uint32_t)sq_;
                const uint4 rnd = philox(make_uint4((uint32_t)index, (uint32_t)(index >> 32), c2, P.episode));
                u = belief_word_to_unit_f64(w == 0 ? rnd.x : (w == 1 ? rnd.y : (w == 2 ? rnd.z : rnd.w)));
            }
            const uint32_t seen = (seen4[(ql >> 5) * kThreads + (warp << 5) + (ql & 31)] >> (8 * w)) & 0xFFu;
            const uint2 res = belief_exact_record<M>(bpt + seen * (M * 101), fa, *rp, -1, u);
            *rp = res;
            atomicAdd(&counts[el_], 1u << (10u * (res.y >> 16)));
            if (belief_dump || pred_dump) dump(trec, res);
        }
        __syncwarp();
        if (t + 1 < P.T1) stage_store();                           // the exact pass above was the last reader of this step's actions
        // ---- partner mode of step t
        for (int x = lane; x < n_envs; x += 32) {
            const uint32_t c = counts[x];
            const int n0 = c & 1023, n1 = (c >> 10) & 1023, n2 = c >> 20;
            int best = 0, bc = n0;
            if (n1 > bc) { best = 1; bc = n1; }
            if (n2 > bc) best = 2;                                   // ties -> lowest action
            P.partner_pred[((int64_t)t * P.E * n_runs + col0 + e0 + x) * N + i] = (uint8_t)best;
            counts[x] = 0u;
        }
        if (lane == 0) queue_n_w[warp] = 0;
        __syncwarp();
    }
    // ---- the final records
    {
        int el = el0, sq = sq0;
#pragma unroll
        for (int s_ = 0; s_ < kEpQuads; ++s_) {
            if (lane + 32 * s_ < total) {
                uint2* wp = reinterpret_cast<uint2*>(P.records + (((col0 + e0 + el) * N + i) * (int64_t)K + 4 * sq) * IA2C_BELIEF_RECORD);
#pragma unroll
                for (int w = 0; w < 4; ++w)
                    if (4 * sq + w < K) wp[w] = st_mem[(4 * s_ + w) * kThreads + threadIdx.x];
            }
            el += d_el; sq += d_sq;
            if (sq >= KQ) { sq -= KQ; ++el; }
        }
    }
}

#undef SEATS_Y

// Launch shape of belief_pairs_episode_kernel for P.E envs (of one run): sets P.envs_per_warp, returns the env blocks (grid x)
// and the dynamic shared memory.  The standalone and the batched launcher share it, so the batch's shared memory always
// matches what the kernel carves out of it.
struct EpisodeShape { int64_t env_blocks; size_t smem; };
template <int M>
EpisodeShape episode_shape(EpisodePairsArgs& P) {
    const int KQ = (P.K + 3) / 4;
    P.envs_per_warp = std::max(1, kEpWarpQuads / KQ);              // whole envs per warp, <= kEpQuads quads per lane
    const int64_t envs_per_block = (int64_t)P.envs_per_warp * kEpWarps;
    EpisodeShape sh;
    sh.env_blocks = (P.E + envs_per_block - 1) / envs_per_block;
    sh.smem = (104 + 3 * M * 101 + M * 3) * sizeof(double) + (((3 * M * 101 + 3) & ~3) + ((2 * M + 3) & ~3)) * sizeof(float) +
              (size_t)kEpWarps * ((P.envs_per_warp + 3) & ~3) * sizeof(uint32_t) +
              (size_t)4 * kEpQuads * kThreads * (sizeof(uint2) + sizeof(uint16_t)) + (size_t)kEpQuads * kThreads * sizeof(uint32_t);
    sh.smem = (sh.smem + 15) & ~size_t(15);
    return sh;
}

template <int M>
int launch_pairs_episode(EpisodePairsArgs& P, cudaStream_t stream) {
    const EpisodeShape sh = episode_shape<M>(P);
    const size_t smem = sh.smem;
    dim3 grid((unsigned)sh.env_blocks, P.N);
    const bool fast = !P.u_injected && !P.belief_dump && !P.pred_dump;
    if (fast) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(belief_pairs_episode_kernel<M, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return launch_pdl("belief_pairs_episode_kernel", belief_pairs_episode_kernel<M, true, false>, grid, dim3(kThreads), smem, stream, P, NoRuns{}, NoSeats{});
    }
    if (smem > 48 * 1024) cudaFuncSetAttribute(belief_pairs_episode_kernel<M, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return launch_pdl("belief_pairs_episode_kernel", belief_pairs_episode_kernel<M, false, false>, grid, dim3(kThreads), smem, stream, P, NoRuns{}, NoSeats{});
}

// The batched form (ia2c_train_episode_runs_many): one run's shape, grid (env blocks of one run, R * N).
template <int M>
int launch_pairs_episode_runs(EpisodePairsArgs& P, const ia2c_runs_desc& runs, cudaStream_t stream) {
    const EpisodeShape sh = episode_shape<M>(P);
    dim3 grid((unsigned)sh.env_blocks, (unsigned)(runs.runs * P.N));
    if (sh.smem > 48 * 1024)
        cudaFuncSetAttribute(belief_pairs_episode_kernel<M, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh.smem);
    return launch_pdl("belief_pairs_episode_kernel", belief_pairs_episode_kernel<M, true, true>, grid, dim3(kThreads), sh.smem, stream, P, runs, NoSeats{});
}

// The SEATS forms (ia2c_train_episode_frozen): grid y covers every filter row, trained rows first (belief_pairs_episode_kernel).
template <int M, bool FAST, bool RUNS>
int launch_episode_seats(EpisodePairsArgs& P, const RunsArg<RUNS>& ra, int rows, const TrainedSeats& f, cudaStream_t stream) {
    const EpisodeShape sh = episode_shape<M>(P);
    auto kernel = belief_pairs_episode_kernel<M, FAST, RUNS, true>;
    if (sh.smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh.smem);
    return launch_pdl("belief_pairs_episode_kernel", kernel, dim3((unsigned)sh.env_blocks, (unsigned)rows), dim3(kThreads), sh.smem, stream,
                      P, ra, f);
}
template <int M>
int launch_pairs_episode_seats(EpisodePairsArgs& P, const ia2c_runs_desc* runs, const TrainedSeats& f, cudaStream_t stream) {
    if (runs) return launch_episode_seats<M, true, true>(P, *runs, runs->runs * P.N, f, stream);
    if (!P.u_injected && !P.belief_dump && !P.pred_dump) return launch_episode_seats<M, true, false>(P, NoRuns{}, P.N, f, stream);
    return launch_episode_seats<M, false, false>(P, NoRuns{}, P.N, f, stream);
}

template <int M>
int launch_pairs(PairsArgs& P, cudaStream_t stream) {
    if (P.K >= 32 && P.N <= 65535) return launch_pairs_table<M>(P, stream);
    const int64_t per_env = (int64_t)P.N * P.K;
    const int target = 4096;  // records per block
    if (per_env <= target) {
        P.envs_per_block = (int)(target / per_env);
        if (P.envs_per_block > 256) P.envs_per_block = 256;
        P.agents_per_block = P.N;
        P.chunks_per_env = 1;
    } else {
        P.envs_per_block = 1;
        const int chunks = (int)((per_env + target - 1) / target);
        P.agents_per_block = (P.N + chunks - 1) / chunks;
        P.chunks_per_env = (P.N + P.agents_per_block - 1) / P.agents_per_block;
    }
    const int64_t env_blocks = (P.E + P.envs_per_block - 1) / P.envs_per_block;
    const int64_t blocks = env_blocks * P.chunks_per_env;
    size_t smem = 104 * sizeof(double) + (size_t)P.agents_per_block * M * 3 * sizeof(double) +
                  (size_t)P.envs_per_block * P.agents_per_block * 3 * sizeof(int) + (size_t)P.envs_per_block * P.N;
    smem = (smem + 15) & ~size_t(15);
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(belief_pairs_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    return launch_pdl("belief_pairs_kernel", belief_pairs_kernel<M>, dim3((unsigned)blocks), dim3(kThreads), smem, stream, P);
}

}  // namespace
}  // namespace ia2c

#ifndef IA2C_BELIEF_SEATS   // the entry points: in belief.cu; belief_seats.cu has the frozen-seat launch alone
using namespace ia2c;

extern "C" int ia2c_belief_update_dense(const double* filter_action, const double* lik, const double* prev,
                                        const double* u, int64_t* ap, double* bprime, double* prediction,
                                        int64_t R, int32_t M, int32_t A, void* stream) {
    IA2C_REQUIRE(R > 0 && filter_action && lik && prev && u && ap && bprime, "ia2c_belief_update_dense: R=%lld or null arrays", (long long)R);
    IA2C_REQUIRE(M >= 1 && M <= kMaxDense && A >= 1 && A <= kMaxDense, "ia2c_belief_update_dense: M=%d A=%d outside 1..8", M, A);
    const int blocks = ceil_div(R, kThreads);
    cudaStream_t s = as_stream(stream);
    if (M == 5 && A == 3) belief_dense_kernel<5, 3><<<blocks, kThreads, 0, s>>>(filter_action, lik, prev, u, ap, bprime, prediction, R);
    else if (M == 3 && A == 3) belief_dense_kernel<3, 3><<<blocks, kThreads, 0, s>>>(filter_action, lik, prev, u, ap, bprime, prediction, R);
    else if (M == 5 && A == 5) belief_dense_kernel<5, 5><<<blocks, kThreads, 0, s>>>(filter_action, lik, prev, u, ap, bprime, prediction, R);
    else belief_dense_generic_kernel<<<blocks, kThreads, 0, s>>>(filter_action, lik, prev, u, ap, bprime, prediction, R, M, A);
    return check_launch("belief_dense_kernel");
}

extern "C" int ia2c_debug_divide(const double* a, const double* b, double* q_seq, double* q_ieee, int64_t n, void* stream) {
    IA2C_REQUIRE(a && b && q_seq && q_ieee && n > 0, "ia2c_debug_divide: null pointer or n=%lld", (long long)n);
    debug_divide_kernel<<<ceil_div(n, 256), 256, 0, as_stream(stream)>>>(a, b, q_seq, q_ieee, n);
    return check_launch("debug_divide_kernel");
}

extern "C" int ia2c_belief_update_pairs(uint8_t* records, const double* filter_action, const uint8_t* actions,
                                        const double* u_injected, uint8_t* pred_out, uint8_t* belief_out,
                                        uint8_t* pred_partner_out, int64_t E, int32_t N, int32_t M,
                                        int32_t reset_prior, uint64_t seed, uint32_t episode, uint32_t t,
                                        int64_t env_offset, void* stream) {
    IA2C_REQUIRE(E > 0 && records && filter_action && actions, "ia2c_belief_update_pairs: E=%lld or null arrays", (long long)E);
    IA2C_REQUIRE(N >= 2 && N <= 1023, "ia2c_belief_update_pairs: N=%d outside 2..1023", N);
    IA2C_REQUIRE(M >= 2 && M <= IA2C_MAX_MODELS, "ia2c_belief_update_pairs: M=%d outside 2..%d", M, IA2C_MAX_MODELS);
    PairsArgs P{records, filter_action, actions, u_injected, pred_out, belief_out, pred_partner_out,
                E, env_offset, N, N - 1, 0, 0, 0, reset_prior, seed, episode, t, 0u, {}};
    for (int r = 0; r < 10; ++r) {
        P.rk[2 * r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
        P.rk[2 * r + 1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
    }
    cudaStream_t s = as_stream(stream);
    switch (M) {
        case 2: return launch_pairs<2>(P, s);
        case 3: return launch_pairs<3>(P, s);
        case 4: return launch_pairs<4>(P, s);
        case 5: return launch_pairs<5>(P, s);
        default: return launch_pairs<6>(P, s);
    }
}

extern "C" int ia2c_belief_supports_episode(int32_t N, int32_t M) { return N >= 9 && N <= 512 && M >= 2 && M <= IA2C_MAX_MODELS; }

extern "C" int ia2c_belief_update_pairs_episode(uint8_t* records, const double* filter_action, const uint8_t* act,
                                                const double* u_injected, uint8_t* pred_dump, uint8_t* belief_dump,
                                                uint8_t* partner_pred, int64_t E, int32_t N, int32_t M, int32_t T1, uint64_t seed,
                                                uint32_t episode, int64_t env_offset, void* stream) {
    IA2C_REQUIRE(E > 0 && T1 > 0 && records && filter_action && act && partner_pred, "ia2c_belief_update_pairs_episode: E=%lld T1=%d or null arrays",
                 (long long)E, T1);
    IA2C_REQUIRE(ia2c_belief_supports_episode(N, M), "ia2c_belief_update_pairs_episode: needs 9 <= N <= 512, 2 <= M <= %d; got N=%d M=%d",
                 IA2C_MAX_MODELS, N, M);
    IA2C_REQUIRE(T1 <= 65535, "ia2c_belief_update_pairs_episode: T1=%d", T1);
    EpisodePairsArgs P{records, filter_action, act, u_injected, pred_dump, belief_dump, partner_pred, E, env_offset, N, N - 1, T1, 0, episode, {}};
    for (int r = 0; r < 10; ++r) {
        P.rk[2 * r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
        P.rk[2 * r + 1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
    }
    cudaStream_t s = as_stream(stream);
    switch (M) {
        case 2: return launch_pairs_episode<2>(P, s);
        case 3: return launch_pairs_episode<3>(P, s);
        case 4: return launch_pairs_episode<4>(P, s);
        case 5: return launch_pairs_episode<5>(P, s);
        default: return launch_pairs_episode<6>(P, s);
    }
}

// The whole-episode belief update of a batch of runs (ia2c_train_episode_runs_many, which has validated both descriptors): the
// stacked trajectory of d (env axis R * E), one filter row per net, each run's seed as its Philox key.
int ia2c::belief_pairs_episode_runs_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, cudaStream_t s) {
    EpisodePairsArgs P{d->belief_records, d->filter_action, d->act, nullptr, nullptr, nullptr, d->partner_pred, d->E, 0, d->N, d->N - 1,
                       d->T + 1, 0, d->episode, {}};
    switch (d->M) {
        case 2: return launch_pairs_episode_runs<2>(P, *runs, s);
        case 3: return launch_pairs_episode_runs<3>(P, *runs, s);
        case 4: return launch_pairs_episode_runs<4>(P, *runs, s);
        case 5: return launch_pairs_episode_runs<5>(P, *runs, s);
        default: return launch_pairs_episode_runs<6>(P, *runs, s);
    }
}

#else
// The whole-episode belief update of a frozen-seat episode (ia2c_train_episode_frozen, which has validated everything): the
// standalone form of ia2c_belief_update_pairs_episode (runs NULL) or the batched form above, over the trained seats' rows.
int ia2c::belief_pairs_episode_seats_launch(const ia2c_episode_desc* d, const ia2c_runs_desc* runs, const TrainedSeats& f, cudaStream_t s) {
    EpisodePairsArgs P{d->belief_records, d->filter_action, d->act, nullptr, nullptr, nullptr, d->partner_pred, d->E, 0, d->N, d->N - 1,
                       d->T + 1, 0, d->episode, {}};
    if (!runs) {
        P.u_injected = d->inj_u_belief, P.pred_dump = d->pred_dump, P.belief_dump = d->belief_dump, P.env_offset = d->env_offset;
        for (int r = 0; r < 10; ++r) {
            P.rk[2 * r] = (uint32_t)d->seed + (uint32_t)r * 0x9E3779B9u;
            P.rk[2 * r + 1] = (uint32_t)(d->seed >> 32) + (uint32_t)r * 0xBB67AE85u;
        }
    }
    switch (d->M) {
        case 2: return launch_pairs_episode_seats<2>(P, runs, f, s);
        case 3: return launch_pairs_episode_seats<3>(P, runs, f, s);
        case 4: return launch_pairs_episode_seats<4>(P, runs, f, s);
        case 5: return launch_pairs_episode_seats<5>(P, runs, f, s);
        default: return launch_pairs_episode_seats<6>(P, runs, f, s);
    }
}
#endif
