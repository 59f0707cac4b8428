// history.cu — learning curves on the device: one reduction of an episode's trajectory into a slot of a caller-owned ring.
//
// After an episode (standalone, or a batch of R runs in the stacked layout of ia2c_runs_desc) the trajectory buffers hold
// what the episode did: own actions, the partner's true and belief-predicted actions, the per-env returns and the losses.
// The next episode overwrites them.  ia2c_record_episode reduces them, in ONE launch, into slot s of a ring that the host
// drains once every many episodes (include/ia2c_b200.h states the definitions).
//
// Kernel in this file
//   record_episode_kernel   grid (row blocks + 1, R, ceil(N / 256)), 256 threads.  Block (x, r, z) covers agents
//                           [256 z, 256 z + W) of run r, W = min(256, N - 256 z), and rows q = t * E + e in
//                           [x * B, (x + 1) * B) of the run's T * E (step, env) rows, B = (256 / min(N, 256)) * kIter * loops
//                           (loops chosen per launch for about 4 blocks per SM in all); G = 256 / W rows at a time
//                           (G * kIter * loops >= B): thread tid owns agent 256 z + tid % W for good and reads rows
//                           x * B + tid / W + G * k, k < kIter * loops, in batches of kIter whose loads are all in flight at
//                           once, with byte loads that a warp issues over consecutive bytes (a run's step row is E * N
//                           contiguous bytes).  Counts live in registers, are summed over the block's G threads of one
//                           agent in shared memory, and reach the slot with one u32 atomicAdd per (agent, field) and block
//                           (integer sums: the same in any order).
//                           The last block column, block (row blocks, r, 0), writes run r's fixed-order return sum and its
//                           loss rows into slot s and zeroes run r's counts and hits in slot (s + 1) mod capacity, so that
//                           the next call needs no memset; it runs alongside the counting blocks.
#include <algorithm>

#include "common.cuh"

namespace ia2c {
namespace {

constexpr int A = IA2C_AGENT_ACTIONS;
constexpr int kThreads = 256;       // also the lane count of the fixed-order return sum (the header's definition)
constexpr int kIter = 8;            // rows per thread and block, all loads in flight at once
constexpr int kFields = A + 1;      // three action counts, then the partner hits
constexpr int kRetBatch = 16;
constexpr int64_t kTargetBlocks = 4 * kSMs;   // counting blocks of one launch, before rounding       // returns per lane loaded at once: E = 4096 is one round trip

struct RecordArgs {
    const uint8_t *act, *ptrue, *ppred;   // u8[T+1, R*E, N]
    const double* ep_return;              // f64[R*E]
    const float* loss_out;                // f32[2, R*N]
    double* return_sum;                   // slot s of f64[capacity, R]
    float* loss;                          // slot s of f32[capacity, 2, R*N]
    uint32_t *counts, *hits;              // slot s of u32[capacity, R*N, 3] / u32[capacity, R*N]
    uint32_t *next_counts, *next_hits;    // slot (s + 1) mod capacity of the same
    int64_t E;
    int32_t N, T, R;
    uint64_t rows_per_block;              // (256 / min(N, 256)) * kIter * loops: the rows of block x are [x, x + 1) * rows_per_block
    uint32_t loops;                       // batches of kIter rows per thread
};

// Run-level outputs of run `run`: the fixed-order return sum, the loss rows, and the next slot's counters zeroed.
__device__ __forceinline__ void record_run(const RecordArgs& a, int run) {
    __shared__ double lane_sum[kThreads];
    const int tid = threadIdx.x, N = a.N;
    const double* ret = a.ep_return + (int64_t)run * a.E;
    double s = 0.0;
    for (int64_t e0 = tid; e0 < a.E; e0 += (int64_t)kRetBatch * kThreads) {   // kRetBatch loads in flight, then the adds in order
        double v[kRetBatch];
#pragma unroll
        for (int k = 0; k < kRetBatch; ++k) {
            const int64_t e = e0 + (int64_t)k * kThreads;
            v[k] = e < a.E ? __ldcg(ret + e) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < kRetBatch; ++k)
            if (e0 + (int64_t)k * kThreads < a.E) s = __dadd_rn(s, v[k]);
    }
    lane_sum[tid] = s;
    __syncthreads();
#pragma unroll
    for (int w = kThreads / 2; w > 0; w >>= 1) {
        if (tid < w) lane_sum[tid] = __dadd_rn(lane_sum[tid], lane_sum[tid + w]);
        __syncthreads();
    }
    if (tid == 0) a.return_sum[run] = lane_sum[0];
    const int64_t RN = (int64_t)a.R * N, n0 = (int64_t)run * N;
    for (int i = tid; i < N; i += kThreads) {
        a.loss[n0 + i] = __ldcg(a.loss_out + n0 + i);
        a.loss[RN + n0 + i] = __ldcg(a.loss_out + RN + n0 + i);
        a.next_hits[n0 + i] = 0u;
    }
    for (int i = tid; i < N * A; i += kThreads) a.next_counts[n0 * A + i] = 0u;
}

__global__ void __launch_bounds__(kThreads) record_episode_kernel(const __grid_constant__ RecordArgs a) {
    __shared__ uint32_t part[kFields][kThreads];
    pdl_prologue();   // every buffer read here is written by the episode's kernels just before: L2 path, after the wait
    const int tid = threadIdx.x, run = blockIdx.y, N = a.N;
    if (blockIdx.x == gridDim.x - 1) {   // the last block column: run-level outputs, alongside the counting blocks
        if (blockIdx.z == 0) record_run(a, run);
        return;
    }
    const int a0 = blockIdx.z * kThreads, W = min(kThreads, N - a0), G = kThreads / W;
    const int col = tid % W, roff = tid / W;
    const uint32_t E = (uint32_t)a.E, rows = (uint32_t)a.T * E;
    const int64_t step = (int64_t)a.R * a.E * N;                   // bytes per step row of all runs
    const int64_t base = (int64_t)run * a.E * N + a0 + col;        // agent a0 + col of env 0 of this run at step 0
    uint32_t c[kFields] = {0u, 0u, 0u, 0u};
    if (roff < G) {   // G * kIter * loops >= rows_per_block: every chunk covers the block's rows
        const uint64_t q0 = (uint64_t)blockIdx.x * a.rows_per_block, q_end = min((uint64_t)rows, q0 + a.rows_per_block);
        for (uint32_t l = 0; l < a.loops; ++l) {
            uint8_t act[kIter], pt[kIter], pp[kIter];
#pragma unroll
            for (int k = 0; k < kIter; ++k) {
                const uint64_t q = q0 + (uint64_t)roff + (uint64_t)G * (l * kIter + k);
                act[k] = A, pt[k] = 0, pp[k] = 1;   // a row past the block's end counts nothing
                if (q < q_end) {
                    const uint32_t t = (uint32_t)q / E, e = (uint32_t)q - t * E;
                    const int64_t off = (int64_t)t * step + base + (int64_t)e * N;
                    act[k] = __ldcg(a.act + off);
                    pt[k] = __ldcg(a.ptrue + off);
                    pp[k] = __ldcg(a.ppred + off);
                }
            }
#pragma unroll
            for (int k = 0; k < kIter; ++k) {
                c[0] += act[k] == 0;
                c[1] += act[k] == 1;
                c[2] += act[k] == 2;
                c[3] += pt[k] == pp[k];
            }
        }
    }
#pragma unroll
    for (int f = 0; f < kFields; ++f) part[f][tid] = c[f];
    __syncthreads();
    for (int j = tid; j < kFields * W; j += kThreads) {   // per (field, agent): the G partial counts, in row-offset order
        const int f = j / W, i = j - f * W;
        uint32_t s = 0u;
        for (int g = 0; g < G; ++g) s += part[f][g * W + i];
        const int64_t net = (int64_t)run * N + a0 + i;
        if (s) atomicAdd(f < A ? a.counts + net * A + f : a.hits + net, s);
    }
}

int validate_record(const ia2c_episode_desc* d, int32_t runs, const ia2c_history_desc* h, int32_t slot) {
    const char* who = "ia2c_record_episode";
    IA2C_REQUIRE(d != nullptr && h != nullptr, "%s: null episode or history descriptor", who);
    IA2C_REQUIRE(d->act && d->partner_true && d->partner_pred && d->ep_return && d->loss_out,
                 "%s: null act / partner_true / partner_pred / ep_return / loss_out pointer", who);
    IA2C_REQUIRE(h->return_sum && h->loss && h->action_counts && h->partner_hits,
                 "%s: null return_sum / loss / action_counts / partner_hits pointer", who);
    IA2C_REQUIRE(runs >= 1, "%s: runs=%d must be >= 1", who, runs);
    IA2C_REQUIRE(d->N >= 1 && d->T >= 1 && d->E >= 1, "%s: N=%d, T=%d, E=%lld must be >= 1", who, d->N, d->T, (long long)d->E);
    IA2C_REQUIRE((int64_t)runs * d->N <= IA2C_MAX_RUN_NETS, "%s: runs * N = %lld above IA2C_MAX_RUN_NETS (%d)", who,
                 (long long)runs * d->N, IA2C_MAX_RUN_NETS);
    IA2C_REQUIRE(h->capacity >= 2, "%s: capacity=%d must be >= 2 (the call clears the slot after its own)", who, h->capacity);
    IA2C_REQUIRE(slot >= 0 && slot < h->capacity, "%s: slot=%d outside [0, capacity=%d)", who, slot, h->capacity);
    if (d->env_offset != 0 || d->E_total != d->E) {
        set_error("%s: env_offset=%lld, E_total=%lld, E=%lld: histories are recorded on one GPU (env_offset 0, E_total = E)", who,
                  (long long)d->env_offset, (long long)d->E_total, (long long)d->E);
        return IA2C_ERR_UNSUPPORTED;
    }
    IA2C_REQUIRE((uint64_t)d->T * (uint64_t)d->E < (1ull << 32), "%s: T * E = %llu not below 2^32 (u32 counts)", who,
                 (unsigned long long)d->T * (unsigned long long)d->E);
    return 0;
}

}  // namespace
}  // namespace ia2c

using namespace ia2c;

extern "C" int ia2c_record_episode(const ia2c_episode_desc* d, int32_t runs, const ia2c_history_desc* h, int32_t slot,
                                   void* stream) {
    if (int rc = validate_record(d, runs, h, slot)) return rc;
    const int64_t RN = (int64_t)runs * d->N;
    const int32_t next = (slot + 1) % h->capacity;
    RecordArgs a;
    a.act = d->act, a.ptrue = d->partner_true, a.ppred = d->partner_pred;
    a.ep_return = d->ep_return, a.loss_out = d->loss_out;
    a.return_sum = h->return_sum + (int64_t)slot * runs;
    a.loss = h->loss + (int64_t)slot * 2 * RN;
    a.counts = h->action_counts + (int64_t)slot * RN * A, a.hits = h->partner_hits + (int64_t)slot * RN;
    a.next_counts = h->action_counts + (int64_t)next * RN * A, a.next_hits = h->partner_hits + (int64_t)next * RN;
    a.E = d->E, a.N = d->N, a.T = d->T, a.R = runs;
    // Few enough blocks that the counters see a few atomics per block and agent, not one per 8 rows: about kTargetBlocks in
    // all, each thread then reading `loops` batches of kIter rows.
    const int64_t rows = (int64_t)d->T * d->E, chunks = ceil_div(d->N, kThreads);
    const int64_t batch = (int64_t)(kThreads / (d->N < kThreads ? d->N : kThreads)) * kIter;   // rows of one batch of a block
    const int64_t per_chunk = std::max<int64_t>(1, kTargetBlocks / (runs * chunks));
    a.loops = (uint32_t)std::max<int64_t>(1, ceil_div(rows, batch * per_chunk));
    a.rows_per_block = (uint64_t)batch * a.loops;
    const dim3 grid((unsigned)ceil_div(rows, a.rows_per_block) + 1, (unsigned)runs, (unsigned)chunks);
    return launch_pdl("record_episode_kernel", record_episode_kernel, grid, dim3(kThreads), 0, as_stream(stream), a);
}
