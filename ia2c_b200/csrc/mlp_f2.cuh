// mlp_f2.cuh — the 6-wide actor/critic MLP on Blackwell's packed fp32 pipe (FFMA2, `fma.rn.f32x2`).
//
// Replaces NeuralNet.forward and autograd through it (ac_nets.py:34-41,71,118) in the hot kernels.
// hidden_size = 6 (ac_nets.py:24) rules tensor cores out, and the profiles show the kernels bound by the
// ISSUE rate of the fma pipe, not by its lanes (profiles/r01_ncu_full_summary.md).  sm_100 has a packed
// instruction that performs two independent IEEE fp32 FMAs per issue and takes a scalar operand as a
// broadcast, so every 6x6 layer becomes 18 FFMA2 instead of 36 FFMA:
//   forward   : outputs in pairs (j, j+1)      acc2[p]   = fma2(W^T-pairs[f][p], x[f],   acc2[p])
//   dL/dinput : inputs in pairs  (k, k+1)      dx2[q]    = fma2(W-row-pairs[o][q], dy[o], dx2[q])
//   dL/dW     : row-major pairs  (k, k+1)      gW2[o][q] = fma2(x-pairs[q],       dy[o], gW2[o][q])
// Each fp32 result is produced by the same sequence of roundings as the scalar code (bias first, then the
// inputs in ascending order), so outputs are bit-identical to the scalar kernels.
//
// Flat parameter layout (MlpDims<6,O>): every block starts at an even offset and rows are 6 wide, so the
// gradient accumulators are simply float2 views of the flat gradient vector.
#pragma once

#include "common.cuh"

namespace ia2c {

constexpr int kIn = IA2C_OBS_FEATURES;   // 6
static_assert(kIn == 6 && H == 6, "mlp_f2 assumes the reference's 6-wide layers");

__device__ __forceinline__ float2 bcast(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 relu2(float2 v) { return make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)); }

template <int O>
struct F2 {
    static constexpr int OP = (O + 1) / 2;          // output pairs of the last layer (last one half-used if O is odd)
    static constexpr int P = MlpDims<kIn, O>::P;
    static constexpr int G2 = (P + 1 + 1) / 2;      // float2 accumulators covering P gradient entries + the loss slot
};

// ------------------------------------------------------------------ register-resident forward (rollout)
template <int O>
struct RegNet {
    float2 w1[kIn][3], b1[3], w2[H][3], b2[3], w3[H][F2<O>::OP], b3[F2<O>::OP];
};

template <int O>
__device__ __forceinline__ void load_regnet(RegNet<O>& R, const float* __restrict__ flat) {
    using D = MlpDims<kIn, O>;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        R.b1[p] = make_float2(flat[D::b1 + 2 * p], flat[D::b1 + 2 * p + 1]);
        R.b2[p] = make_float2(flat[D::b2 + 2 * p], flat[D::b2 + 2 * p + 1]);
#pragma unroll
        for (int f = 0; f < kIn; ++f) {
            R.w1[f][p] = make_float2(flat[D::w1 + (2 * p) * kIn + f], flat[D::w1 + (2 * p + 1) * kIn + f]);
            R.w2[f][p] = make_float2(flat[D::w2 + (2 * p) * H + f], flat[D::w2 + (2 * p + 1) * H + f]);
        }
    }
#pragma unroll
    for (int p = 0; p < F2<O>::OP; ++p) {
        const bool two = 2 * p + 1 < O;
        R.b3[p] = make_float2(flat[D::b3 + 2 * p], two ? flat[D::b3 + 2 * p + 1] : 0.f);
#pragma unroll
        for (int k = 0; k < H; ++k)
            R.w3[k][p] = make_float2(flat[D::w3 + (2 * p) * H + k], two ? flat[D::w3 + (2 * p + 1) * H + k] : 0.f);
    }
}

template <int O>
__device__ __forceinline__ void forward_regnet(const RegNet<O>& R, const float (&x)[kIn], float2 (&h1)[3], float2 (&h2)[3],
                                               float (&y)[O]) {
    float2 yo[F2<O>::OP];
#pragma unroll
    for (int p = 0; p < 3; ++p) h1[p] = R.b1[p];
#pragma unroll
    for (int f = 0; f < kIn; ++f)
#pragma unroll
        for (int p = 0; p < 3; ++p) h1[p] = __ffma2_rn(R.w1[f][p], bcast(x[f]), h1[p]);
#pragma unroll
    for (int p = 0; p < 3; ++p) { h1[p] = relu2(h1[p]); h2[p] = R.b2[p]; }
#pragma unroll
    for (int k = 0; k < H; ++k)
#pragma unroll
        for (int p = 0; p < 3; ++p) h2[p] = __ffma2_rn(R.w2[k][p], bcast((k & 1) ? h1[k / 2].y : h1[k / 2].x), h2[p]);
#pragma unroll
    for (int p = 0; p < 3; ++p) h2[p] = relu2(h2[p]);
#pragma unroll
    for (int p = 0; p < F2<O>::OP; ++p) yo[p] = R.b3[p];
#pragma unroll
    for (int k = 0; k < H; ++k)
#pragma unroll
        for (int p = 0; p < F2<O>::OP; ++p) yo[p] = __ffma2_rn(R.w3[k][p], bcast((k & 1) ? h2[k / 2].y : h2[k / 2].x), yo[p]);
#pragma unroll
    for (int o = 0; o < O; ++o) y[o] = (o & 1) ? yo[o / 2].y : yo[o / 2].x;
}

template <int O>
__device__ __forceinline__ void forward_regnet(const RegNet<O>& R, const float (&x)[kIn], float (&y)[O]) {
    float2 h1[3], h2[3];
    forward_regnet<O>(R, x, h1, h2, y);
}

// ------------------------------------------------------------------ shared-memory weights (gradient kernels)
// Staged layout (floats).  Forward blocks are [input][output pair] float2, each input's pairs padded to a
// multiple of two float2 so a row is fetched with 128-bit loads; backward blocks are the natural rows padded
// to 8 floats.
template <int O>
struct SmemNet {
    static constexpr int OP = F2<O>::OP;
    static constexpr int OPP = (OP + 1) / 2 * 2;                  // pairs per input row, padded even
    static constexpr int w1f = 0;                                 // [6][4] float2
    static constexpr int b1f = w1f + kIn * 8;                     // [4] float2 (3 used)
    static constexpr int w2f = b1f + 8;                           // [6][4] float2
    static constexpr int b2f = w2f + H * 8;
    static constexpr int w3f = b2f + 8;                           // [6][OPP] float2
    static constexpr int b3f = w3f + H * OPP * 2;                 // [OPP] float2
    static constexpr int w2b = b3f + OPP * 2;                     // [6][8] natural rows (dL/dh1)
    static constexpr int w3b = w2b + H * 8;                       // [O][8] natural rows (dL/dh2)
    static constexpr int size = w3b + O * 8;
};

template <int O>
__device__ __forceinline__ void stage_smemnet(float* sw, const float* __restrict__ flat) {
    using L = SmemNet<O>;
    using D = MlpDims<kIn, O>;
    for (int i = threadIdx.x; i < L::size; i += blockDim.x) {
        float v = 0.f;
        if (i < L::b1f) {                      // w1f[f][p].{x,y} = W1[2p + {0,1}][f]
            const int f = i / 8, c = i % 8, j = c;       // c = 2p + half
            if (j < H) v = flat[D::w1 + j * kIn + f];
        } else if (i < L::w2f) {
            const int j = i - L::b1f;
            if (j < H) v = flat[D::b1 + j];
        } else if (i < L::b2f) {
            const int r = i - L::w2f, k = r / 8, j = r % 8;
            if (j < H) v = flat[D::w2 + j * H + k];
        } else if (i < L::w3f) {
            const int j = i - L::b2f;
            if (j < H) v = flat[D::b2 + j];
        } else if (i < L::b3f) {
            const int r = i - L::w3f, k = r / (L::OPP * 2), o = r % (L::OPP * 2);
            if (o < O) v = flat[D::w3 + o * H + k];
        } else if (i < L::w2b) {
            const int o = i - L::b3f;
            if (o < O) v = flat[D::b3 + o];
        } else if (i < L::w3b) {
            const int r = i - L::w2b, j = r / 8, k = r % 8;
            if (k < H) v = flat[D::w2 + j * H + k];
        } else {
            const int r = i - L::w3b, o = r / 8, k = r % 8;
            if (k < H) v = flat[D::w3 + o * H + k];
        }
        sw[i] = v;
    }
}

__device__ __forceinline__ void lds_pairs4(const float* p, float2 (&r)[4]) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    const float4 b = *reinterpret_cast<const float4*>(p + 4);
    r[0] = make_float2(a.x, a.y); r[1] = make_float2(a.z, a.w); r[2] = make_float2(b.x, b.y); r[3] = make_float2(b.z, b.w);
}
__device__ __forceinline__ float half_of(const float2 (&v)[3], int k) { return (k & 1) ? v[k / 2].y : v[k / 2].x; }

// Forward of one input; h1/h2 are kept as pairs (post-ReLU) for the backward pass.
template <int O>
__device__ __forceinline__ void fwd_f2(const float* sw, const float (&x)[kIn], float2 (&h1)[3], float2 (&h2)[3],
                                       float (&y)[O]) {
    using L = SmemNet<O>;
    float2 r[4];
    lds_pairs4(sw + L::b1f, r);
#pragma unroll
    for (int p = 0; p < 3; ++p) h1[p] = r[p];
#pragma unroll
    for (int f = 0; f < kIn; ++f) {
        lds_pairs4(sw + L::w1f + f * 8, r);
#pragma unroll
        for (int p = 0; p < 3; ++p) h1[p] = __ffma2_rn(r[p], bcast(x[f]), h1[p]);
    }
    lds_pairs4(sw + L::b2f, r);
#pragma unroll
    for (int p = 0; p < 3; ++p) { h1[p] = relu2(h1[p]); h2[p] = r[p]; }
#pragma unroll
    for (int k = 0; k < H; ++k) {
        lds_pairs4(sw + L::w2f + k * 8, r);
#pragma unroll
        for (int p = 0; p < 3; ++p) h2[p] = __ffma2_rn(r[p], bcast(half_of(h1, k)), h2[p]);
    }
#pragma unroll
    for (int p = 0; p < 3; ++p) h2[p] = relu2(h2[p]);
    float2 yo[L::OPP];
#pragma unroll
    for (int p = 0; p < L::OPP; p += 2) {
        const float4 b = *reinterpret_cast<const float4*>(sw + L::b3f + 2 * p);
        yo[p] = make_float2(b.x, b.y);
        yo[p + 1] = make_float2(b.z, b.w);
    }
#pragma unroll
    for (int k = 0; k < H; ++k) {
#pragma unroll
        for (int p = 0; p < L::OPP; p += 2) {
            const float4 wv = *reinterpret_cast<const float4*>(sw + L::w3f + (k * L::OPP + p) * 2);
            yo[p] = __ffma2_rn(make_float2(wv.x, wv.y), bcast(half_of(h2, k)), yo[p]);
            if (p + 1 < L::OP) yo[p + 1] = __ffma2_rn(make_float2(wv.z, wv.w), bcast(half_of(h2, k)), yo[p + 1]);
        }
    }
#pragma unroll
    for (int o = 0; o < O; ++o) y[o] = (o & 1) ? yo[o / 2].y : yo[o / 2].x;
}

// Backward of one input: dy(o) = dL/d(pre-softmax output o).  g2 is the float2 view of the flat gradient
// (MlpDims<6,O> layout).  x2 = the input as pairs.
template <int O, typename DY, int GN>
__device__ __forceinline__ void bwd_f2(const float* sw, const float (&x)[kIn], const float2 (&h1)[3],
                                       const float2 (&h2)[3], DY dy, float2 (&g2)[GN]) {
    using L = SmemNet<O>;
    using D = MlpDims<kIn, O>;
    static_assert(GN * 2 >= D::P, "gradient accumulator too small");
    float2 dh2[3], dh1[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) dh2[q] = dh1[q] = make_float2(0.f, 0.f);
#pragma unroll
    for (int o = 0; o < O; ++o) {
        const float dyv = dy(o);
        float2 r[4];
        lds_pairs4(sw + L::w3b + o * 8, r);
        // b3 gradient: entry D::b3 + o of the flat vector
        if (((D::b3 + o) & 1) == 0) g2[(D::b3 + o) / 2].x += dyv; else g2[(D::b3 + o) / 2].y += dyv;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            g2[(D::w3 + o * H) / 2 + q] = __ffma2_rn(h2[q], bcast(dyv), g2[(D::w3 + o * H) / 2 + q]);
            dh2[q] = __ffma2_rn(r[q], bcast(dyv), dh2[q]);
        }
    }
    float2 dz2[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        dz2[q] = make_float2(h2[q].x > 0.f ? dh2[q].x : 0.f, h2[q].y > 0.f ? dh2[q].y : 0.f);
        g2[D::b2 / 2 + q].x += dz2[q].x;
        g2[D::b2 / 2 + q].y += dz2[q].y;
    }
#pragma unroll
    for (int j = 0; j < H; ++j) {
        const float dz = half_of(dz2, j);
        float2 r[4];
        lds_pairs4(sw + L::w2b + j * 8, r);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            g2[(D::w2 + j * H) / 2 + q] = __ffma2_rn(h1[q], bcast(dz), g2[(D::w2 + j * H) / 2 + q]);
            dh1[q] = __ffma2_rn(r[q], bcast(dz), dh1[q]);
        }
    }
    float2 dz1[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        dz1[q] = make_float2(h1[q].x > 0.f ? dh1[q].x : 0.f, h1[q].y > 0.f ? dh1[q].y : 0.f);
        g2[D::b1 / 2 + q].x += dz1[q].x;
        g2[D::b1 / 2 + q].y += dz1[q].y;
    }
    const float2 x2[3] = {make_float2(x[0], x[1]), make_float2(x[2], x[3]), make_float2(x[4], x[5])};
#pragma unroll
    for (int j = 0; j < H; ++j) {
        const float dz = half_of(dz1, j);
#pragma unroll
        for (int q = 0; q < 3; ++q)
            g2[(D::w1 + j * kIn) / 2 + q] = __ffma2_rn(x2[q], bcast(dz), g2[(D::w1 + j * kIn) / 2 + q]);
    }
}

// ---- register-resident backward (fused rollout, critic-backprop stage) ------------------------------------
// Natural row pairs of W3 and W2 in registers; accumulates the W3/b3/W2/b2 gradient and hands dz1 to the stage
// that owns the W1/b1 gradient (splitting the 147 accumulators over two warps keeps both below the register
// limit WITH their weights resident, so neither waits on shared-memory loads).
template <int O>
struct RegBack {
    float2 w3[O][3], w2[H][3];
};
template <int O>
__device__ __forceinline__ void load_regback(RegBack<O>& R, const float* __restrict__ flat) {
    using D = MlpDims<kIn, O>;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
#pragma unroll
        for (int o = 0; o < O; ++o) R.w3[o][q] = make_float2(flat[D::w3 + o * H + 2 * q], flat[D::w3 + o * H + 2 * q + 1]);
#pragma unroll
        for (int j = 0; j < H; ++j) R.w2[j][q] = make_float2(flat[D::w2 + j * H + 2 * q], flat[D::w2 + j * H + 2 * q + 1]);
    }
}
// gA covers flat entries [D::w2, D::P): W2 | b2 | W3 | b3 as float2 (offset D::w2 / 2).
template <int O, typename DY, int GN>
__device__ __forceinline__ void bwd_regback(const RegBack<O>& R, const float2 (&h1)[3], const float2 (&h2)[3], DY dy,
                                            float2 (&gA)[GN], float2 (&dz1)[3]) {
    using D = MlpDims<kIn, O>;
    constexpr int base = D::w2 / 2;
    static_assert(GN >= (D::P + 1) / 2 - base, "accumulator too small");
    float2 dh2[3], dh1[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) dh2[q] = dh1[q] = make_float2(0.f, 0.f);
#pragma unroll
    for (int o = 0; o < O; ++o) {
        const float dyv = dy(o);
        if (((D::b3 + o) & 1) == 0) gA[(D::b3 + o) / 2 - base].x += dyv; else gA[(D::b3 + o) / 2 - base].y += dyv;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            gA[(D::w3 + o * H) / 2 + q - base] = __ffma2_rn(h2[q], bcast(dyv), gA[(D::w3 + o * H) / 2 + q - base]);
            dh2[q] = __ffma2_rn(R.w3[o][q], bcast(dyv), dh2[q]);
        }
    }
    float2 dz2[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        dz2[q] = make_float2(h2[q].x > 0.f ? dh2[q].x : 0.f, h2[q].y > 0.f ? dh2[q].y : 0.f);
        gA[D::b2 / 2 + q - base].x += dz2[q].x;
        gA[D::b2 / 2 + q - base].y += dz2[q].y;
    }
#pragma unroll
    for (int j = 0; j < H; ++j) {
        const float dz = half_of(dz2, j);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            gA[(D::w2 + j * H) / 2 + q - base] = __ffma2_rn(h1[q], bcast(dz), gA[(D::w2 + j * H) / 2 + q - base]);
            dh1[q] = __ffma2_rn(R.w2[j][q], bcast(dz), dh1[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) dz1[q] = make_float2(h1[q].x > 0.f ? dh1[q].x : 0.f, h1[q].y > 0.f ? dh1[q].y : 0.f);
}
// gB covers flat entries [0, D::w2): W1 | b1.
__device__ __forceinline__ void accumulate_w1(const float (&x)[kIn], const float2 (&dz1)[3], float2 (&gB)[21]) {
    const float2 x2[3] = {make_float2(x[0], x[1]), make_float2(x[2], x[3]), make_float2(x[4], x[5])};
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        gB[18 + q].x += dz1[q].x;
        gB[18 + q].y += dz1[q].y;
    }
#pragma unroll
    for (int j = 0; j < H; ++j) {
        const float dz = half_of(dz1, j);
#pragma unroll
        for (int q = 0; q < 3; ++q) gB[j * 3 + q] = __ffma2_rn(x2[q], bcast(dz), gB[j * 3 + q]);
    }
}

__device__ __forceinline__ void load_obs6(const float* __restrict__ p, float (&x)[kIn]) {
    const float2* p2 = reinterpret_cast<const float2*>(p);
    const float2 a = __ldg(p2), b = __ldg(p2 + 1), c = __ldg(p2 + 2);
    x[0] = a.x; x[1] = a.y; x[2] = b.x; x[3] = b.y; x[4] = c.x; x[5] = c.y;
}

// float2 gradient accumulators -> the flat gradient vector (+ loss slot) that block_reduce_store takes
template <int GN>
__device__ __forceinline__ void unpack_g2(const float2 (&g2)[GN], float (&g)[2 * GN]) {
#pragma unroll
    for (int i = 0; i < GN; ++i) { g[2 * i] = g2[i].x; g[2 * i + 1] = g2[i].y; }
}

template <int O>
__device__ __forceinline__ float select_out(const float (&q)[O], int idx) {
    float v = 0.f;
#pragma unroll
    for (int o = 0; o < O; ++o) v = (o == idx) ? q[o] : v;
    return v;
}

// Policy table (evaluation, frozen partners per env): row idx = net * 9 + c holds net's softmax at observation class
// c = 3 * prev_cls + cur_cls, computed with the training samplers' forward and softmax, so it holds the very probabilities they
// sample from.  Loads through L2 (the rows may come from the kernels just before).
constexpr int kObsClasses = 9;
__device__ __forceinline__ void policy_row(const float* actor_params, float* policy, int64_t idx) {
    constexpr int A = IA2C_AGENT_ACTIONS;
    const int64_t net = idx / kObsClasses;
    const int c = (int)(idx - net * kObsClasses);
    float flat[kActorP];
#pragma unroll
    for (int k = 0; k < kActorP; ++k) flat[k] = __ldcg(actor_params + net * kActorP + k);
    RegNet<A> w;
    load_regnet<A>(w, flat);
    float x[kIn], y[A];
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

}  // namespace ia2c

