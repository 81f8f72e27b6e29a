// mlp_kernels.cuh -- SURVEY section 8 row f-1: the tiny decoder MLP that consumes the grid features, fused with
// the image loss: forward, MSE, backward to the features AND all weight gradients in ONE pass over the points.
//
// Reference: NeuralImage.rgb -> BasicDecoder (wisp/models/nefs/image.py:109-120,152; hidden 16, two hidden layers,
// ReLU, bias; wisp/models/decoders/basic_decoders.py:60-100) followed by ((pred - gt)**2).mean()
// (wisp/trainers/image_trainer.py:298-300). In PyTorch that is ~15 kernels per step, each streaming an
// [N, 16] activation through HBM/L2; here the activations never leave registers / shared memory:
// per point 64 B features in, 12 B target in, 64 B feature gradient out (+12 B prediction when asked for).
//
//   y  = W3 relu(W2 relu(W1 x + b1) + b2) + b3            (torch.nn.Linear layout: W[out][in])
//   L  = sum((y - gt)^2) / (N * OUT)
//
// One lane owns one point for forward + backward (weights broadcast from shared memory as 16-byte vectors);
// the weight gradients dW = sum_p a_p b_p^T are formed per warp from the 32 points' activations staged in shared
// memory, each lane accumulating an 8-wide slice in registers across ALL its warp's points (persistent CTAs),
// then reduced over the block in shared memory and added to global memory once per CTA and value.
#pragma once
#include "common.cuh"
#include "mlp_tc_common.cuh"

namespace shacira {

constexpr int kMlpThreads = 256;
constexpr int kMlpWarps = kMlpThreads / 32;

template <int IN, int H, int OUT>
struct MlpSmem {
    // weights, and their transposes for the backward products (row = reduction index -> 16-byte broadcast loads)
    float W1[H][IN], W2[H][H], W3[OUT][H];
    float W1t[IN][H], W2t[H][H], W3t[H][4];  // W3t padded to 4 outputs
    float b1[H], b2[H], b3[4];
    // per-warp staging of the 32 points' activations for the weight-gradient products
    float x[kMlpWarps][32][IN + 4];
    float h1[kMlpWarps][32][H + 4], h2[kMlpWarps][32][H + 4];
    float d1[kMlpWarps][32][H + 4], d2[kMlpWarps][32][H + 4];
    float dy[kMlpWarps][32][4];
    // block reduction of the per-warp gradient slices
    float gW1[H * IN], gW2[H * H], gW3[OUT * H], gb1[H], gb2[H], gb3[4];
    double loss;
};

template <int IN, int H, int OUT>
__global__ void __launch_bounds__(kMlpThreads, 2)
mlp_mse_step_kernel(const float* __restrict__ x, const float* __restrict__ gt, int64_t n, const float* __restrict__ W1,
                    const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                    const float* __restrict__ W3, const float* __restrict__ b3, float grad_scale /* 2 / (N*OUT) */,
                    float* __restrict__ gx, float* __restrict__ pred, double* __restrict__ loss_sum,
                    float* __restrict__ grad_params) {
    // packed gradient buffer: W1 [H][IN] | b1 [H] | W2 [H][H] | b2 [H] | W3 [OUT][H] | b3 [OUT]
    float* gW1 = grad_params;
    float* gb1 = gW1 + H * IN;
    float* gW2 = gb1 + H;
    float* gb2 = gW2 + H * H;
    float* gW3 = gb2 + H;
    float* gb3 = gW3 + OUT * H;
    static_assert(IN % 8 == 0 && H == 16 && OUT <= 4, "shape");
    extern __shared__ __align__(16) unsigned char s_raw[];
    MlpSmem<IN, H, OUT>& S = *reinterpret_cast<MlpSmem<IN, H, OUT>*>(s_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < H * IN; e += kMlpThreads) {
        const float w = W1[e];
        S.W1[e / IN][e % IN] = w;
        S.W1t[e % IN][e / IN] = w;
        S.gW1[e] = 0.0f;
    }
    for (int e = tid; e < H * H; e += kMlpThreads) {
        const float w = W2[e];
        S.W2[e / H][e % H] = w;
        S.W2t[e % H][e / H] = w;
        S.gW2[e] = 0.0f;
    }
    for (int e = tid; e < H * 4; e += kMlpThreads) S.W3t[e / 4][e % 4] = 0.0f;
    __syncthreads();
    for (int e = tid; e < OUT * H; e += kMlpThreads) {
        const float w = W3[e];
        S.W3[e / H][e % H] = w;
        S.W3t[e % H][e / H] = w;
        S.gW3[e] = 0.0f;
    }
    if (tid < H) { S.b1[tid] = b1[tid]; S.b2[tid] = b2[tid]; S.gb1[tid] = 0.0f; S.gb2[tid] = 0.0f; }
    if (tid < 4) { S.b3[tid] = tid < OUT ? b3[tid] : 0.0f; S.gb3[tid] = 0.0f; }
    if (tid == 0) S.loss = 0.0;
    __syncthreads();

    // register slices of the weight gradients owned by this lane (summed over all points of this warp)
    //   dW1[i][m0..m0+IN/2)  i = lane/2, m0 = (lane&1) * IN/2         (H*IN/32 values per lane)
    //   dW2[i][j0..j0+8)     i = lane/2, j0 = (lane&1) * 8
    //   dW3[k][j]            lanes < OUT*H/2 own two values; biases: lane < H owns db1[lane], db2[lane]; lane < OUT db3
    constexpr int S1 = IN / 2;
    float aW1[S1], aW2[8], aW3[2] = {0.0f, 0.0f}, ab1 = 0.0f, ab2 = 0.0f, ab3 = 0.0f;
#pragma unroll
    for (int e = 0; e < S1; ++e) aW1[e] = 0.0f;
#pragma unroll
    for (int e = 0; e < 8; ++e) aW2[e] = 0.0f;
    float my_loss = 0.0f;
    const int wi = lane >> 1, wj0 = (lane & 1) * 8, wm0 = (lane & 1) * S1;

    const int64_t warps_total = (int64_t)gridDim.x * kMlpWarps;
    for (int64_t base = ((int64_t)blockIdx.x * kMlpWarps + warp) * 32; base < n; base += warps_total * 32) {
        const int64_t p = base + lane;
        const bool live = p < n;
        float xi[IN], h1[H], h2[H], y[4] = {0.0f, 0.0f, 0.0f, 0.0f}, tgt[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int e = 0; e < IN; ++e) xi[e] = 0.0f;
        if (live) {
#pragma unroll
            for (int q = 0; q < IN / 4; ++q) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(x + p * IN) + q);
                xi[4 * q] = v.x; xi[4 * q + 1] = v.y; xi[4 * q + 2] = v.z; xi[4 * q + 3] = v.w;
            }
#pragma unroll
            for (int k = 0; k < OUT; ++k) tgt[k] = __ldg(gt + p * OUT + k);
        }
        // ---- forward ----
#pragma unroll
        for (int i = 0; i < H; ++i) {
            float acc = S.b1[i];
#pragma unroll
            for (int q = 0; q < IN / 4; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(&S.W1[i][4 * q]);
                acc = fmaf(xi[4 * q], w.x, acc); acc = fmaf(xi[4 * q + 1], w.y, acc);
                acc = fmaf(xi[4 * q + 2], w.z, acc); acc = fmaf(xi[4 * q + 3], w.w, acc);
            }
            h1[i] = fmaxf(acc, 0.0f);
        }
#pragma unroll
        for (int j = 0; j < H; ++j) {
            float acc = S.b2[j];
#pragma unroll
            for (int q = 0; q < H / 4; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(&S.W2[j][4 * q]);
                acc = fmaf(h1[4 * q], w.x, acc); acc = fmaf(h1[4 * q + 1], w.y, acc);
                acc = fmaf(h1[4 * q + 2], w.z, acc); acc = fmaf(h1[4 * q + 3], w.w, acc);
            }
            h2[j] = fmaxf(acc, 0.0f);
        }
#pragma unroll
        for (int k = 0; k < OUT; ++k) {
            float acc = S.b3[k];
#pragma unroll
            for (int q = 0; q < H / 4; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(&S.W3[k][4 * q]);
                acc = fmaf(h2[4 * q], w.x, acc); acc = fmaf(h2[4 * q + 1], w.y, acc);
                acc = fmaf(h2[4 * q + 2], w.z, acc); acc = fmaf(h2[4 * q + 3], w.w, acc);
            }
            y[k] = acc;
        }
        // ---- loss and its gradient ----
        float dy[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (live) {
#pragma unroll
            for (int k = 0; k < OUT; ++k) {
                const float e = y[k] - tgt[k];
                my_loss = fmaf(e, e, my_loss);
                dy[k] = e * grad_scale;
                if (pred) pred[p * OUT + k] = y[k];
            }
        }
        // ---- backward to the features ----
        float d2[H], d1[H];
#pragma unroll
        for (int j = 0; j < H; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(&S.W3t[j][0]);
            float acc = dy[0] * w.x;
            acc = fmaf(dy[1], w.y, acc); acc = fmaf(dy[2], w.z, acc); acc = fmaf(dy[3], w.w, acc);
            d2[j] = h2[j] > 0.0f ? acc : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < H; ++i) {
            float acc = 0.0f;
#pragma unroll
            for (int q = 0; q < H / 4; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(&S.W2t[i][4 * q]);  // W2[j][i], j = 4q..
                acc = fmaf(d2[4 * q], w.x, acc); acc = fmaf(d2[4 * q + 1], w.y, acc);
                acc = fmaf(d2[4 * q + 2], w.z, acc); acc = fmaf(d2[4 * q + 3], w.w, acc);
            }
            d1[i] = h1[i] > 0.0f ? acc : 0.0f;
        }
        if (live) {
#pragma unroll
            for (int q = 0; q < IN / 4; ++q) {
                float o[4];
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int m = 4 * q + r;
                    float acc = 0.0f;
#pragma unroll
                    for (int qq = 0; qq < H / 4; ++qq) {
                        const float4 w = *reinterpret_cast<const float4*>(&S.W1t[m][4 * qq]);  // W1[i][m], i = 4qq..
                        acc = fmaf(d1[4 * qq], w.x, acc); acc = fmaf(d1[4 * qq + 1], w.y, acc);
                        acc = fmaf(d1[4 * qq + 2], w.z, acc); acc = fmaf(d1[4 * qq + 3], w.w, acc);
                    }
                    o[r] = acc;
                }
                reinterpret_cast<float4*>(gx + p * IN)[q] = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
        // ---- weight gradients: stage this warp's 32 points, every lane accumulates its slice ----
        __syncwarp();
        // 16-byte stores, row stride (IN|H)+4 floats = 20 banks: a quarter-warp covers all 32 banks, no conflicts
#pragma unroll
        for (int q = 0; q < IN / 4; ++q)
            *reinterpret_cast<float4*>(&S.x[warp][lane][4 * q]) = make_float4(xi[4 * q], xi[4 * q + 1], xi[4 * q + 2], xi[4 * q + 3]);
#pragma unroll
        for (int q = 0; q < H / 4; ++q) {
            *reinterpret_cast<float4*>(&S.h1[warp][lane][4 * q]) = make_float4(h1[4 * q], h1[4 * q + 1], h1[4 * q + 2], h1[4 * q + 3]);
            *reinterpret_cast<float4*>(&S.h2[warp][lane][4 * q]) = make_float4(h2[4 * q], h2[4 * q + 1], h2[4 * q + 2], h2[4 * q + 3]);
            *reinterpret_cast<float4*>(&S.d1[warp][lane][4 * q]) = make_float4(d1[4 * q], d1[4 * q + 1], d1[4 * q + 2], d1[4 * q + 3]);
            *reinterpret_cast<float4*>(&S.d2[warp][lane][4 * q]) = make_float4(d2[4 * q], d2[4 * q + 1], d2[4 * q + 2], d2[4 * q + 3]);
        }
        *reinterpret_cast<float4*>(&S.dy[warp][lane][0]) = make_float4(dy[0], dy[1], dy[2], dy[3]);
        __syncwarp();
#pragma unroll 4
        for (int q = 0; q < 32; ++q) {
            const float d1q = S.d1[warp][q][wi];   // dW1[i][m] += d1[i] * x[m]
#pragma unroll
            for (int e = 0; e < S1; e += 4) {
                const float4 v = *reinterpret_cast<const float4*>(&S.x[warp][q][wm0 + e]);
                aW1[e] = fmaf(d1q, v.x, aW1[e]); aW1[e + 1] = fmaf(d1q, v.y, aW1[e + 1]);
                aW1[e + 2] = fmaf(d1q, v.z, aW1[e + 2]); aW1[e + 3] = fmaf(d1q, v.w, aW1[e + 3]);
            }
            const float d2q = S.d2[warp][q][wi];   // dW2[j][i'] += d2[j] * h1[i'] : row j = wi, columns wj0..wj0+8
#pragma unroll
            for (int e = 0; e < 8; e += 4) {
                const float4 v = *reinterpret_cast<const float4*>(&S.h1[warp][q][wj0 + e]);
                aW2[e] = fmaf(d2q, v.x, aW2[e]); aW2[e + 1] = fmaf(d2q, v.y, aW2[e + 1]);
                aW2[e + 2] = fmaf(d2q, v.z, aW2[e + 2]); aW2[e + 3] = fmaf(d2q, v.w, aW2[e + 3]);
            }
            if (lane < OUT * H / 2) {               // dW3[k][j] += dy[k] * h2[j] : two values per lane
                const int v0 = 2 * lane, k0 = v0 / H, j0 = v0 % H;
                const float dyk = S.dy[warp][q][k0];
                aW3[0] = fmaf(dyk, S.h2[warp][q][j0], aW3[0]);
                aW3[1] = fmaf(dyk, S.h2[warp][q][j0 + 1], aW3[1]);
            }
            if (lane < H) {
                ab1 += S.d1[warp][q][lane];
                ab2 += S.d2[warp][q][lane];
            }
            if (lane < OUT) ab3 += S.dy[warp][q][lane];
        }
    }
    // ---- block reduction (shared memory, 8 warps) then one global add per CTA and value ----
#pragma unroll
    for (int e = 0; e < S1; ++e) atomicAdd(&S.gW1[wi * IN + wm0 + e], aW1[e]);
#pragma unroll
    for (int e = 0; e < 8; ++e) atomicAdd(&S.gW2[wi * H + wj0 + e], aW2[e]);
    if (lane < OUT * H / 2) {
        atomicAdd(&S.gW3[2 * lane], aW3[0]);
        atomicAdd(&S.gW3[2 * lane + 1], aW3[1]);
    }
    if (lane < H) { atomicAdd(&S.gb1[lane], ab1); atomicAdd(&S.gb2[lane], ab2); }
    if (lane < OUT) atomicAdd(&S.gb3[lane], ab3);
    const float wl = warp_sum(my_loss);
    if (lane == 0) atomicAdd(&S.loss, (double)wl);
    __syncthreads();
    for (int e = tid; e < H * IN; e += kMlpThreads) red_add(gW1 + e, S.gW1[e]);
    for (int e = tid; e < H * H; e += kMlpThreads) red_add(gW2 + e, S.gW2[e]);
    for (int e = tid; e < OUT * H; e += kMlpThreads) red_add(gW3 + e, S.gW3[e]);
    if (tid < H) { red_add(gb1 + tid, S.gb1[tid]); red_add(gb2 + tid, S.gb2[tid]); }
    if (tid < OUT) red_add(gb3 + tid, S.gb3[tid]);
    if (tid == 0) atomicAdd(loss_sum, S.loss);
}

// ---------------------------------------------------------------------------------------------------------------
// IN = 16 on the tensor cores: mma.sync m16n8k8 TF32 with 3xTF32 error compensation.
//
// Every product of the step is a small dense contraction -- forward [32 points x 16] x [16 x 16], backward the same
// with the transposed weights, weight gradients [16 x 32 points] x [32 points x 16] -- so one warp runs its 32 points
// as two m16 tiles through `mma.sync`. Operands are split a = hi + lo in TF32 and each product is issued three
// times (lo*hi + hi*lo + hi*hi, the 2^-22 lo*lo term dropped): fp32-grade results (the tests hold this kernel to the
// same 1e-5 / 1e-4 gates as the FP32 SIMT kernels) at a third of the instruction count of the FFMA formulations
// (measured: those are issue-bound, 3700 instructions per 32 points).
//
// Layout trick: the accumulator fragment of one layer (lane (g, t) holds rows g, g+8, columns 2t, 2t+1 of each
// 8-column tile) is fed straight back as the A fragment of the next product by PERMUTING THE K INDEX -- logical
// k = t is column 2t, logical k = t+4 is column 2t+1 -- and the weight fragments are built with the same permutation
// once per CTA (shared memory, one LDS.128 per fragment: {b0.hi, b1.hi, b0.lo, b1.lo}). No shuffles between layers.
// Weight gradients need the point index as K: the activations are staged per warp in shared memory ([point][24],
// conflict-free for both the fragment-layout stores and the transposed fragment loads).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kMlp16Params = 16 * 16 + 16 + 16 * 16 + 16 + 3 * 16 + 3;  // W1 | b1 | W2 | b2 | W3 | b3 (packed order)

// MT = m16 tiles (16 points each) a warp runs per iteration; WARPS per CTA. MT = 2 halves the per-point overhead
// (weight-fragment loads, loop control); MT = 1 halves the registers and the staging rows, i.e. doubles the warps
// an SM can hold. The launcher builds MT = 2 with 6 warps x 2 CTAs per SM: measured against MT = 1 (6 warps x 3 CTAs,
// 8 warps x 2 CTAs), which was then removed.
template <int MT, int WARPS>
struct MlpTcSmem {
    uint4 wf[20][32];                       // weight fragments (see the enum in the kernel)
    float b1[16], b2[16], b3[4];
    float x[WARPS][16 * MT][kTcStride], h1[WARPS][16 * MT][kTcStride], h2[WARPS][16 * MT][kTcStride];
    float d1[WARPS][16 * MT][kTcStride], d2[WARPS][16 * MT][kTcStride];
    float dy[WARPS][16 * MT][8];
    float g[kMlp16Params + 1];              // block reduction of the gradients (packed order)
    unsigned cmax[16];                      // max |feature gradient| per input column (bit patterns)
    double loss;
};

template <int MT, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
mlp16_tc_step_kernel(const float* __restrict__ x, const float* __restrict__ gt, int64_t n,
                     const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                     const float* __restrict__ b2, const float* __restrict__ W3, const float* __restrict__ b3,
                     float grad_scale, float* __restrict__ gx, float* __restrict__ pred, double* __restrict__ loss_sum,
                     float* __restrict__ grad_params, unsigned* __restrict__ gx_absmax) {
    constexpr int H = 16, OUT = 3;
    constexpr int oW1 = 0, ob1 = oW1 + 256, oW2 = ob1 + H, ob2 = oW2 + 256, oW3 = ob2 + H, ob3 = oW3 + OUT * H;
    // weight-fragment table: forward L1 (ks, nt) 0..3, L2 4..7, L3 (ks) 8..9; backward d2 (nt) 10..11, d1 (ks, nt)
    // 12..15, feature gradient (ks, nt) 16..19
    extern __shared__ __align__(16) unsigned char s_raw[];
    constexpr int kTcThreads = WARPS * 32, kTcWarps = WARPS, PTS = 16 * MT;
    using Smem = MlpTcSmem<MT, WARPS>;
    Smem& S = *reinterpret_cast<Smem*>(s_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    tc_build_fragments(S.wf, W1, W2, W3, tid, kTcThreads);
    for (int e = tid; e < kMlp16Params + 1; e += kTcThreads) S.g[e] = 0.0f;
    if (tid < H) { S.b1[tid] = b1[tid]; S.b2[tid] = b2[tid]; }
    if (tid < 4) S.b3[tid] = tid < OUT ? b3[tid] : 0.0f;
    if (tid == 0) S.loss = 0.0;
    if (tid < 16) S.cmax[tid] = 0u;
    __syncthreads();

    float accW1[2][4], accW2[2][4], accW3[1][4], accb1[2][2], accb2[2][2], accb3[2] = {0.0f, 0.0f};
#pragma unroll
    for (int a = 0; a < 2; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b) { accW1[a][b] = 0.0f; accW2[a][b] = 0.0f; }
        accb1[a][0] = accb1[a][1] = accb2[a][0] = accb2[a][1] = 0.0f;
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) accW3[0][b] = 0.0f;
    float my_loss = 0.0f;
    float cmax[2][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}};   // max |gx| of this lane's columns 8 nt + 2 t + e
    float (*sx)[kTcStride] = S.x[warp];
    float (*sh1)[kTcStride] = S.h1[warp];
    float (*sh2)[kTcStride] = S.h2[warp];
    float (*sd1)[kTcStride] = S.d1[warp];
    float (*sd2)[kTcStride] = S.d2[warp];
    float (*sdy)[8] = S.dy[warp];

    const int64_t warps_total = (int64_t)gridDim.x * kTcWarps;
    float X[MT][2][4];
    auto load_x = [&](int64_t b) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int64_t row = b + 16 * mt + g + 8 * hh;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    float2 v = make_float2(0.0f, 0.0f);
                    if (row < n) v = __ldg(reinterpret_cast<const float2*>(x + row * 16 + 8 * ks + 2 * t));
                    X[mt][ks][2 * hh] = v.x;
                    X[mt][ks][2 * hh + 1] = v.y;
                }
            }
    };
    load_x(((int64_t)blockIdx.x * kTcWarps + warp) * PTS);
    for (int64_t base = ((int64_t)blockIdx.x * kTcWarps + warp) * PTS; base < n; base += warps_total * PTS) {
        // rows of this lane: base + 16 mt + g + 8 h. X was loaded by the previous iteration (software pipeline);
        // the targets of this iteration are requested now, long before the loss needs them
        float T[MT][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int col = 2 * t + (r & 1);
                const int64_t row = base + 16 * mt + g + 8 * (r >> 1);
                T[mt][r] = (col < OUT && row < n) ? __ldg(gt + row * OUT + col) : 0.0f;
            }
        __syncwarp();  // the previous iteration's weight-gradient reads of the staging rows are done
        tc_stage<MT>(sx, g, t, X);
        // ---- forward ----
        float h1[MT][2][4], h2[MT][2][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b1[8 * nt + 2 * t]);
                h1[mt][nt][0] = h1[mt][nt][2] = bb.x;
                h1[mt][nt][1] = h1[mt][nt][3] = bb.y;
            }
        tc_layer<2, 2, MT>(S.wf, F_L1, lane, X, h1);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b2[8 * nt + 2 * t]);
#pragma unroll
                for (int r = 0; r < 4; ++r) h1[mt][nt][r] = fmaxf(h1[mt][nt][r], 0.0f);
                h2[mt][nt][0] = h2[mt][nt][2] = bb.x;
                h2[mt][nt][1] = h2[mt][nt][3] = bb.y;
            }
        tc_stage<MT>(sh1, g, t, h1);
        tc_layer<2, 2, MT>(S.wf, F_L2, lane, h1, h2);
        float Y[MT][2][4];   // [mt][0] used (8 padded outputs); the second tile is a dummy of the generic helper
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int r = 0; r < 4; ++r) h2[mt][nt][r] = fmaxf(h2[mt][nt][r], 0.0f);
            }
        tc_stage<MT>(sh2, g, t, h2);
        {
            const float2 bb = *reinterpret_cast<const float2*>(&S.b3[(2 * t) & 3]);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                Y[mt][0][0] = Y[mt][0][2] = (t < 2) ? bb.x : 0.0f;
                Y[mt][0][1] = Y[mt][0][3] = (t < 2) ? bb.y : 0.0f;
#pragma unroll
                for (int r = 0; r < 4; ++r) Y[mt][1][r] = 0.0f;
            }
        }
        {   // 16 -> 3 (padded to one 8-column tile): K = 16 in two k-steps, fragments F_L3 + ks
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const uint4 f = S.wf[F_L3 + ks][lane];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    uint32_t ahi[4], alo[4];
                    tile_to_a(h2[mt][ks], ahi, alo);
                    mma3(Y[mt][0], ahi, alo, f.x, f.y, f.z, f.w);
                }
            }
        }
        // ---- loss and its gradient (columns 2t, 2t+1 < 3 are real) ----
        float DY[MT][2][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int col = 2 * t + (r & 1);
                const int64_t row = base + 16 * mt + g + 8 * (r >> 1);
                float d = 0.0f;
                if (col < OUT && row < n) {
                    const float y = Y[mt][0][r];
                    const float e = y - T[mt][r];
                    my_loss = fmaf(e, e, my_loss);
                    d = e * grad_scale;
                    if (pred) pred[row * OUT + col] = y;
                }
                DY[mt][0][r] = d;
                DY[mt][1][r] = 0.0f;
            }
            *reinterpret_cast<float2*>(&sdy[16 * mt + g][2 * t]) = make_float2(DY[mt][0][0], DY[mt][0][1]);
            *reinterpret_cast<float2*>(&sdy[16 * mt + g + 8][2 * t]) = make_float2(DY[mt][0][2], DY[mt][0][3]);
            accb3[0] += DY[mt][0][0] + DY[mt][0][2];
            accb3[1] += DY[mt][0][1] + DY[mt][0][3];
        }
        // ---- backward to the features ----
        float D[MT][2][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) D[mt][nt][r] = 0.0f;
        tc_layer<1, 2, MT>(S.wf, B_D2, lane, DY, D);                  // d2 = dy W3   (K = 8 padded outputs)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int r = 0; r < 4; ++r) D[mt][nt][r] = h2[mt][nt][r] > 0.0f ? D[mt][nt][r] : 0.0f;
                accb2[nt][0] += D[mt][nt][0] + D[mt][nt][2];
                accb2[nt][1] += D[mt][nt][1] + D[mt][nt][3];
            }
        tc_stage<MT>(sd2, g, t, D);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) h2[mt][nt][r] = 0.0f;   // h2 is dead: reuse as d1
        tc_layer<2, 2, MT>(S.wf, B_D1, lane, D, h2);                  // d1 = d2 W2
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    h2[mt][nt][r] = h1[mt][nt][r] > 0.0f ? h2[mt][nt][r] : 0.0f;
                    D[mt][nt][r] = 0.0f;
                }
                accb1[nt][0] += h2[mt][nt][0] + h2[mt][nt][2];
                accb1[nt][1] += h2[mt][nt][1] + h2[mt][nt][3];
            }
        tc_stage<MT>(sd1, g, t, h2);
        tc_layer<2, 2, MT>(S.wf, B_GX, lane, h2, D);                  // gx = d1 W1
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int64_t row = base + 16 * mt + g + 8 * hh;
                if (row < n) {
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt) {
                        *reinterpret_cast<float2*>(gx + row * 16 + 8 * nt + 2 * t) =
                            make_float2(D[mt][nt][2 * hh], D[mt][nt][2 * hh + 1]);
                        cmax[nt][0] = nan_max(cmax[nt][0], fabsf(D[mt][nt][2 * hh]));
                        cmax[nt][1] = nan_max(cmax[nt][1], fabsf(D[mt][nt][2 * hh + 1]));
                    }
                }
            }
        load_x(base + warps_total * PTS);   // next iteration's features: in flight behind the weight-gradient stage
        __syncwarp();
        // ---- weight gradients: K = the warp's 32 points, operands from the staged rows ----
        tc_wgrad<2, kTcStride, MT>(sd1, sx, g, t, accW1);    // dW1[i][m] = sum_p d1[p][i] x[p][m]
        tc_wgrad<2, kTcStride, MT>(sd2, sh1, g, t, accW2);   // dW2[j][i] = sum_p d2[p][j] h1[p][i]
        tc_wgrad<1, 8, MT>(sh2, sdy, g, t, accW3);           // dW3^T[j][k] = sum_p h2[p][j] dy[p][k]
    }
    // ---- block reduction in shared memory, then one global add per CTA and value ----
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = g + 8 * (r >> 1), col = 8 * nt + 2 * t + (r & 1);
            atomicAdd(&S.g[oW1 + row * 16 + col], accW1[nt][r]);
            atomicAdd(&S.g[oW2 + row * 16 + col], accW2[nt][r]);
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            atomicAdd(&S.g[ob1 + 8 * nt + 2 * t + e], accb1[nt][e]);
            atomicAdd(&S.g[ob2 + 8 * nt + 2 * t + e], accb2[nt][e]);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int j = g + 8 * (r >> 1), k = 2 * t + (r & 1);
        if (k < OUT) atomicAdd(&S.g[oW3 + k * 16 + j], accW3[0][r]);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e)
        if (2 * t + e < OUT) atomicAdd(&S.g[ob3 + 2 * t + e], accb3[e]);
    if (gx_absmax) {   // non-negative floats order like their bit patterns
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                unsigned m = __float_as_uint(cmax[nt][e]);
                m = max(m, __shfl_xor_sync(0xffffffffu, m, 4));
                m = max(m, __shfl_xor_sync(0xffffffffu, m, 8));
                m = max(m, __shfl_xor_sync(0xffffffffu, m, 16));
                if (g == 0) atomicMax(&S.cmax[8 * nt + 2 * t + e], m);
            }
    }
    const float wl = warp_sum(my_loss);
    if (lane == 0) atomicAdd(&S.loss, (double)wl);
    __syncthreads();
    for (int e = tid; e < kMlp16Params; e += kTcThreads) red_add(grad_params + e, S.g[e]);
    if (gx_absmax && tid < 16) atomicMax(gx_absmax + tid, S.cmax[tid]);
    if (tid == 0) atomicAdd(loss_sum, S.loss);
}

}  // namespace shacira
