// nerf_heads_kernels.cuh -- the NeRF decoder heads (NeuralRadianceField.rgba, wisp/models/nefs/nerf.py:218-233) on the
// tensor cores: tcgen05.mma with bf16 operands and fp32 accumulators in tensor memory (TMEM).
//
//   h1 = relu(b(X) b(W1)^T + b1)          X [S, IN], W1 [H, IN]          (IN = 64 or 96, H = 128)
//   d  = b(h1) b(W2)^T + b2               W2 [16, H]                      density = relu(d[:, 0])
//   u  = [b(d), b(V[ridx])]               V [R, E], E <= 32, K padded to 48
//   h2 = relu(u b(W3)^T + b3)             W3 [H, 16 + E]
//   h3 = relu(b(h2) b(W4)^T + b4)         W4 [H, H]
//   o  = b(h3) b(W5)^T + b5               W5 [3, H], N padded to 16      rgb = sigmoid(o)
//
// b() is round-to-nearest-even to bf16 (DESIGN section 9). One CTA of 128 threads works on tiles of 128 samples;
// thread t owns sample row t of the tile, which is TMEM lane t of every M = 128 product. Every operand lives in
// shared memory in the canonical 128-byte-swizzled layout: a tile of `rows` rows and 64-column blocks stores element
// (r, c) at byte (c / 64) * rows * 128 + r * 128 + ((c / 8 % 8) ^ (r % 8)) * 16 + (c % 8) * 2. The same bytes read
// as a K-major operand (K = columns: forward products, input gradients) or, with the descriptor's transpose bit, as
// an MN-major operand (K = rows = samples: weight gradients; K = output features: input gradients through a weight
// tile), so no tile is ever transposed.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace shacira {
namespace heads {

constexpr int kH = 128;          // hidden width of both heads
constexpr int kD = 16;           // width of the density head's output (density + 15 features)
constexpr int kOut = 3;          // rgb
constexpr int kUK = 48;          // K of the colour head's first product: 16 + E padded to a multiple of 16
constexpr int kMaxE = kUK - kD;  // 32
constexpr int kTile = 128;       // samples per tile = threads per CTA = TMEM lanes
constexpr int kThreads = 128;

// TMEM columns (fp32, 128 lanes). The per-tile products share the first 144 columns; the weight-gradient
// accumulators of the backward stay resident for the CTA's whole life.
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kAccBig = 0;      // [128 x <=128]: h1, h2, h3 pre-activations; g_h3, g_h2, g_h1, g_X
constexpr uint32_t kAccSmall = 128;  // [128 x 16]: d, o, g_u
constexpr uint32_t kAccW4 = 192;     // dW4   [j][i], 128 columns
constexpr uint32_t kAccW1 = 320;     // dW1   [j][i], IN columns (<= 96)
constexpr uint32_t kAccW3 = 416;     // dW3   [j][i], 48 columns
constexpr uint32_t kAccW2 = 464;     // dW2^T [j][o], 16 columns
constexpr uint32_t kAccW5 = 480;     // dW5^T [j][o], 16 columns

// Bias-gradient lanes: 32-column groups, reduced across the warp with a butterfly reduce-scatter.
constexpr int kBiasGroups = 4 /*b1*/ + 1 /*b2*/ + 4 /*b3*/ + 4 /*b4*/ + 1 /*b5*/;

// Per-CTA partial sums the backward writes and nerf_heads_reduce_kernel folds, in CTA order:
// [kW columns][128 lanes] of the TMEM weight-gradient accumulators, then [kBiasGroups * 32] bias sums.
template <int IN>
struct Partial {
    static constexpr int kWCols = kH + IN + kUK + kD + kD;   // dW4, dW1, dW3, dW2^T, dW5^T
    static constexpr int kFloats = kWCols * kTile + kBiasGroups * 32;
};

// Shared-memory map (bytes from a 1024-aligned base). Weight tiles first, then the four activation regions.
template <int IN>
struct Smem {
    static constexpr int kInBlocks = (IN + 63) / 64;
    static constexpr uint32_t W1 = 0;                                  // [128][IN]
    static constexpr uint32_t W2 = W1 + kInBlocks * kH * 128;          // [16][128]
    static constexpr uint32_t W3 = W2 + 2 * kD * 128;                  // [128][48]
    static constexpr uint32_t W4 = W3 + kH * 128;                      // [128][128]
    static constexpr uint32_t W5 = W4 + 2 * kH * 128;                  // [16][128] (rows 3..15 zero)
    static constexpr uint32_t R0 = W5 + 2 * kD * 128;                  // X, then h3 / g_h3, then X again
    static constexpr uint32_t R1 = R0 + 2 * kTile * 128;               // h1 / g_h1
    static constexpr uint32_t R2 = R1 + 2 * kTile * 128;               // u, g_o, u again, g_d
    static constexpr uint32_t R3 = R2 + kTile * 128;                   // h2 / g_h2
    static constexpr uint32_t Bias = R3 + 2 * kTile * 128;             // b1 | b2 | b3 | b4 | b5 (fp32)
    static constexpr uint32_t kBiasFloats = kH + kD + kH + kH + kD;
    static constexpr uint32_t Red = Bias + kBiasFloats * 4;            // [4 warps][kBiasGroups * 32] fp32
    static constexpr uint32_t kBytes = Red + 4 * kBiasGroups * 32 * 4;
    static constexpr uint32_t kDynamic = kBytes + 1024;                // room to align the base to 1024
};

// ---------------------------------------------------------------------------------------------------------------
// tcgen05 primitives

__device__ __forceinline__ uint32_t swz(int rows, int r, int c) {
    return (uint32_t)((c >> 6) * rows * 128 + r * 128 + ((((c >> 3) & 7) ^ (r & 7)) << 4) + (c & 7) * 2);
}

// Shared-memory matrix descriptor, sm_100 format: start >> 4 in [0, 14), leading byte offset >> 4 in [16, 30),
// stride byte offset >> 4 in [32, 46), version 1 in [46, 48), layout SWIZZLE_128B (2) in [61, 64).
__device__ __forceinline__ uint64_t sdesc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}
// K-major view of a tile (K = columns): 16-column step k starts 32 bytes further inside its 64-column block;
// 8-row groups are 1024 bytes apart.
__device__ __forceinline__ uint64_t desc_k(uint32_t tile, int rows, int k) {
    const int c = k * 16;
    return sdesc(tile + (uint32_t)((c >> 6) * rows * 128 + (c & 63) * 2), 16, 1024);
}
// MN-major view (K = rows, MN = columns): step k starts 16 rows further down; 8-row groups along K are 1024 bytes
// apart (stride byte offset) and 64-column blocks along MN are rows * 128 bytes apart (leading byte offset).
__device__ __forceinline__ uint64_t desc_mn(uint32_t tile, int rows, int k) {
    return sdesc(tile + (uint32_t)(k * 16 * 128), (uint32_t)rows * 128u, 1024);
}

// Instruction descriptor of kind::f16: fp32 accumulator, bf16 A and B, transpose (MN-major) bits, N >> 3, M >> 4.
__host__ __device__ constexpr uint32_t idesc(int M, int N, bool a_mn, bool b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t id, bool accumulate) {
    asm volatile(
        "{.reg .pred p; setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;}" ::"r"(d_tmem),
        "l"(a), "l"(b), "r"(id), "r"((uint32_t)accumulate));
}
__device__ __forceinline__ void commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    asm volatile(
        "{.reg .pred p;\n"
        "WAIT_%=: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra WAIT_%=;}" ::"r"(mbar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 16 consecutive fp32 columns of this thread's TMEM lane.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);   // round to nearest even, NaN stays NaN
    return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
// torch.relu keeps NaN (fmaxf would not)
__device__ __forceinline__ float relu(float z) { return z < 0.f ? 0.f : z; }

// Eight bf16 values (columns c .. c + 7, c a multiple of 8) of row r, one 16-byte store.
__device__ __forceinline__ void st_row8(uint8_t* tile, int rows, int r, int c, const float* v) {
    uint4 q;
    q.x = pack_bf16(v[0], v[1]);
    q.y = pack_bf16(v[2], v[3]);
    q.z = pack_bf16(v[4], v[5]);
    q.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + swz(rows, r, c)) = q;
}

// fp32 matrix [rows][cols] (row-major) -> bf16 tile of rows_p rows, columns padded to cols_p with zeros.
__device__ __forceinline__ void stage_weight(uint8_t* tile, const float* __restrict__ W, int rows, int cols, int rows_p,
                                             int cols_p) {
    for (int e = threadIdx.x; e < rows_p * cols_p; e += kThreads) {
        const int r = e / cols_p, c = e % cols_p;
        const float v = (r < rows && c < cols) ? __ldg(W + (int64_t)r * cols + c) : 0.f;
        *reinterpret_cast<__nv_bfloat16*>(tile + swz(rows_p, r, c)) = __float2bfloat16_rn(v);
    }
}

struct Params {
    const float* X;        // [S, IN]
    const float* V;        // [R, E]
    const int32_t* ridx;   // [S]
    int64_t S;
    int32_t R, E;
    const float *W1, *b1, *W2, *b2, *W3, *b3, *W4, *b4, *W5, *b5;
    float* density;        // [S]      forward
    float* rgb;            // [S, 3]   forward
    const float* g_density;  // [S]    backward
    const float* g_rgb;      // [S, 3] backward
    float* g_X;              // [S, IN] backward
    float* partial;          // [gridDim.x][Partial<IN>::kFloats] backward
};

// One CTA's resources: dynamic shared memory aligned to 1024, the MMA mbarrier and the TMEM allocation.
struct Cta {
    uint8_t* smem;
    uint32_t sbase;       // shared-space address of smem
    uint32_t mbar;
    uint32_t tmem;        // TMEM base (lane 0, first column)
    uint32_t lane_off;    // this warp's TMEM lanes, << 16
    uint32_t phase;

    // Make this thread's shared-memory writes visible to the tensor cores, order earlier TMEM loads before the
    // products that overwrite them, then let thread 0 issue.
    __device__ __forceinline__ void publish() {
        fence_async_smem();
        fence_before();
        __syncthreads();
        fence_after();
    }
    __device__ __forceinline__ void wait() {
        if (threadIdx.x == 0) commit(mbar);
        mbar_wait(mbar, phase);
        phase ^= 1u;
        fence_after();
    }
    __device__ __forceinline__ uint8_t* at(uint32_t off) const { return smem + off; }
    __device__ __forceinline__ uint32_t sa(uint32_t off) const { return sbase + off; }
    __device__ __forceinline__ uint32_t col(uint32_t c) const { return tmem + lane_off + c; }
};

__device__ __forceinline__ Cta cta_setup(uint8_t* dyn, uint32_t* tmem_slot, uint64_t* mbar_slot) {
    Cta c;
    const uint32_t raw = (uint32_t)__cvta_generic_to_shared(dyn);
    const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
    c.smem = dyn + pad;
    c.sbase = raw + pad;
    c.mbar = (uint32_t)__cvta_generic_to_shared(mbar_slot);
    c.phase = 0;
    if (threadIdx.x < 32) {
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(tmem_slot);
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(c.mbar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    c.tmem = *tmem_slot;
    c.lane_off = (uint32_t)((threadIdx.x >> 5) * 32) << 16;
    return c;
}

__device__ __forceinline__ void cta_teardown(const Cta& c) {
    fence_before();
    __syncthreads();
    fence_after();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(c.tmem), "r"(kTmemCols));
}

template <int IN>
__device__ __forceinline__ void stage_weights(const Cta& c, const Params& p, bool density_only) {
    using L = Smem<IN>;
    stage_weight(c.at(L::W1), p.W1, kH, IN, kH, IN);
    stage_weight(c.at(L::W2), p.W2, kD, kH, kD, kH);
    float* bias = reinterpret_cast<float*>(c.at(L::Bias));
    for (int i = threadIdx.x; i < kH; i += kThreads) bias[i] = __ldg(p.b1 + i);
    for (int i = threadIdx.x; i < kD; i += kThreads) bias[kH + i] = __ldg(p.b2 + i);
    if (density_only) return;
    stage_weight(c.at(L::W3), p.W3, kH, kD + p.E, kH, kUK);
    stage_weight(c.at(L::W4), p.W4, kH, kH, kH, kH);
    stage_weight(c.at(L::W5), p.W5, kOut, kH, kD, kH);
    for (int i = threadIdx.x; i < kH; i += kThreads) bias[kH + kD + i] = __ldg(p.b3 + i);
    for (int i = threadIdx.x; i < kH; i += kThreads) bias[2 * kH + kD + i] = __ldg(p.b4 + i);
    for (int i = threadIdx.x; i < kD; i += kThreads) bias[3 * kH + kD + i] = i < kOut ? __ldg(p.b5 + i) : 0.f;
}

// X rows t0 .. t0 + 127 -> b(X) in R0, rows past S zero. Coalesced: the tile is one contiguous block of floats.
template <int IN>
__device__ __forceinline__ void load_x(const Cta& c, const float* __restrict__ X, int64_t t0, int valid) {
    uint8_t* tile = c.at(Smem<IN>::R0);
#pragma unroll 4
    for (int it = 0; it < IN / 4; ++it) {
        const int e = 4 * (threadIdx.x + kThreads * it);
        const int r = e / IN, col = e % IN;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < valid) v = __ldg(reinterpret_cast<const float4*>(X + t0 * IN + e));
        uint2 q;
        q.x = pack_bf16(v.x, v.y);
        q.y = pack_bf16(v.z, v.w);
        *reinterpret_cast<uint2*>(tile + swz(kTile, r, col)) = q;
    }
}

// u = [b(d), b(V[ridx]), 0 ...] of this thread's row into R2. A ridx outside [0, R) takes a zero embedding.
template <int IN>
__device__ __forceinline__ void store_u(const Cta& c, const Params& p, int64_t s, bool valid, const float (&d)[kD]) {
    const int r = threadIdx.x;
    uint8_t* tile = c.at(Smem<IN>::R2);
    const float* v = nullptr;
    if (valid) {
        const int32_t ray = __ldg(p.ridx + s);
        if (ray >= 0 && ray < p.R) v = p.V + (int64_t)ray * p.E;
    }
    st_row8(tile, kTile, r, 0, d);
    st_row8(tile, kTile, r, 8, d + 8);
#pragma unroll
    for (int c8 = kD; c8 < kUK; c8 += 8) {
        float e[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = c8 - kD + i;
            e[i] = (v && k < p.E) ? __ldg(v + k) : 0.f;
        }
        st_row8(tile, kTile, r, c8, e);
    }
}

// TMEM [128 x 128] pre-activation + bias -> relu -> b() into a 128-column tile; ReLU mask bits into `mask`.
__device__ __forceinline__ void hidden_epilogue(const Cta& c, uint32_t acc, const float* bias, uint8_t* tile,
                                                uint32_t (&mask)[4]) {
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
        float v[32];
        tmem_ld16(c.col(acc + 32 * g), *reinterpret_cast<float(*)[16]>(v));
        tmem_ld16(c.col(acc + 32 * g + 16), *reinterpret_cast<float(*)[16]>(v + 16));
        uint32_t bits = 0;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            v[i] = relu(v[i] + bias[32 * g + i]);
            bits |= (uint32_t)(v[i] > 0.f) << i;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) mask[i] = g == i ? bits : mask[i];
#pragma unroll
        for (int i = 0; i < 32; i += 8) st_row8(tile, kTile, threadIdx.x, 32 * g + i, v + i);
    }
}

// Forward of one tile. On return: h1 (R1), h2 (R3), h3 (R0) hold the bf16 activations, `dq` the bf16-rounded d,
// `d0` = d[:, 0], `o` the three colour pre-activations and `mask*` the ReLU masks. DENSITY_ONLY stops after d.
template <int IN, bool DENSITY_ONLY>
__device__ __forceinline__ void forward_tile(Cta& c, const Params& p, int64_t t0, int valid, float (&dq)[kD], float& d0,
                                             float (&o)[kOut], uint32_t (&m1)[4], uint32_t (&m2)[4],
                                             uint32_t (&m3)[4]) {
    using L = Smem<IN>;
    const float* bias = reinterpret_cast<const float*>(c.at(L::Bias));
    const int r = threadIdx.x;
    const int64_t s = t0 + r;
    load_x<IN>(c, p.X, t0, valid);
    c.publish();
    if (r == 0) {
#pragma unroll
        for (int k = 0; k < IN / 16; ++k)
            mma(c.tmem + kAccBig, desc_k(c.sa(L::R0), kTile, k), desc_k(c.sa(L::W1), kH, k), idesc(128, kH, false, false),
                k > 0);
    }
    c.wait();
    hidden_epilogue(c, kAccBig, bias, c.at(L::R1), m1);
    c.publish();
    if (r == 0) {
#pragma unroll
        for (int k = 0; k < kH / 16; ++k)
            mma(c.tmem + kAccSmall, desc_k(c.sa(L::R1), kTile, k), desc_k(c.sa(L::W2), kD, k),
                idesc(128, kD, false, false), k > 0);
    }
    c.wait();
    {
        float v[16];
        tmem_ld16(c.col(kAccSmall), v);
#pragma unroll
        for (int i = 0; i < kD; ++i) v[i] += bias[kH + i];
        d0 = v[0];
#pragma unroll
        for (int i = 0; i < kD; ++i) dq[i] = bf16_round(v[i]);
    }
    if (DENSITY_ONLY) return;
    store_u<IN>(c, p, s, r < valid, dq);
    c.publish();
    if (r == 0) {
#pragma unroll
        for (int k = 0; k < kUK / 16; ++k)
            mma(c.tmem + kAccBig, desc_k(c.sa(L::R2), kTile, k), desc_k(c.sa(L::W3), kH, k), idesc(128, kH, false, false),
                k > 0);
    }
    c.wait();
    hidden_epilogue(c, kAccBig, bias + kH + kD, c.at(L::R3), m2);
    c.publish();
    if (r == 0) {
#pragma unroll
        for (int k = 0; k < kH / 16; ++k)
            mma(c.tmem + kAccBig, desc_k(c.sa(L::R3), kTile, k), desc_k(c.sa(L::W4), kH, k), idesc(128, kH, false, false),
                k > 0);
    }
    c.wait();
    hidden_epilogue(c, kAccBig, bias + 2 * kH + kD, c.at(L::R0), m3);
    c.publish();
    if (r == 0) {
#pragma unroll
        for (int k = 0; k < kH / 16; ++k)
            mma(c.tmem + kAccSmall, desc_k(c.sa(L::R0), kTile, k), desc_k(c.sa(L::W5), kD, k),
                idesc(128, kD, false, false), k > 0);
    }
    c.wait();
    {
        float v[16];
        tmem_ld16(c.col(kAccSmall), v);
#pragma unroll
        for (int i = 0; i < kOut; ++i) o[i] = v[i] + bias[3 * kH + kD + i];
    }
}

__device__ __forceinline__ float sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

template <int IN, bool DENSITY_ONLY>
__global__ void __launch_bounds__(kThreads, 1) nerf_heads_fwd_kernel(const Params p) {
    extern __shared__ uint8_t dyn[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t mbar_slot;
    Cta c = cta_setup(dyn, &tmem_slot, &mbar_slot);
    stage_weights<IN>(c, p, DENSITY_ONLY);
    const int64_t tiles = (p.S + kTile - 1) / kTile;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int64_t t0 = t * kTile;
        const int valid = (int)(p.S - t0 < kTile ? p.S - t0 : kTile);
        float dq[kD], d0, o[kOut];
        uint32_t m1[4], m2[4], m3[4];
        forward_tile<IN, DENSITY_ONLY>(c, p, t0, valid, dq, d0, o, m1, m2, m3);
        const int64_t s = t0 + threadIdx.x;
        if ((int)threadIdx.x < valid) {
            p.density[s] = relu(d0);
            if (!DENSITY_ONLY) {
#pragma unroll
                for (int i = 0; i < kOut; ++i) p.rgb[s * kOut + i] = sigmoid(o[i]);
            }
        }
    }
    cta_teardown(c);
}

// ---------------------------------------------------------------------------------------------------------------
// Backward

// Sum of v[0..31] over the warp, scattered: lane l returns the warp's sum of column l. Fixed order (deterministic).
__device__ __forceinline__ float warp_column_sums(float (&v)[32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool upper = lane & s;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = upper ? v[i] : v[i + s];
            const float keep = upper ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

// Gradient of a 128-wide hidden layer: TMEM [128 x 128] -> mask -> b() into `tile`; its fp32 column sums are added
// to the four 32-column groups of bias-sum slots at `bsum` (this lane's slot of each group).
__device__ __forceinline__ void hidden_grad_epilogue(const Cta& c, const uint32_t (&mask)[4], uint8_t* tile,
                                                     float* bsum) {
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
        float v[32];
        tmem_ld16(c.col(kAccBig + 32 * g), *reinterpret_cast<float(*)[16]>(v));
        tmem_ld16(c.col(kAccBig + 32 * g + 16), *reinterpret_cast<float(*)[16]>(v + 16));
        const uint32_t m = g == 0 ? mask[0] : g == 1 ? mask[1] : g == 2 ? mask[2] : mask[3];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = ((m >> i) & 1u) ? v[i] : 0.f;
#pragma unroll
        for (int i = 0; i < 32; i += 8) st_row8(tile, kTile, threadIdx.x, 32 * g + i, v + i);
        bsum[g * 32] += warp_column_sums(v);
    }
}

template <int IN>
__global__ void __launch_bounds__(kThreads, 1) nerf_heads_bwd_kernel(const Params p) {
    using L = Smem<IN>;
    extern __shared__ uint8_t dyn[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t mbar_slot;
    Cta c = cta_setup(dyn, &tmem_slot, &mbar_slot);
    stage_weights<IN>(c, p, false);
    const int r = threadIdx.x;
    // bias-gradient sums: [warp][group][lane], lane l holding column l of the group over this warp's rows
    float* red = reinterpret_cast<float*>(c.at(L::Red));
    float* bsum = red + (r >> 5) * kBiasGroups * 32 + (r & 31);
#pragma unroll
    for (int i = 0; i < kBiasGroups; ++i) bsum[i * 32] = 0.f;
    constexpr int kB1 = 0, kB2 = 4 * 32, kB3 = 5 * 32, kB4 = 9 * 32, kB5 = 13 * 32;

    const int64_t tiles = (p.S + kTile - 1) / kTile;
    bool first = true;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x, first = false) {
        const int64_t t0 = t * kTile;
        const int valid = (int)(p.S - t0 < kTile ? p.S - t0 : kTile);
        const int64_t s = t0 + r;
        const bool live = r < valid;
        float dq[kD], d0, o[kOut];
        uint32_t m1[4], m2[4], m3[4];
        forward_tile<IN, false>(c, p, t0, valid, dq, d0, o, m1, m2, m3);

        // g_o = g_rgb * rgb (1 - rgb) -> R2 (g_o), columns 3..15 zero
        {
            float go[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) go[i] = 0.f;
#pragma unroll
            for (int i = 0; i < kOut; ++i) {
                const float y = sigmoid(o[i]);
                go[i] = live ? __ldg(p.g_rgb + s * kOut + i) * (y * (1.f - y)) : 0.f;
            }
            st_row8(c.at(L::R2), kTile, r, 0, go);
            st_row8(c.at(L::R2), kTile, r, 8, go + 8);
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = i < 16 ? go[i] : 0.f;
            bsum[kB5] += warp_column_sums(v);
        }
        c.publish();
        if (r == 0) {
            // dW5^T[j][o] += h3^T g_o ; g_h3 = g_o W5
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
                mma(c.tmem + kAccW5, desc_mn(c.sa(L::R0), kTile, k), desc_mn(c.sa(L::R2), kTile, k),
                    idesc(128, kD, true, true), !first || k > 0);
            mma(c.tmem + kAccBig, desc_k(c.sa(L::R2), kTile, 0), desc_mn(c.sa(L::W5), kD, 0), idesc(128, kH, false, true),
                false);
        }
        c.wait();
        hidden_grad_epilogue(c, m3, c.at(L::R0), bsum + kB4);   // g_h3 (pre-activation) -> R0
        c.publish();
        if (r == 0) {
            // dW4[j][i] += g_h3^T h2 ; g_h2 = g_h3 W4
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
                mma(c.tmem + kAccW4, desc_mn(c.sa(L::R0), kTile, k), desc_mn(c.sa(L::R3), kTile, k),
                    idesc(128, kH, true, true), !first || k > 0);
#pragma unroll
            for (int k = 0; k < kH / 16; ++k)
                mma(c.tmem + kAccBig, desc_k(c.sa(L::R0), kTile, k), desc_mn(c.sa(L::W4), kH, k),
                    idesc(128, kH, false, true), k > 0);
        }
        c.wait();
        hidden_grad_epilogue(c, m2, c.at(L::R3), bsum + kB3);   // g_h2 -> R3
        store_u<IN>(c, p, s, live, dq);                          // u again -> R2
        c.publish();
        if (r == 0) {
            // dW3[j][i] += g_h2^T u ; g_u[:, 0:16] = g_h2 W3[:, 0:16]
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
                mma(c.tmem + kAccW3, desc_mn(c.sa(L::R3), kTile, k), desc_mn(c.sa(L::R2), kTile, k),
                    idesc(128, kUK, true, true), !first || k > 0);
#pragma unroll
            for (int k = 0; k < kH / 16; ++k)
                mma(c.tmem + kAccSmall, desc_k(c.sa(L::R3), kTile, k), desc_mn(c.sa(L::W3), kH, k),
                    idesc(128, kD, false, true), k > 0);
        }
        c.wait();
        {
            // g_d = g_u[:, 0:16], plus g_density through relu(d[:, 0])
            float v[32];
            tmem_ld16(c.col(kAccSmall), *reinterpret_cast<float(*)[16]>(v));
            if (live && d0 > 0.f) v[0] += __ldg(p.g_density + s);
            st_row8(c.at(L::R2), kTile, r, 0, v);
            st_row8(c.at(L::R2), kTile, r, 8, v + 8);
#pragma unroll
            for (int i = 16; i < 32; ++i) v[i] = 0.f;
            bsum[kB2] += warp_column_sums(v);
        }
        c.publish();
        if (r == 0) {
            // dW2^T[j][o] += h1^T g_d ; g_h1 = g_d W2
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
                mma(c.tmem + kAccW2, desc_mn(c.sa(L::R1), kTile, k), desc_mn(c.sa(L::R2), kTile, k),
                    idesc(128, kD, true, true), !first || k > 0);
            mma(c.tmem + kAccBig, desc_k(c.sa(L::R2), kTile, 0), desc_mn(c.sa(L::W2), kD, 0), idesc(128, kH, false, true),
                false);
        }
        c.wait();
        hidden_grad_epilogue(c, m1, c.at(L::R1), bsum + kB1);   // g_h1 -> R1
        load_x<IN>(c, p.X, t0, valid);                            // X again -> R0
        c.publish();
        if (r == 0) {
            // dW1[j][i] += g_h1^T X ; g_X = g_h1 W1
#pragma unroll
            for (int k = 0; k < kTile / 16; ++k)
                mma(c.tmem + kAccW1, desc_mn(c.sa(L::R1), kTile, k), desc_mn(c.sa(L::R0), kTile, k),
                    idesc(128, IN, true, true), !first || k > 0);
#pragma unroll
            for (int k = 0; k < kH / 16; ++k)
                mma(c.tmem + kAccBig, desc_k(c.sa(L::R1), kTile, k), desc_mn(c.sa(L::W1), kH, k),
                    idesc(128, IN, false, true), k > 0);
        }
        c.wait();
#pragma unroll
        for (int c0 = 0; c0 < IN; c0 += 16) {
            float v[16];
            tmem_ld16(c.col(kAccBig + c0), v);
            if (live) {
                float4* dst = reinterpret_cast<float4*>(p.g_X + s * IN + c0);
#pragma unroll
                for (int i = 0; i < 4; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
            }
        }
    }

    // This CTA's partial sums: TMEM weight-gradient columns [col][lane], then the bias column sums of its 4 warps.
    float* out = p.partial + (int64_t)blockIdx.x * Partial<IN>::kFloats;
    constexpr int kWCols = Partial<IN>::kWCols;
    const uint32_t w_first[5] = {kAccW4, kAccW1, kAccW3, kAccW2, kAccW5};
    const int w_cols[5] = {kH, IN, kUK, kD, kD};
    int base = 0;
#pragma unroll
    for (int m = 0; m < 5; ++m) {
        for (int c0 = 0; c0 < w_cols[m]; c0 += 16) {
            float v[16];
            if (first) {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = 0.f;   // a CTA without a tile never wrote its accumulators
            } else {
                tmem_ld16(c.col(w_first[m] + c0), v);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) out[(int64_t)(base + c0 + i) * kTile + r] = v[i];
        }
        base += w_cols[m];
    }
    __syncthreads();
    for (int i = r; i < kBiasGroups * 32; i += kThreads)
        out[kWCols * kTile + i] = ((red[i] + red[kBiasGroups * 32 + i]) + red[2 * kBiasGroups * 32 + i]) +
                                  red[3 * kBiasGroups * 32 + i];
    cta_teardown(c);
}

// Folds the per-CTA partials in CTA order into the ten torch-layout gradients. One thread per output element.
template <int IN>
__global__ void nerf_heads_reduce_kernel(const float* __restrict__ partial, int ctas, int E, float* gW1, float* gb1,
                                         float* gW2, float* gb2, float* gW3, float* gb3, float* gW4, float* gb4,
                                         float* gW5, float* gb5) {
    constexpr int kWCols = Partial<IN>::kWCols;
    const int K3 = kD + E;
    // output element ranges, in the order of the ten tensors
    const int n1 = kH * IN, n2 = kD * kH, n3 = kH * K3, n4 = kH * kH, n5 = kOut * kH;
    const int nb = kH + kD + kH + kH + kOut;
    const int total = n1 + n2 + n3 + n4 + n5 + nb;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    int src;       // index into one CTA's partial
    float* dst;
    int q = e;
    // weight-gradient partial columns: dW4 [0, 128), dW1 [128, 128 + IN), dW3, dW2^T, dW5^T
    const int cW4 = 0, cW1 = kH, cW3 = kH + IN, cW2 = cW3 + kUK, cW5 = cW2 + kD;
    if (q < n1) { const int j = q / IN, i = q % IN; src = (cW1 + i) * kTile + j; dst = gW1 + q; }
    else if ((q -= n1) < n2) { const int o = q / kH, j = q % kH; src = (cW2 + o) * kTile + j; dst = gW2 + q; }
    else if ((q -= n2) < n3) { const int j = q / K3, i = q % K3; src = (cW3 + i) * kTile + j; dst = gW3 + q; }
    else if ((q -= n3) < n4) { const int j = q / kH, i = q % kH; src = (cW4 + i) * kTile + j; dst = gW4 + q; }
    else if ((q -= n4) < n5) { const int o = q / kH, j = q % kH; src = (cW5 + o) * kTile + j; dst = gW5 + q; }
    else {
        q -= n5;
        const int B = kWCols * kTile;   // bias groups: b1 (4 x 32), b2 (16 of 32), b3 (4 x 32), b4 (4 x 32), b5 (3 of 32)
        if (q < kH) { src = B + q; dst = gb1 + q; }
        else if ((q -= kH) < kD) { src = B + 4 * 32 + q; dst = gb2 + q; }
        else if ((q -= kD) < kH) { src = B + 5 * 32 + q; dst = gb3 + q; }
        else if ((q -= kH) < kH) { src = B + 9 * 32 + q; dst = gb4 + q; }
        else { q -= kH; src = B + 13 * 32 + q; dst = gb5 + q; }
    }
    float acc = 0.f;
    for (int b = 0; b < ctas; ++b) acc += partial[(int64_t)b * Partial<IN>::kFloats + src];
    *dst = acc;
}

}  // namespace heads
}  // namespace shacira
