// tiled_kernels.cuh -- the B200 fast path: spatially tiled fused latent grid kernels.
//
// Why: measured on B200 (profiles/r01_microbench_b200.csv) random 4-byte gathers from an L2-resident
// table run at ~300 Glanes/s and float REDG at ~200 Glanes/s -- collapsing to ~4 Glanes/s when a
// few hundred addresses take all the traffic (coarse levels) -- while shared memory serves random
// gathers at ~2300 Glanes/s and *integer* shared atomics at ~1600 Glanes/s irrespective of conflicts.
// So points are binned into spatial tiles once per coordinate set (the "plan"), and one CTA per
// tile stages the grid NODES its tile touches (about 2-3 per point, all levels together, instead
// of 2^D * L gathers per point) in shared memory:
//   forward : nodes <- rint(latents) once per tile; every point lerps from shared memory, applies
//             the affine decode and writes its output row at its ORIGINAL index;
//   backward: every point adds w_k * (A^T g) to its tile's node accumulators in shared memory as
//             fixed-point integers (exact, order-independent sums; per-tile per-level power-of-two
//             scale from the tile's max |gradient|), then the tile flushes each touched node with ONE
//             float REDG. Decoder gradients use warp REDUX on the same fixed-point values.
// Levels whose node box does not fit the shared-memory budget (fine 3D levels, huge resolutions)
// fall back per level to direct global gathers / REDG inside the same kernel.
//
// Indices, weights and rounding are computed by the same device functions as the point-parallel
// kernels (common.cuh), so hash indices and quantised latents stay bit-identical to the reference.
#pragma once
#include "common.cuh"

namespace shacira {

#ifndef SHACIRA_TILE_THREADS
#define SHACIRA_TILE_THREADS 128
#endif
constexpr int kTileThreads = SHACIRA_TILE_THREADS;
constexpr int kMaxTiles = 4096;
#ifndef SHACIRA_KP1
#define SHACIRA_KP1 2   // points per thread in flight in the backward's max pass (F = 1)
#endif
#ifndef SHACIRA_KPTS
#define SHACIRA_KPTS 2
#endif
constexpr int kPts = SHACIRA_KPTS;  // points per thread whose loads are issued together (memory-level parallelism)
constexpr int kBatch = 2048;  // points accumulated between two flushes of a tile (bounds the fixed-point sums)

struct PlanView {
    const int32_t* perm;          // sorted position -> original point index; NULL: rows are exchanged in SORTED order
    const float* coords_sorted;   // [n, D] coordinates in sorted order
    const int32_t* tile_off;      // [ntiles + 1]
    int64_t n;
    int32_t g;                    // tiles per axis (power of two)
    int32_t ntiles;
    // per (plan, level configuration): for every tile and staged node slot, the absolute table row (.x) and the
    // level | kNodeInvalid (.y). Depends on the tile grid and the levels only -- not on coordinates or latents --
    // so it is built once (plan_nodes_kernel) and turns the per-node index math of staging / flush into a load.
    const int2* node_tab;         // [ntiles][node_stride]
    int32_t node_stride;
};
constexpr int kNodeInvalid = 0x100;  // node outside its level: only ever carries weight 0 (SURVEY Q4)

// ---------------------------------------------------------------------------------------------
// plan construction: tile id -> histogram -> scan -> scatter
// ---------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ int tile_of(const float* __restrict__ coords, int64_t i, int g) {
    int id = 0, mul = 1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        const double t = unit_coord(__ldg(coords + i * D + d));
        int ti = (int)floor(t * (double)g);
        ti = max(0, min(g - 1, ti));
        id += ti * mul;
        mul *= g;
    }
    return id;
}

template <int D>
__global__ void __launch_bounds__(1024)
plan_count_kernel(const float* __restrict__ coords, int64_t n, int g, int ntiles, int32_t* __restrict__ tile_id,
                  int32_t* __restrict__ counts) {
    extern __shared__ int s_hist[];
    for (int e = threadIdx.x; e < ntiles; e += blockDim.x) s_hist[e] = 0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int t = tile_of<D>(coords, i, g);
        tile_id[i] = t;
        atomicAdd(&s_hist[t], 1);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < ntiles; e += blockDim.x)
        if (s_hist[e]) atomicAdd(&counts[e], s_hist[e]);
}

// single block: exclusive scan of counts[ntiles] -> tile_off[ntiles+1]; cursor = tile_off
__global__ void __launch_bounds__(1024)
plan_scan_kernel(const int32_t* __restrict__ counts, int ntiles, int32_t* __restrict__ tile_off,
                 int32_t* __restrict__ cursor) {
    __shared__ int s_part[1024];
    const int per = (ntiles + 1023) / 1024;
    const int b = threadIdx.x * per;
    int sum = 0;
    for (int k = 0; k < per; ++k)
        if (b + k < ntiles) sum += counts[b + k];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
        const int v = (threadIdx.x >= o) ? s_part[threadIdx.x - o] : 0;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    int run = s_part[threadIdx.x] - sum;
    for (int k = 0; k < per; ++k)
        if (b + k < ntiles) {
            tile_off[b + k] = run;
            cursor[b + k] = run;
            run += counts[b + k];
        }
    if (threadIdx.x == 1023) tile_off[ntiles] = s_part[1023];
}

template <int D>
__global__ void __launch_bounds__(1024)
plan_scatter_kernel(const float* __restrict__ coords, int64_t n, int ntiles, const int32_t* __restrict__ tile_id,
                    int32_t* __restrict__ cursor, int32_t* __restrict__ perm, float* __restrict__ coords_sorted) {
    extern __shared__ int s_plan_mem[];
    int* s_hist = s_plan_mem;            // local count per tile, then global base of this block's run
    for (int e = threadIdx.x; e < ntiles; e += blockDim.x) s_hist[e] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int t = 0, rank = 0;
    if (i < n) {
        t = tile_id[i];
        rank = atomicAdd(&s_hist[t], 1);  // rank of this point among the block's points of tile t
    }
    __syncthreads();
    for (int e = threadIdx.x; e < ntiles; e += blockDim.x) {
        const int c = s_hist[e];
        if (c) s_hist[e] = atomicAdd(&cursor[e], c);  // reserve a run in the tile's segment
    }
    __syncthreads();
    if (i < n) {
        const int pos = s_hist[t] + rank;
        perm[pos] = (int32_t)i;
#pragma unroll
        for (int d = 0; d < D; ++d) coords_sorted[(int64_t)pos * D + d] = __ldg(coords + i * D + d);
    }
}

// ---------------------------------------------------------------------------------------------
// per-tile level geometry
// ---------------------------------------------------------------------------------------------
template <int D>
struct TileGeom {
    int c0[SHACIRA_MAX_LEVELS][D];   // first cell of the tile's node box per level/axis
    int w[SHACIRA_MAX_LEVELS][D];    // nodes per axis (cells + 1)
    int off[SHACIRA_MAX_LEVELS + 1]; // first shared-memory node slot of the level
    int offp[SHACIRA_MAX_LEVELS];    // off - sum_d c0[d] * stride[d]: slot = offp + sum_d cell[d] * stride[d]
    unsigned magic[SHACIRA_MAX_LEVELS][D];  // ceil(2^32 / w): e / w == umulhi(e, magic) for the small e used here
    unsigned staged;                 // bit l: level l lives in shared memory for this tile
    int total;
    // backward accumulators: levels with a small node box keep one copy PER LANE (slot = off + node*32 + lane),
    // so the 32 lanes of a warp never collide on an address -- coarse levels otherwise serialise 32-way
    int acc_off[SHACIRA_MAX_LEVELS];
    int acc_mul[SHACIRA_MAX_LEVELS]; // 32 (lane-replicated) or 1
    int acc_total;
};
#ifndef SHACIRA_REP_BUDGET
#define SHACIRA_REP_BUDGET 2048
#endif
constexpr int kRepBudget = SHACIRA_REP_BUDGET;  // ints of lane-replicated accumulators per tile (all channels together)

// Cells reachable by points of the tile's axis interval [ti/g, (ti+1)/g]: locate() is monotone in t.
// Warp 0 computes everything: lane l owns level l; the slot offsets are a warp prefix sum. Levels are
// staged coarse to fine until the first one that does not fit `cap`; that one and all finer levels
// use the direct path.
template <int D>
__device__ __forceinline__ void tile_geometry(TileGeom<D>& tg, const LevelParams& lp, const int (&ti)[D], int g,
                                              int cap, int cap_acc = 0x3fffffff, int rep_budget = 0,
                                              int max_staged = SHACIRA_MAX_LEVELS) {
    if (threadIdx.x < 32) {
        const int l = threadIdx.x;
        const double inv_g = 1.0 / (double)g;  // g is a power of two: exact
        int nodes = 0, c0[D], w[D];
        if (l < lp.num_lods) {
            nodes = 1;
#pragma unroll
            for (int d = 0; d < D; ++d) {
                int ca, cb;
                float f, gg;
                locate((double)ti[d] * inv_g, lp.res[l], lp.hi[l], ca, f, gg);
                locate((double)(ti[d] + 1) * inv_g, lp.res[l], lp.hi[l], cb, f, gg);
                c0[d] = ca;
                w[d] = cb - ca + 2;
                nodes = (nodes > cap) ? nodes : nodes * w[d];  // saturate: anything above cap is unstaged anyway
            }
        }
        int incl = nodes;  // inclusive prefix sum over levels (values saturate far below 2^31)
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (l >= o) incl = min(incl + v, 0x3fffffff);
        }
        // accumulator slots: lane-replicated while the replicated prefix fits kRepBudget
        int rep_incl = min(nodes, 1 << 20) * 32;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, rep_incl, o);
            if (l >= o) rep_incl = min(rep_incl + v, 0x3fffffff);
        }
        const bool rep = (l < lp.num_lods) && rep_incl <= rep_budget;
        const int acc_size = rep ? nodes * 32 : nodes;
        int acc_incl = acc_size;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, acc_incl, o);
            if (l >= o) acc_incl = min(acc_incl + v, 0x3fffffff);
        }
        const bool fits = (l < lp.num_lods) && l < max_staged && incl <= cap && acc_incl <= cap_acc;
        const unsigned fit_mask = __ballot_sync(0xffffffffu, fits);
        // staged = the leading run of levels that fit
        const unsigned all = (lp.num_lods >= 32) ? 0xffffffffu : ((1u << lp.num_lods) - 1u);
        const unsigned miss = ~fit_mask & all;
        const unsigned staged = miss ? (fit_mask & ((1u << (__ffs(miss) - 1)) - 1u)) : fit_mask;
        const int first_unstaged = miss ? (__ffs(miss) - 1) : lp.num_lods;
        const int total = (first_unstaged > 0) ? __shfl_sync(0xffffffffu, incl, first_unstaged - 1) : 0;
        const int acc_total = (first_unstaged > 0) ? __shfl_sync(0xffffffffu, acc_incl, first_unstaged - 1) : 0;
        if (l < lp.num_lods) {
            const bool st = (staged >> l) & 1u;
            const int off = st ? incl - nodes : total;
            int offp = off, stride = 1;
#pragma unroll
            for (int d = 0; d < D; ++d) {
                tg.c0[l][d] = c0[d];
                tg.w[l][d] = w[d];
                tg.magic[l][d] = (unsigned)((0x100000000ull + (unsigned)w[d] - 1) / (unsigned)w[d]);
                offp -= c0[d] * stride;
                stride *= w[d];
            }
            tg.off[l] = off;
            tg.offp[l] = offp;
            tg.acc_off[l] = st ? acc_incl - acc_size : acc_total;
            tg.acc_mul[l] = rep ? 32 : 1;
        }
        if (l == 0) {
            tg.off[lp.num_lods] = total;
            tg.staged = staged;
            tg.total = total;
            tg.acc_total = acc_total;
        }
    }
    __syncthreads();
}

// node e (0 <= e < prod w) of level l -> level-local table row; -1 (or the last row when clamp_inside)
// for nodes outside the level, which only ever carry weight 0 (SURVEY Q4).
template <int D>
__device__ __forceinline__ int node_row(const TileGeom<D>& tg, const LevelParams& lp, int l, int e, bool clamp_inside) {
    const int res = lp.res[l];
    int nx[D];
    int r = e;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        if (d == D - 1) {
            nx[d] = tg.c0[l][d] + r;
        } else {
            const int q = (int)__umulhi((unsigned)r, tg.magic[l][d]);
            nx[d] = tg.c0[l][d] + (r - q * tg.w[l][d]);
            r = q;
        }
    }
    if ((lp.dense_mask >> l) & 1u) {
        // dense level: res^D < 2^30 rows, node coordinates <= res: the index fits 32 bits
        bool outside = nx[0] >= res;
        int idx = nx[0], mul = res;
#pragma unroll
        for (int d = 1; d < D; ++d) {
            outside |= nx[d] >= res;
            idx += nx[d] * mul;
            mul *= res;
        }
        if (outside || idx >= lp.rows[l]) return clamp_inside ? lp.rows[l] - 1 : -1;
        return idx;
    }
    uint32_t h = (uint32_t)nx[0];
    if (D > 1) h ^= (uint32_t)nx[1] * kPrimeY;
    if (D > 2) h ^= (uint32_t)nx[2] * kPrimeZ;
    return (int)(h & lp.hash_mask);
}

// Per-level constants of the hot loop, loaded ONCE per chunk of 4 levels into registers (the compiler
// cannot hoist them itself: the shared-memory atomics may alias them as far as it can tell).
struct LevelRegs {
    double resd;   // (double)res: x = float(resd * t)
    float hi;      // upper clamp bound
    int w0, w01;   // slot strides of axis 1 and axis 2
    int offp;      // slot = offp + sum_d cell[d] * stride[d]
    int accd;      // accumulator slot = (slot + accd) * amul + alane   (backward)
    int amul, alane;
    bool staged;
};

template <int D>
__device__ __forceinline__ void load_level_regs(const LevelParams& lp, const TileGeom<D>& tg, int l, LevelRegs& r) {
    r.resd = lp.resd[l];
    r.hi = lp.hi[l];
    r.w0 = tg.w[l][0];
    r.w01 = (D > 2) ? tg.w[l][0] * tg.w[l][1] : 0;
    r.offp = tg.offp[l];
    r.amul = tg.acc_mul[l];
    r.alane = (r.amul == 32) ? (int)(threadIdx.x & 31) : 0;
    // node index within the level = slot - off; accumulator = acc_off + node * amul + alane
    r.accd = -tg.off[l];
    r.alane += tg.acc_off[l];
    r.staged = (tg.staged >> l) & 1u;
}

// Cell, weights and the shared-memory slots of the 2^D corners of one point at one staged level.
template <int D>
struct Stencil {
    int slot[1 << D];
    float w[1 << D];
};

__device__ __forceinline__ void locate_r(double t, const LevelRegs& r, int32_t& cell, float& f, float& g) {
    float x = __double2float_rn(__dmul_rn(r.resd, t));
    x = fmaxf(0.0f, fminf(r.hi, x));
    float cf;
    floor_cell(x, cell, cf);
    f = __fsub_rn(x, cf);
    g = __fsub_rn(1.0f, f);
}

template <int D>
__device__ __forceinline__ void stencil(const double (&t)[D], const LevelRegs& r, Stencil<D>& s) {
    int p[D];
    float f[D], g1[D];
#pragma unroll
    for (int d = 0; d < D; ++d) locate_r(t[d], r, p[d], f[d], g1[d]);
    if constexpr (D == 2) {
        const int base = r.offp + p[0] + p[1] * r.w0;
        s.w[0] = __fmul_rn(g1[0], g1[1]);
        s.w[1] = __fmul_rn(g1[0], f[1]);
        s.w[2] = __fmul_rn(f[0], g1[1]);
        s.w[3] = __fmul_rn(f[0], f[1]);
        s.slot[0] = base;              // (x, y)
        s.slot[1] = base + r.w0;       // (x, y+1)
        s.slot[2] = base + 1;          // (x+1, y)
        s.slot[3] = base + r.w0 + 1;   // (x+1, y+1)
    } else {
        const int base = r.offp + p[0] + p[1] * r.w0 + p[2] * r.w01;
        const float gg = __fmul_rn(g1[0], g1[1]), gf = __fmul_rn(g1[0], f[1]);
        const float fg = __fmul_rn(f[0], g1[1]), ff = __fmul_rn(f[0], f[1]);
        s.w[0] = __fmul_rn(gg, g1[2]); s.w[1] = __fmul_rn(gg, f[2]);
        s.w[2] = __fmul_rn(gf, g1[2]); s.w[3] = __fmul_rn(gf, f[2]);
        s.w[4] = __fmul_rn(fg, g1[2]); s.w[5] = __fmul_rn(fg, f[2]);
        s.w[6] = __fmul_rn(ff, g1[2]); s.w[7] = __fmul_rn(ff, f[2]);
#pragma unroll
        for (int k = 0; k < 8; ++k) s.slot[k] = base + ((k >> 2) & 1) + ((k >> 1) & 1) * r.w0 + (k & 1) * r.w01;
    }
}

// z[ch] = sum_k w_k * q_k in the contraction order of the reference build: fma(v0,w0, v1*w1), then k = 2..
template <int NC, int C>
__device__ __forceinline__ void lerp_rows(const float (&v)[NC][C], const float (&w)[NC], float (&z)[C]) {
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {
        float acc = __fmul_rn(v[1][ch], w[1]);
        acc = __fmaf_rn(v[0][ch], w[0], acc);
#pragma unroll
        for (int k = 2; k < NC; ++k) acc = __fmaf_rn(v[k][ch], w[k], acc);
        z[ch] = acc;
    }
}

template <int C>
__device__ __forceinline__ void lds_row(const float* p, float (&v)[C]) {
    if constexpr (C == 1) {
        v[0] = p[0];
    } else if constexpr (C == 2) {
        const float2 a = *reinterpret_cast<const float2*>(p);
        v[0] = a.x; v[1] = a.y;
    } else {
        const float4 a = *reinterpret_cast<const float4*>(p);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    }
}

// Interpolated (rounded) latents of one point at one level: from the tile's staged nodes, or by
// direct global gathers when the level did not fit the tile's shared-memory box.
template <int D, int C>
__device__ __forceinline__ void interp_level(const double (&t)[D], const LevelParams& lp, const LevelRegs& r, int l,
                                             const float* s_nodes, const float* __restrict__ latents, int round_flag,
                                             float (&z)[C]) {
    constexpr int NC = 1 << D;
    float v[NC][C];
    if (r.staged) {
        Stencil<D> st;
        stencil<D>(t, r, st);
#pragma unroll
        for (int k = 0; k < NC; ++k) lds_row<C>(s_nodes + (size_t)st.slot[k] * C, v[k]);
        lerp_rows<NC, C>(v, st.w, z);
    } else {
        Corners<D> c;
        corners<D>(t, lp, l, c);
        const float* base = latents + (int64_t)lp.first[l] * C;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            load_row<C>(base + (int64_t)c.idx[k] * C, v[k]);
            if (round_flag) {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) v[k][ch] = rintf(v[k][ch]);
            }
        }
        lerp_rows<NC, C>(v, c.w, z);
    }
}

// Staged-level interpolation without the staged/direct branch: used when a whole chunk of levels is staged, so
// that the unrolled levels form ONE basic block and their dependent chains (DMUL -> F2F -> F2I -> LDS -> FMA)
// interleave -- the per-level branch otherwise serialises them.
template <int D, int C>
__device__ __forceinline__ void interp_staged(const double (&t)[D], const LevelRegs& r, const float* s_nodes,
                                              float (&z)[C]) {
    constexpr int NC = 1 << D;
    Stencil<D> st;
    stencil<D>(t, r, st);
    float v[NC][C];
#pragma unroll
    for (int k = 0; k < NC; ++k) lds_row<C>(s_nodes + (size_t)st.slot[k] * C, v[k]);
    lerp_rows<NC, C>(v, st.w, z);
}

// staged levels are a prefix of the levels and their slots are contiguous: level of slot e by binary search
template <int D>
__device__ __forceinline__ int level_of_slot(const TileGeom<D>& tg, int num_staged, int e) {
    int a = 0, b = num_staged;  // last staged level with off <= e
    while (b - a > 1) {
        const int m = (a + b) >> 1;
        if (tg.off[m] <= e) a = m; else b = m;
    }
    return a;
}

// Stage the (rounded) latents of every node of the tile's staged levels into shared memory: row index from the
// plan's node table, then the gather; unrolled so that each thread has kStageUnroll independent chains in flight.
#ifndef SHACIRA_STAGE_UNROLL
#define SHACIRA_STAGE_UNROLL 4
#endif
constexpr int kStageUnroll = SHACIRA_STAGE_UNROLL;
#ifndef SHACIRA_MIN_CTAS
#define SHACIRA_MIN_CTAS 7
#endif
#ifndef SHACIRA_LV
#define SHACIRA_LV 4
#endif
#ifndef SHACIRA_BWD_PREFETCH
#define SHACIRA_BWD_PREFETCH 0   // measured: the extra row registers spill at the 72-register cap (38.1 vs 36.7 us)
#endif
constexpr int kLv = SHACIRA_LV;  // levels per inner iteration (register blocking of the level loop): 4 or 2
template <int D, int C>
__device__ __forceinline__ void stage_nodes(const TileGeom<D>& tg, const int2* __restrict__ tab,
                                            const float* __restrict__ latents, int round_flag, float* s_nodes) {
    const int total = tg.total;
    for (int e0 = threadIdx.x; e0 < total; e0 += kTileThreads * kStageUnroll) {
        int row[kStageUnroll];
#pragma unroll
        for (int u = 0; u < kStageUnroll; ++u) {
            const int e = e0 + u * kTileThreads;
            row[u] = (e < total) ? __ldg(&tab[e]).x : 0;
        }
        float v[kStageUnroll][C];
#pragma unroll
        for (int u = 0; u < kStageUnroll; ++u) load_row<C>(latents + (int64_t)row[u] * C, v[u]);
#pragma unroll
        for (int u = 0; u < kStageUnroll; ++u) {
            const int e = e0 + u * kTileThreads;
            if (e < total) {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) s_nodes[(size_t)e * C + ch] = round_flag ? rintf(v[u][ch]) : v[u][ch];
            }
        }
    }
}

// Forward-kernel variant: the table rows of the thread's first kPre slots are requested at kernel entry, BEFORE the
// tile geometry is known (they only depend on the tile id), so their latency hides behind the tile_off load, the
// geometry and its barrier; the gathers of all kPre slots are then in flight together.
constexpr int kPre = 8;
__device__ __forceinline__ void prefetch_rows(const int2* __restrict__ tab, int stride, int (&pre)[kPre]) {
#pragma unroll
    for (int u = 0; u < kPre; ++u) {
        const int e = threadIdx.x + u * kTileThreads;
        pre[u] = (e < stride) ? __ldg(reinterpret_cast<const int*>(tab + e)) : 0;  // .x = absolute row
    }
}
template <int D, int C>
__device__ __forceinline__ void stage_nodes_prefetched(const TileGeom<D>& tg, const int2* __restrict__ tab,
                                                       const int (&pre)[kPre], const float* __restrict__ latents,
                                                       int round_flag, float* s_nodes) {
    const int total = tg.total;
    float v[kPre][C];
#pragma unroll
    for (int u = 0; u < kPre; ++u)
        if (threadIdx.x + u * kTileThreads < total) load_row<C>(latents + (int64_t)pre[u] * C, v[u]);
#pragma unroll
    for (int u = 0; u < kPre; ++u) {
        const int e = threadIdx.x + u * kTileThreads;
        if (e < total) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) s_nodes[(size_t)e * C + ch] = round_flag ? rintf(v[u][ch]) : v[u][ch];
        }
    }
    for (int e = threadIdx.x + kPre * kTileThreads; e < total; e += kTileThreads) {  // larger node boxes
        float w[C];
        load_row<C>(latents + (int64_t)__ldg(&tab[e]).x * C, w);
#pragma unroll
        for (int ch = 0; ch < C; ++ch) s_nodes[(size_t)e * C + ch] = round_flag ? rintf(w[ch]) : w[ch];
    }
}

// Fills one tile's row of the node table (see PlanView::node_tab). One CTA per tile.
template <int D>
__global__ void __launch_bounds__(kTileThreads)
plan_nodes_kernel(const __grid_constant__ LevelParams lp, int g, int cap, int2* __restrict__ node_tab) {
    __shared__ TileGeom<D> tg;
    int ti[D];
    {
        int r = blockIdx.x;
#pragma unroll
        for (int d = 0; d < D; ++d) { ti[d] = r % g; r /= g; }
    }
    tile_geometry<D>(tg, lp, ti, g, cap);
    const int ns = __popc(tg.staged);
    int2* tab = node_tab + (size_t)blockIdx.x * cap;
    for (int e = threadIdx.x; e < tg.total; e += kTileThreads) {
        const int l = level_of_slot<D>(tg, ns, e);
        const int row = node_row<D>(tg, lp, l, e - tg.off[l], false);
        const int inside = (row >= 0) ? row : lp.rows[l] - 1;  // a readable row for the staging gather
        tab[e] = make_int2(lp.first[l] + inside, l | (row >= 0 ? 0 : kNodeInvalid));
    }
}

// ---------------------------------------------------------------------------------------------
// forward: 4 levels per iteration, outputs written as 16-byte vectors (needs num_lods % 4 == 0)
// ---------------------------------------------------------------------------------------------
template <int D, int C, int F>
__global__ void __launch_bounds__(kTileThreads, (C * F <= 4) ? SHACIRA_MIN_CTAS : 3)
latent_fwd_tiled_kernel(const PlanView pv, const float* __restrict__ latents, const __grid_constant__ LevelParams lp,
                        const float* __restrict__ A, const float* __restrict__ shift, int per_level, int round_flag,
                        float* __restrict__ feats, int cap, int rows_via_smem) {
    extern __shared__ float s_dyn[];
    __shared__ TileGeom<D> tg;
    const int L = lp.num_lods;
    const int nA = per_level ? L : 1;
    float* s_nodes = s_dyn;                  // [cap][C]
    float* s_A = s_dyn + (size_t)cap * C;    // [nA][C][F]
    float* s_shift = s_A + nA * C * F;       // [nA][F]
    // rows_via_smem (rows go back to their ORIGINAL index, i.e. scattered): a batch's rows are collected in shared memory
    // and written as whole contiguous rows by neighbouring threads, instead of one 16-byte piece per thread and level
    // chunk -- every row then reaches L2 as full sectors in one request
    const int RL = L * F, RS = RL + 4;       // row length / padded stride (floats): conflict-free 16-byte accesses
    float* s_rows = s_dyn + (((size_t)cap * C + nA * C * F + nA * F + 3) & ~(size_t)3);   // [kTileThreads * kPts][RS]
    int* s_orig = reinterpret_cast<int*>(s_rows + (size_t)kTileThreads * kPts * RS);      // [kTileThreads * kPts]
    const int tile = blockIdx.x;
    const int beg = pv.tile_off[tile], end = pv.tile_off[tile + 1];
    if (beg == end) return;
    int ti[D];
    {
        int r = tile;
#pragma unroll
        for (int d = 0; d < D; ++d) { ti[d] = r % pv.g; r /= pv.g; }
    }
    const int2* tab = pv.node_tab + (size_t)tile * pv.node_stride;
    int pre[kPre];
    prefetch_rows(tab, pv.node_stride, pre);
    for (int e = threadIdx.x; e < nA * C * F; e += kTileThreads) s_A[e] = A[e];
    for (int e = threadIdx.x; e < nA * F; e += kTileThreads) s_shift[e] = shift ? shift[e] : 0.0f;
    tile_geometry<D>(tg, lp, ti, pv.g, cap);
    stage_nodes_prefetched<D, C>(tg, tab, pre, latents, round_flag, s_nodes);
    __syncthreads();

    for (int base = beg; base < end; base += kTileThreads * kPts) {
        // kPts points per thread: permutation entries and coordinates of all of them are requested first
        int orig[kPts];
        double t[kPts][D];
#pragma unroll
        for (int k = 0; k < kPts; ++k) {
            const int j = base + k * kTileThreads + threadIdx.x;
            orig[k] = -1;
#pragma unroll
            for (int d = 0; d < D; ++d) t[k][d] = 0.5;
            if (j < end) {
                orig[k] = pv.perm ? __ldg(pv.perm + j) : j;
                load_unit_coords<D>(pv.coords_sorted, j, t[k]);
            }
        }
        for (int l0 = 0; l0 < L; l0 += kLv) {
            LevelRegs lr[kLv];
            float sh[kLv][F], Am[kLv][C * F];
#pragma unroll
            for (int q = 0; q < kLv; ++q) {
                load_level_regs<D>(lp, tg, l0 + q, lr[q]);
                const int la = per_level ? (l0 + q) : 0;
#pragma unroll
                for (int jf = 0; jf < F; ++jf) sh[q][jf] = s_shift[la * F + jf];
#pragma unroll
                for (int e = 0; e < C * F; ++e) Am[q][e] = s_A[la * C * F + e];
            }
            bool all_staged = true;
#pragma unroll
            for (int q = 0; q < kLv; ++q) all_staged &= lr[q].staged;
#pragma unroll
            for (int k = 0; k < kPts; ++k) {
                if (orig[k] < 0) continue;
                float o[kLv * F];
                float z[kLv][C];
                if (all_staged) {  // uniform: one basic block for the kLv levels
#pragma unroll
                    for (int q = 0; q < kLv; ++q) interp_staged<D, C>(t[k], lr[q], s_nodes, z[q]);
                } else {
#pragma unroll
                    for (int q = 0; q < kLv; ++q)
                        interp_level<D, C>(t[k], lp, lr[q], l0 + q, s_nodes, latents, round_flag, z[q]);
                }
#pragma unroll
                for (int q = 0; q < kLv; ++q) {
#pragma unroll
                    for (int jf = 0; jf < F; ++jf) {
                        float acc = sh[q][jf];
#pragma unroll
                        for (int ch = 0; ch < C; ++ch) acc = __fmaf_rn(z[q][ch], Am[q][ch * F + jf], acc);
                        o[q * F + jf] = acc;
                    }
                }
                if (rows_via_smem) store_row<kLv * F>(s_rows + (size_t)(k * kTileThreads + threadIdx.x) * RS + l0 * F, o);
                else store_row<kLv * F>(feats + (int64_t)orig[k] * L * F + l0 * F, o);
            }
        }
        if (rows_via_smem) {
#pragma unroll
            for (int k = 0; k < kPts; ++k) s_orig[k * kTileThreads + threadIdx.x] = orig[k];
            __syncthreads();
            const int pieces = RL >> 2;   // 16-byte pieces per row
            for (int idx = threadIdx.x; idx < kTileThreads * kPts * pieces; idx += kTileThreads) {
                const int r = idx / pieces, pc = idx - r * pieces;
                const int og = s_orig[r];
                if (og >= 0)
                    *reinterpret_cast<float4*>(feats + (int64_t)og * RL + 4 * pc) =
                        *reinterpret_cast<const float4*>(s_rows + (size_t)r * RS + 4 * pc);
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// Power-of-two scale so that the sum of up to 2^k terms of magnitude <= m stays below 2^30.
__device__ __forceinline__ float fixed_scale(float m, int k, float& inv) {
    if (!(m > 0.0f) || !isfinite(m)) {
        // all-zero level: nothing to add. Inf/NaN upstream gradients cannot be scaled: poison the level's nodes of
        // this tile with NaN at flush time, like the reference's float atomics would
        inv = (m != m || m > 3.0e38f) ? __int_as_float(0x7fc00000) : 0.0f;
        return 0.0f;
    }
    const int ex = (int)((__float_as_uint(m) >> 23) & 0xffu) - 126;   // m < 2^ex (exponent field; subnormals: 2^-126)
    // sums of 2^k terms below 2^30, and every single term below 2^21 so that fixed_rn() can convert without the XU pipe
    const int e = max(-126, min(min(30 - k, 21) - ex, 126));
    inv = __int_as_float((127 - e) << 23);   // 2^-e, exact
    return __int_as_float((127 + e) << 23);  // 2^e
}
// round-to-nearest-even float -> int for |v| <= 2^22 as one FADD + one IADD (v + 1.5 * 2^23 lands in [2^23, 2^24), where
// floats are the integers): F2I sits on the quarter-rate conversion pipe with scoreboard latency, 64 of them per point.
__device__ __forceinline__ int fixed_rn(float v) { return __float_as_int(__fadd_rn(v, 12582912.0f)) - 0x4B400000; }

// Two formulations, chosen at compile time:
//   scatter-gz (SG = false): accumulate w_k * (A^T g) per node (C channels). Decoder gradients, when wanted,
//       need the interpolated latents z per point: the tile stages the latents and re-interpolates.
//   scatter-g  (SG = true, used when decoder gradients are wanted and F <= C): accumulate G[node] = sum w_k * g
//       per node (F channels). Everything else is linear in G and is applied ONCE PER NODE at flush time:
//       grad_latent[node] = A G[node];  grad_A += q[node] G[node]^T;  grad_shift += G[node]  (sum_k w_k = 1).
//       That is ~2-3 nodes per point instead of 2^D * L corner visits per point.
template <int D, int C, int F, bool DEC>
__global__ void __launch_bounds__(kTileThreads, (C * F <= 4) ? SHACIRA_MIN_CTAS : 3)
latent_bwd_tiled_kernel(const PlanView pv, const float* __restrict__ grad_out, const float* __restrict__ latents,
                        const __grid_constant__ LevelParams lp, const float* __restrict__ A, int per_level,
                        int round_flag, float* __restrict__ grad_latents, float* __restrict__ grad_A,
                        float* __restrict__ grad_shift, int cap, int cap_acc, const float* __restrict__ level_max,
                        int max_staged, int skip_direct) {
    // max_staged / skip_direct (3D): stage exactly the first max_staged levels (the host sized `cap` for them) and leave
    // every other level to the lane-pair kernel that runs beside this one (latent_bwd3d_lp_kernel, skip_mask).
    constexpr bool SG = DEC && (F <= C);
    constexpr bool ZP = DEC && !SG;          // per-point z recomputation
    constexpr int CA = SG ? F : C;           // accumulator channels
    extern __shared__ float s_dyn[];
    __shared__ TileGeom<D> tg;
    __shared__ unsigned s_gmax[SHACIRA_MAX_LEVELS];   // max |accumulated quantity| per level over the batch
    __shared__ float s_scale[SHACIRA_MAX_LEVELS], s_inv[SHACIRA_MAX_LEVELS];
    const int L = lp.num_lods;
    const int nA = per_level ? L : 1;
    constexpr int NW = kTileThreads / 32;
    constexpr int NC = 1 << D;
    constexpr int KP = (F == 1) ? kPts : ((F == 2) ? 2 : 1);  // keeps the in-flight rows within ~16 registers
    int* s_acc = reinterpret_cast<int*>(s_dyn);                           // [cap_acc][CA] fixed-point node sums
    float* s_lat = s_dyn + (size_t)cap_acc * CA;                          // [cap][C] staged latents (DEC)
    float* s_A = s_lat + (DEC ? (size_t)cap * C : 0);                     // [nA][C][F]
    float* s_gA = s_A + nA * C * F;                                       // ZP: [NW][L][C][F]; SG: [L][C][F]
    float* s_gS = s_gA + (ZP ? NW : 1) * (DEC ? L * C * F : 0);           // ZP: [NW][L][F];    SG: [L][F]
    const int tile = blockIdx.x;
    const int beg = pv.tile_off[tile], end = pv.tile_off[tile + 1];
    if (beg == end) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ti[D];
    {
        int r = tile;
#pragma unroll
        for (int d = 0; d < D; ++d) { ti[d] = r % pv.g; r /= pv.g; }
    }
    for (int e = threadIdx.x; e < nA * C * F; e += kTileThreads) s_A[e] = A[e];
    if (DEC)
        for (int e = threadIdx.x; e < (ZP ? NW : 1) * L * (C * F + F); e += kTileThreads) s_gA[e] = 0.0f;
    tile_geometry<D>(tg, lp, ti, pv.g, cap, cap_acc, cap_acc - cap, max_staged);
    bool staged_lat = false;
    // levels this launch touches: all of them, or the staged prefix rounded up to the level blocking
    const int Lrun = skip_direct ? min(L, ((__popc(tg.staged) + kLv - 1) / kLv) * kLv) : L;

    // Points per thread held in registers for a whole batch: each 16-byte piece of a gradient row is read ONCE, its
    // levels' maxima (the fixed-point scales) are reduced from the registers, and after one barrier the same registers
    // feed the accumulation -- no separate max pass over the rows (round 1: a second, latency-bound read of every row).
    // A tile with more points than one register batch (uneven sample sets; the test suite's clustered case) runs the
    // max pass of round 1 over up to kBatch points first and then several register batches into the SAME accumulators:
    // one zero-fill and one flush per kBatch points either way.
    constexpr int KB = (F == 1) ? 3 : ((F == 2) ? 2 : 1);
    constexpr int kBatchPts = kTileThreads * KB;
    for (int s0 = beg; s0 < end; s0 += kBatch) {
        const int s1 = min(end, s0 + kBatch);
        // (the 3D staged-prefix launches always take this form: their tiles average 128 samples around a batch of 128,
        // measured 206 / 243 us against 220 / 253 us with per-batch maxima and 263 us with two samples per thread)
        const bool multi = skip_direct || (s1 - s0) > kBatchPts;
        int kbits = 0;
        while ((1 << kbits) < (s1 - s0)) ++kbits;
        {
            const int n4 = (tg.acc_total * CA + 3) >> 2;  // capacities are multiples of 4 slots: whole int4 stores
            int4* z4 = reinterpret_cast<int4*>(s_acc);
            for (int e = threadIdx.x; e < n4; e += kTileThreads) z4[e] = make_int4(0, 0, 0, 0);
        }
        if (threadIdx.x < SHACIRA_MAX_LEVELS) {
            unsigned bound = 0u;
            if (level_max && threadIdx.x < L) {
                // The caller knows an upper bound of |grad_output| per level (e.g. the kernel that produced the rows
                // reduced it on the way). The bound of the accumulated quantity is |g| itself in scatter-g mode, else
                // |A^T g| <= max|g| * max_c sum_f |A[c][f]|.
                float m = fabsf(__ldg(level_max + threadIdx.x * F));
#pragma unroll
                for (int jf = 1; jf < F; ++jf) m = nan_max(m, fabsf(__ldg(level_max + threadIdx.x * F + jf)));
                if (!SG) {
                    const int la = per_level ? threadIdx.x : 0;
                    float amax = 0.0f;
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) {
                        float sum = 0.0f;
#pragma unroll
                        for (int jf = 0; jf < F; ++jf) sum += fabsf(__ldg(A + (la * C + ch) * F + jf));
                        amax = fmaxf(amax, sum);
                    }
                    m *= amax;
                }
                bound = __float_as_uint(m);
            }
            s_gmax[threadIdx.x] = bound;
        }
        if (multi && !level_max) {
            __syncthreads();   // s_gmax cleared
            for (int base = s0; base < s1; base += kTileThreads) {
                const int j = base + threadIdx.x;
                const float* rowp = (j < s1) ? grad_out + (int64_t)(pv.perm ? __ldg(pv.perm + j) : j) * L * F : nullptr;
                for (int l0 = 0; l0 < Lrun; l0 += kLv) {
                    float g[kLv * F];
#pragma unroll
                    for (int e = 0; e < kLv * F; ++e) g[e] = 0.0f;
                    if (rowp) load_row<kLv * F>(rowp + l0 * F, g);
#pragma unroll
                    for (int q = 0; q < kLv; ++q) {
                        float m = 0.0f;
                        if (SG) {
#pragma unroll
                            for (int jf = 0; jf < F; ++jf) m = nan_max(m, fabsf(g[q * F + jf]));
                        } else {
                            const int la = per_level ? (l0 + q) : 0;
#pragma unroll
                            for (int ch = 0; ch < C; ++ch) {
                                float acc = 0.0f;
#pragma unroll
                                for (int jf = 0; jf < F; ++jf) acc = __fmaf_rn(g[q * F + jf], s_A[(la * C + ch) * F + jf], acc);
                                m = nan_max(m, fabsf(acc));
                            }
                        }
                        const unsigned wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                        if (lane == 0 && wm) atomicMax(&s_gmax[l0 + q], wm);
                    }
                }
            }
        }
        const bool own_max = !level_max && !multi;   // the chunk loop reduces the maxima itself (one register batch)
      for (int b0 = s0; b0 < s1; b0 += kBatchPts) {
        const int b1 = min(s1, b0 + kBatchPts);
        // this thread's points of the batch: row index, coordinates
        // (coordinates as floats when a thread holds several points -- the double unit coordinate is then rebuilt per
        // level chunk, 6 registers instead of 12 at the image shape -- and as doubles when it holds one)
        constexpr bool kKeepUnit = KB * D <= 4;
        int64_t rowk[KB];
        float ck[KB][D];
        double tu[kKeepUnit ? KB : 1][D];
        bool livek[KB];
#pragma unroll
        for (int k = 0; k < KB; ++k) {
            const int j = b0 + k * kTileThreads + threadIdx.x;
            livek[k] = j < b1;
            rowk[k] = 0;
#pragma unroll
            for (int d = 0; d < D; ++d) ck[k][d] = 0.0f;
            if (livek[k]) {
                rowk[k] = (int64_t)(pv.perm ? __ldg(pv.perm + j) : j) * L * F;
#pragma unroll
                for (int d = 0; d < D; ++d) ck[k][d] = __ldg(pv.coords_sorted + (int64_t)j * D + d);
            }
            if (kKeepUnit) {
#pragma unroll
                for (int d = 0; d < D; ++d) tu[k][d] = unit_coord(ck[k][d]);
            }
        }
        // latents for the decoder gradients (ZP: per-point z; SG: q[node] at flush), staged once, behind the loads above
        if (DEC && !staged_lat) {
            stage_nodes<D, C>(tg, pv.node_tab + (size_t)tile * pv.node_stride, latents, round_flag, s_lat);
            staged_lat = true;
        }
        // the first chunk's gradient pieces are requested before the barrier, every later chunk's while the previous one
        // is being accumulated (SHACIRA_BWD_PREFETCH: one more set of row registers)
        float gk[KB][kLv * F];
#pragma unroll
        for (int k = 0; k < KB; ++k) {
#pragma unroll
            for (int e = 0; e < kLv * F; ++e) gk[k][e] = 0.0f;
            if (livek[k] && Lrun > 0) load_row<kLv * F>(grad_out + rowk[k], gk[k]);
        }
        __syncthreads();
        for (int l0 = 0; l0 < Lrun; l0 += kLv) {
#if !SHACIRA_BWD_PREFETCH
            if (l0 > 0) {
#pragma unroll
                for (int k = 0; k < KB; ++k)
                    if (livek[k]) load_row<kLv * F>(grad_out + rowk[k] + l0 * F, gk[k]);
            }
#endif
            if (own_max) {
                // maxima of what this chunk of levels will accumulate, over the batch: REDUX over the warp, one shared
                // atomicMax per warp and level; NaN propagates (nan_max; its bit pattern compares above +Inf)
#pragma unroll
                for (int q = 0; q < kLv; ++q) {
                    const int l = l0 + q;
                    float m = 0.0f;
#pragma unroll
                    for (int k = 0; k < KB; ++k) {
                        if (SG) {
#pragma unroll
                            for (int jf = 0; jf < F; ++jf) m = nan_max(m, fabsf(gk[k][q * F + jf]));
                        } else {
                            const int la = per_level ? l : 0;
#pragma unroll
                            for (int ch = 0; ch < C; ++ch) {
                                float acc = 0.0f;
#pragma unroll
                                for (int jf = 0; jf < F; ++jf)
                                    acc = __fmaf_rn(gk[k][q * F + jf], s_A[(la * C + ch) * F + jf], acc);
                                m = nan_max(m, fabsf(acc));
                            }
                        }
                    }
                    const unsigned wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                    if (lane == 0 && wm) atomicMax(&s_gmax[l], wm);
                }
                __syncthreads();
            }
#if SHACIRA_BWD_PREFETCH
            float gn[KB][kLv * F];
#pragma unroll
            for (int k = 0; k < KB; ++k) {
#pragma unroll
                for (int e = 0; e < kLv * F; ++e) gn[k][e] = 0.0f;
                if (livek[k] && l0 + kLv < Lrun) load_row<kLv * F>(grad_out + rowk[k] + (l0 + kLv) * F, gn[k]);
            }
#endif
            float accS[ZP ? kLv * F : 1], accA[ZP ? kLv * C * F : 1];
            if (ZP) {
#pragma unroll
                for (int e = 0; e < kLv * F; ++e) accS[e] = 0.0f;
#pragma unroll
                for (int e = 0; e < kLv * C * F; ++e) accA[e] = 0.0f;
            }
            LevelRegs lr[kLv];
            float scq[kLv], Am[kLv][SG ? 1 : C * F];
#pragma unroll
            for (int q = 0; q < kLv; ++q) {
                load_level_regs<D>(lp, tg, l0 + q, lr[q]);
                float inv_unused;
                scq[q] = fixed_scale(__uint_as_float(s_gmax[l0 + q]), kbits, inv_unused);
                if (!SG) {
                    const int la = per_level ? (l0 + q) : 0;
#pragma unroll
                    for (int e = 0; e < C * F; ++e) Am[q][e] = s_A[la * C * F + e];
                }
            }
            bool all_staged = true;
#pragma unroll
            for (int q = 0; q < kLv; ++q) all_staged &= lr[q].staged;
            {
#pragma unroll
                for (int k = 0; k < KB; ++k) {
                    if (!livek[k]) continue;
                    double tk1[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) tk1[d] = kKeepUnit ? tu[k][d] : unit_coord(ck[k][d]);
                    const double (&t)[D] = tk1;
                    const float (&g)[kLv * F] = gk[k];
                    if (all_staged) {
                        // every level of the chunk is staged (uniform): stencils first, as one basic block, so the
                        // kLv dependent chains interleave; then the shared-memory adds
                        Stencil<D> st[kLv];
#pragma unroll
                        for (int q = 0; q < kLv; ++q) stencil<D>(t, lr[q], st[q]);
#pragma unroll
                        for (int q = 0; q < kLv; ++q) {
                            float gz[CA];
                            if (SG) {
#pragma unroll
                                for (int jf = 0; jf < F; ++jf) gz[jf] = g[q * F + jf];
                            } else {
#pragma unroll
                                for (int ch = 0; ch < C; ++ch) {
                                    float acc = 0.0f;
#pragma unroll
                                    for (int jf = 0; jf < F; ++jf) acc = __fmaf_rn(g[q * F + jf], Am[q][ch * F + jf], acc);
                                    gz[ch] = acc;
                                }
                            }
#pragma unroll
                            for (int ch = 0; ch < CA; ++ch) {
                                const float gs = __fmul_rn(gz[ch], scq[q]);  // power-of-two scale: exact
#pragma unroll
                                for (int kk = 0; kk < NC; ++kk)
                                    atomicAdd(&s_acc[(size_t)((st[q].slot[kk] + lr[q].accd) * lr[q].amul + lr[q].alane) * CA + ch],
                                              fixed_rn(__fmul_rn(gs, st[q].w[kk])));
                            }
                            if (ZP) {
                                float v[NC][C], z[C];
#pragma unroll
                                for (int kk = 0; kk < NC; ++kk) lds_row<C>(s_lat + (size_t)st[q].slot[kk] * C, v[kk]);
                                lerp_rows<NC, C>(v, st[q].w, z);
#pragma unroll
                                for (int jf = 0; jf < F; ++jf) {
                                    accS[q * F + jf] += g[q * F + jf];
#pragma unroll
                                    for (int ch = 0; ch < C; ++ch)
                                        accA[(q * C + ch) * F + jf] = __fmaf_rn(z[ch], g[q * F + jf], accA[(q * C + ch) * F + jf]);
                                }
                            }
                        }
                        continue;
                    }
#pragma unroll
                    for (int q = 0; q < kLv; ++q) {
                        const int l = l0 + q;
                        if (skip_direct && !lr[q].staged) continue;
                        float gz[CA], z[C];
#pragma unroll
                        for (int ch = 0; ch < C; ++ch) z[ch] = 0.0f;
                        if (SG) {
#pragma unroll
                            for (int jf = 0; jf < F; ++jf) gz[jf] = g[q * F + jf];
                        } else {
#pragma unroll
                            for (int ch = 0; ch < C; ++ch) {
                                float acc = 0.0f;
#pragma unroll
                                for (int jf = 0; jf < F; ++jf) acc = __fmaf_rn(g[q * F + jf], Am[q][ch * F + jf], acc);
                                gz[ch] = acc;
                            }
                        }
                        if (lr[q].staged) {
                            Stencil<D> st;
                            stencil<D>(t, lr[q], st);
                            const float sc = scq[q];
#pragma unroll
                            for (int ch = 0; ch < CA; ++ch) {
                                const float gs = __fmul_rn(gz[ch], sc);  // power-of-two scale: exact
#pragma unroll
                                for (int kk = 0; kk < NC; ++kk)
                                    atomicAdd(&s_acc[(size_t)((st.slot[kk] + lr[q].accd) * lr[q].amul + lr[q].alane) * CA + ch],
                                              fixed_rn(__fmul_rn(gs, st.w[kk])));
                            }
                            if (ZP) {
                                float v[NC][C];
#pragma unroll
                                for (int kk = 0; kk < NC; ++kk) lds_row<C>(s_lat + (size_t)st.slot[kk] * C, v[kk]);
                                lerp_rows<NC, C>(v, st.w, z);
                            }
                        } else {  // direct level: float REDG to global (and, for the decoder, gathers for z)
                            Corners<D> c;
                            corners<D>(t, lp, l, c);
                            float gl[C];
                            if (SG) {
                                const int la = per_level ? l : 0;
#pragma unroll
                                for (int ch = 0; ch < C; ++ch) {
                                    float acc = 0.0f;
#pragma unroll
                                    for (int jf = 0; jf < F; ++jf) acc = __fmaf_rn(g[q * F + jf], s_A[(la * C + ch) * F + jf], acc);
                                    gl[ch] = acc;
                                }
                            } else {
#pragma unroll
                                for (int ch = 0; ch < C; ++ch) gl[ch] = gz[ch];
                            }
                            float* gbase = grad_latents + (int64_t)lp.first[l] * C;
#pragma unroll
                            for (int kk = 0; kk < NC; ++kk) {
                                float gv[C];
#pragma unroll
                                for (int ch = 0; ch < C; ++ch) gv[ch] = __fmul_rn(gl[ch], c.w[kk]);
                                red_add_row<C>(gbase + (int64_t)c.idx[kk] * C, gv);
                            }
                            if (DEC) {
                                const float* lb = latents + (int64_t)lp.first[l] * C;
                                float v[NC][C];
#pragma unroll
                                for (int kk = 0; kk < NC; ++kk) {
                                    load_row<C>(lb + (int64_t)c.idx[kk] * C, v[kk]);
                                    if (round_flag) {
#pragma unroll
                                        for (int ch = 0; ch < C; ++ch) v[kk][ch] = rintf(v[kk][ch]);
                                    }
                                }
                                lerp_rows<NC, C>(v, c.w, z);
                                if (SG) {  // direct levels are rare on this path: warp-reduce per point
#pragma unroll
                                    for (int jf = 0; jf < F; ++jf) {
                                        atomicAdd(&s_gS[l * F + jf], g[q * F + jf]);
#pragma unroll
                                        for (int ch = 0; ch < C; ++ch) atomicAdd(&s_gA[(l * C + ch) * F + jf], z[ch] * g[q * F + jf]);
                                    }
                                }
                            }
                        }
                        if (ZP) {
#pragma unroll
                            for (int jf = 0; jf < F; ++jf) {
                                accS[q * F + jf] += g[q * F + jf];
#pragma unroll
                                for (int ch = 0; ch < C; ++ch)
                                    accA[(q * C + ch) * F + jf] = __fmaf_rn(z[ch], g[q * F + jf], accA[(q * C + ch) * F + jf]);
                            }
                        }
                    }
                }
            }
            if (ZP) {
#pragma unroll
                for (int e = 0; e < kLv * F; ++e) {
                    const float v = warp_sum(accS[e]);
                    if (lane == 0) s_gS[(warp * L + l0) * F + e] += v;   // [l0 + q][jf] is contiguous: e = q*F + jf
                }
#pragma unroll
                for (int e = 0; e < kLv * C * F; ++e) {
                    const float v = warp_sum(accA[e]);
                    if (lane == 0) s_gA[(warp * L + l0) * C * F + e] += v;  // e = (q*C + ch)*F + jf
                }
            }
#if SHACIRA_BWD_PREFETCH
#pragma unroll
            for (int k = 0; k < KB; ++k)
#pragma unroll
                for (int e = 0; e < kLv * F; ++e) gk[k][e] = gn[k][e];
#endif
        }
      }   // register batches of this span
        if (threadIdx.x < L) {
            float inv;
            fixed_scale(__uint_as_float(s_gmax[threadIdx.x]), kbits, inv);
            s_inv[threadIdx.x] = inv;
        }
        // the flush's node-table entries (absolute row, level) are requested now, ahead of the barrier: the flush is
        // the tail of the CTA, nothing else would hide their latency
        constexpr int kFlushPre = 9;
        int2 pre[kFlushPre];
        {
            const int2* tab_p = pv.node_tab ? pv.node_tab + (size_t)tile * pv.node_stride : nullptr;
#pragma unroll
            for (int u = 0; u < kFlushPre; ++u) {
                const int e = threadIdx.x + u * kTileThreads;
                pre[u] = (tab_p && e < tg.total) ? __ldg(tab_p + e) : make_int2(0, 0);
            }
        }
        __syncthreads();
        // flush: one float REDG per touched node (+ the per-node decoder gradients in scatter-g mode)
        // flush: one float REDG per touched node (+ the per-node decoder gradients in scatter-g mode).
        // pS / pA: scatter-g decoder partial sums of this thread.
        float pS[SG ? F : 1], pA[SG ? C * F : 1];
#pragma unroll
        for (int e = 0; e < (SG ? F : 1); ++e) pS[e] = 0.0f;
#pragma unroll
        for (int e = 0; e < (SG ? C * F : 1); ++e) pA[e] = 0.0f;
        const int num_staged = __popc(tg.staged);
        const int total_nodes = tg.total;
        const int2* tab = pv.node_tab ? pv.node_tab + (size_t)tile * pv.node_stride : nullptr;
        // One thread per node over ALL staged levels at once (flat slot index; level and table row come from the
        // plan's node table): full lanes on the small coarse levels, no per-node index math. With per-level
        // decoders in scatter-g mode the partial sums must be kept per level, so that (rare) case walks level by level.
        const bool by_level = SG && per_level;
        // one node: fixed-point sums -> float, one REDG (+ the per-node decoder gradients in scatter-g mode)
        auto flush_node = [&](int e, int2 ent) {
            const int l = ent.y & 0xff;
            const int nloc = e - tg.off[l];
            const float inv = s_inv[l];
            const bool rep = tg.acc_mul[l] == 32;
            const int abase = tg.acc_off[l];
            bool any = false;
            float gv[CA];
#pragma unroll
            for (int ch = 0; ch < CA; ++ch) {
                int qv = 0;
                if (rep) {
                    // the node's 32 lane copies, read starting at this thread's lane: 32 different banks per warp
#pragma unroll 8
                    for (int jj = 0; jj < 32; ++jj) qv += s_acc[(size_t)(abase + nloc * 32 + ((lane + jj) & 31)) * CA + ch];
                } else {
                    qv = s_acc[(size_t)(abase + nloc) * CA + ch];
                }
                any |= (qv != 0);
                gv[ch] = (float)qv * inv;
            }
            if (inv != inv) {  // non-finite upstream gradient in this tile/level (see fixed_scale)
                any = true;
#pragma unroll
                for (int ch = 0; ch < CA; ++ch) gv[ch] = inv;
            }
            if (!any || (ent.y & kNodeInvalid)) return;
            float* dst = grad_latents + (int64_t)ent.x * C;
            if constexpr (SG) {
                const int la = per_level ? l : 0;
                float qn[C], gl[C];
                lds_row<C>(s_lat + (size_t)e * C, qn);  // staged (already rounded)
#pragma unroll
                for (int ch = 0; ch < C; ++ch) {
                    float acc = 0.0f;
#pragma unroll
                    for (int jf = 0; jf < F; ++jf) {
                        acc = __fmaf_rn(gv[jf], s_A[(la * C + ch) * F + jf], acc);
                        pA[ch * F + jf] = __fmaf_rn(qn[ch], gv[jf], pA[ch * F + jf]);
                    }
                    gl[ch] = acc;
                }
#pragma unroll
                for (int jf = 0; jf < F; ++jf) pS[jf] += gv[jf];
                red_add_row<C>(dst, gl);
            } else {
                red_add_row<C>(dst, gv);
            }
        };
        auto node_entry = [&](int e) -> int2 {
            if (pv.node_tab) return __ldg(&tab[e]);
            // no node table (3D: it would be tens of MB): level and table row from the tile geometry
            const int le = level_of_slot<D>(tg, num_staged, e);
            const int r = node_row<D>(tg, lp, le, e - tg.off[le], false);
            return make_int2(lp.first[le] + max(r, 0), le | (r >= 0 ? 0 : kNodeInvalid));
        };
        for (int lvl = 0; lvl < (by_level ? num_staged : 1); ++lvl) {
            const int e_begin = by_level ? tg.off[lvl] : 0;
            const int e_end = by_level ? ((lvl + 1 < num_staged) ? tg.off[lvl + 1] : total_nodes) : total_nodes;
            int e = e_begin + threadIdx.x;
            if (!by_level && pv.node_tab) {
                // the first kFlushPre entries of this thread were requested before the barrier (see `pre`)
#pragma unroll
                for (int u = 0; u < kFlushPre; ++u, e += kTileThreads)
                    if (e < e_end) flush_node(e, pre[u]);
            }
            for (; e < e_end; e += kTileThreads) flush_node(e, node_entry(e));
            if (SG) {
                // one shared decoder: only the SUM over the L rows is defined (the caller adds them), so every tile
                // puts its share in row (tile mod L): 1024 CTAs adding into ONE address serialise in L2
                const int dl = by_level ? lvl : (tile % L);
#pragma unroll
                for (int e = 0; e < F; ++e) {
                    const float v = warp_sum(pS[e]);
                    if (lane == 0 && v != 0.0f) atomicAdd(&s_gS[dl * F + e], v);
                    pS[e] = 0.0f;
                }
#pragma unroll
                for (int e = 0; e < C * F; ++e) {
                    const float v = warp_sum(pA[e]);
                    if (lane == 0 && v != 0.0f) atomicAdd(&s_gA[dl * C * F + e], v);
                    pA[e] = 0.0f;
                }
            }
        }
        __syncthreads();
    }
    if (DEC) {
        constexpr int NP = ZP ? NW : 1;
        for (int e = threadIdx.x; e < L * C * F; e += kTileThreads) {
            float s = 0.0f;
#pragma unroll
            for (int wq = 0; wq < NP; ++wq) s += s_gA[wq * L * C * F + e];
            if (grad_A && s != 0.0f) red_add(grad_A + e, s);
        }
        for (int e = threadIdx.x; e < L * F; e += kTileThreads) {
            float s = 0.0f;
#pragma unroll
            for (int wq = 0; wq < NP; ++wq) s += s_gS[wq * L * F + e];
            if (grad_shift && s != 0.0f) red_add(grad_shift + e, s);
        }
    }
}

}  // namespace shacira
