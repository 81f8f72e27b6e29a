// grid3d_kernels.cuh -- 3D latent-grid kernels built around the REQUEST economy of the B200 memory system.
//
// Reference: hashgrid_interpolate_cuda.cu:47-109 (forward) and :143-271 (backward): one thread per point and level,
// 8 scalar corner gathers / 8 scalar atomicAdds. On the fine levels of a NeRF-shape grid every sample sits in a cell of
// its own, so nothing is shared between samples (profiles/r01b_ncu_3d_fwd_summary.txt: one sector per 4-byte gather,
// 31.4 sectors per request).
//
// Lane pairs: TWO lanes per sample, lane parity = the x side of the cell (dx).
// Measured on the B200 (benchmarks/microbench2.cu, profiles/r02a_microbench2.csv; ncu of an earlier one-lane-per-sample
// form with merged 16-byte x-pair loads, profiles/r02a_ncu_3d_*.txt): what bounds the 3D path is the number of
// REQUESTS an SM sends to L2 -- ~1 per clock per SM ("L1: M L1tex2xbar Req Cycles Active" 83 %), one per (instruction,
// 128-byte line) for loads and stores and one per (instruction, 32-byte sector) for reds -- not bytes, sectors or
// instructions. Two lanes of ONE instruction that touch the same line (loads) / sector (reds) share a request:
// 294 G pairs/s for loads and 198 G pairs/s for reds, the rates of single accesses. So lanes 2s and 2s+1 work on sample
// s of the warp's 16 samples: both locate the cell, lane parity picks x or x+1, and every load / red instruction carries
// the two x-neighbour corners of 16 samples side by side: 4 requests per sample and level instead of 8, on any
// alignment of the level in the table. Indices, weights and rounding are those of common.cuh, and the interpolation sum
// keeps the reference's order: the even lane runs corners 0..3, hands its partial sum to the odd lane (one shuffle),
// which continues with corners 4..7 -- bit-identical to latent_fwd_kernel.
// Rows (features, upstream gradients, saved z) move through per-warp shared-memory tiles so that every global access
// is a full 128-byte line: 2 requests per 256-byte row instead of 16.
//
// Samples may be given in the plan's tile-sorted order (`perm` != NULL: coords are the plan's sorted copy, row i of the
// result belongs to sample perm[i]): neighbouring lanes then share the coarse and middle levels' cache lines in L1.
#pragma once
#include "common.cuh"

namespace shacira {

constexpr int kLpWarps = 8;                  // warps per CTA
constexpr int kLpBlock = kLpWarps * 32;
constexpr int kLpSamples = 16;               // samples per warp pass
constexpr int kLpChunk = kLpWarps * kLpSamples;  // samples per CTA pass
#ifndef SHACIRA_LP_LV
#define SHACIRA_LP_LV 2
#endif
#ifndef SHACIRA_LP_MINB
#define SHACIRA_LP_MINB 5
#endif
constexpr int kLpLv = SHACIRA_LP_LV;         // levels in flight per lane (4 loads each)
constexpr int kLpFlush = 8;                  // levels per output flush of the forward

// this lane's side of the cell at level l: 4 corner rows (absolute) j = dy*2 + dz and their weights
struct Side3 {
    int32_t idx[4];
    float w[4];
};
__device__ __forceinline__ void locate_d(double t, double resd, float hi, int32_t& cell, float& f, float& g) {
    float x = __double2float_rn(__dmul_rn(resd, t));
    x = fmaxf(0.0f, fminf(hi, x));
    float cf;
    floor_cell(x, cell, cf);
    f = __fsub_rn(x, cf);
    g = __fsub_rn(1.0f, f);
}
__device__ __forceinline__ void side3(const double (&t)[3], const LevelParams& lp, int l, int dx, Side3& o) {
    const double resd = lp.resd[l];
    const float hi = lp.hi[l];
    const int32_t first = lp.first[l];
    int32_t p[3];
    float f[3], g[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) locate_d(t[d], resd, hi, p[d], f[d], g[d]);
    const float X = dx ? f[0] : g[0];
    const float xy0 = __fmul_rn(X, g[1]), xy1 = __fmul_rn(X, f[1]);   // reference: (wx * wy) * wz, left to right
    o.w[0] = __fmul_rn(xy0, g[2]);
    o.w[1] = __fmul_rn(xy0, f[2]);
    o.w[2] = __fmul_rn(xy1, g[2]);
    o.w[3] = __fmul_rn(xy1, f[2]);
    if ((lp.dense_mask >> l) & 1u) {
        const int32_t res = lp.res[l];
        const int32_t last = first + lp.rows[l] - 1;   // SURVEY Q4: zero-weight corners stay inside the level
        const int32_t rr = res * res;
        const int32_t base = first + p[0] + dx + p[1] * res + p[2] * rr;
        o.idx[0] = min(base, last);
        o.idx[1] = min(base + rr, last);
        o.idx[2] = min(base + res, last);
        o.idx[3] = min(base + res + rr, last);
    } else {
        const uint32_t m = lp.hash_mask;
        const uint32_t hx = (uint32_t)(p[0] + dx);
        const uint32_t hy0 = (uint32_t)p[1] * kPrimeY, hz0 = (uint32_t)p[2] * kPrimeZ;
        const uint32_t a0 = hx ^ hy0, a1 = hx ^ (hy0 + kPrimeY);
        const uint32_t hz1 = hz0 + kPrimeZ;
        o.idx[0] = first + (int32_t)((a0 ^ hz0) & m);
        o.idx[1] = first + (int32_t)((a0 ^ hz1) & m);
        o.idx[2] = first + (int32_t)((a1 ^ hz0) & m);
        o.idx[3] = first + (int32_t)((a1 ^ hz1) & m);
    }
}

// Shared memory of one CTA: decoder A / shift | per warp { row index of its 16 samples | staging tiles }.
// Tile rows are padded by 4 floats so that the 16 samples' rows start in different banks.
__host__ __device__ inline int lp_dec_floats(int nA, int C, int F) { return (nA * (C * F + F) + 3) & ~3; }
template <int C, int F>
struct LpFwdLayout {
    static constexpr int WF = kLpFlush * F + 4;   // feature tile row stride (floats)
    static constexpr int WZ = kLpFlush * C + 4;   // z tile row stride
    static constexpr int kWarpFloats = 2 * kLpSamples /* int64 rows */ + kLpSamples * (WF + WZ);
    static size_t bytes(int nA) { return sizeof(float) * (size_t)(lp_dec_floats(nA, C, F) + kLpWarps * kWarpFloats); }
};

template <int N>
__device__ __forceinline__ void sts_row(float* p, const float (&v)[N]) {
    if constexpr (N == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else if constexpr (N == 8) {
        reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
        reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
    } else if constexpr (N == 2) {
        *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    } else {
#pragma unroll
        for (int e = 0; e < N; ++e) p[e] = v[e];
    }
}

// NQ levels l .. l+NQ-1 of one lane: sides, the 4*NQ gathers in flight together, interpolation, decode into the tile
template <int C, int F, int NQ>
__device__ __forceinline__ void lp_fwd_levels(const double (&t)[3], const LevelParams& lp, int l, int dx, int per_level,
                                              int round_flag, const float* __restrict__ latents, const float* s_A,
                                              const float* s_shift, float* ft, float* zt) {
    Side3 sd[NQ];
    float v[NQ][4][C];
#pragma unroll
    for (int q = 0; q < NQ; ++q) side3(t, lp, l + q, dx, sd[q]);
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) load_row<C>(latents + (int64_t)sd[q].idx[j] * C, v[q][j]);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const int la = per_level ? (l + q) : 0;
        float z[C];
#pragma unroll
        for (int ch = 0; ch < C; ++ch) {
            float r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) r[j] = round_flag ? rintf(v[q][j][ch]) : v[q][j][ch];
            // reference order: fma(v0,w0, v1*w1), then corners 2..7; the even lane (x) runs 0..3 and hands over
            float acc = __fmul_rn(r[1], sd[q].w[1]);
            acc = __fmaf_rn(r[0], sd[q].w[0], acc);
            acc = __fmaf_rn(r[2], sd[q].w[2], acc);
            acc = __fmaf_rn(r[3], sd[q].w[3], acc);
            float cont = __shfl_xor_sync(0xffffffffu, acc, 1);   // odd lane: the even lane's partial sum
#pragma unroll
            for (int j = 0; j < 4; ++j) cont = __fmaf_rn(r[j], sd[q].w[j], cont);
            z[ch] = cont;   // meaningful on odd lanes
        }
        if (dx) {
            float o[F];
            if (C == F && s_A == nullptr) {   // plain table (wisp._C.ops entry points): features = interpolated rows
#pragma unroll
                for (int jf = 0; jf < F; ++jf) o[jf] = z[jf < C ? jf : 0];
            } else {
                const float* Ap = s_A + la * C * F;
#pragma unroll
                for (int jf = 0; jf < F; ++jf) {
                    float acc = s_shift[la * F + jf];
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) acc = __fmaf_rn(z[ch], Ap[ch * F + jf], acc);
                    o[jf] = acc;
                }
            }
            sts_row<F>(ft + q * F, o);
            sts_row<C>(zt + q * C, z);
        }
    }
}

template <int C, int F>
__global__ void __launch_bounds__(kLpBlock, SHACIRA_LP_MINB)
latent_fwd3d_lp_kernel(const float* __restrict__ coords, const int32_t* __restrict__ perm, int64_t n,
                       const float* __restrict__ latents, const __grid_constant__ LevelParams lp,
                       const float* __restrict__ A, const float* __restrict__ shift, int per_level, int round_flag,
                       float* __restrict__ feats, float* __restrict__ zsave) {
    extern __shared__ __align__(16) float s_dyn[];
    using LY = LpFwdLayout<C, F>;
    constexpr int WF = LY::WF, WZ = LY::WZ;
    const int L = lp.num_lods;
    const int nA = per_level ? L : 1;
    float* s_A = s_dyn;                       // [nA][C][F]
    float* s_shift = s_A + nA * C * F;        // [nA][F]
    const float* dec_A = A ? s_A : nullptr;   // A == NULL (C == F only): identity decoder, the plain hash grid
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_warp = s_dyn + lp_dec_floats(nA, C, F) + warp * LY::kWarpFloats;
    long long* s_row = reinterpret_cast<long long*>(s_warp);   // [16] output row of each sample
    float* s_tile = s_warp + 2 * kLpSamples;                     // [16][WF]
    float* s_ztile = s_tile + kLpSamples * WF;                   // [16][WZ]
    if (A)
        for (int e = threadIdx.x; e < nA * C * F; e += kLpBlock) s_A[e] = A[e];
    for (int e = threadIdx.x; e < nA * F; e += kLpBlock) s_shift[e] = shift ? shift[e] : 0.0f;
    __syncthreads();
    const int dx = lane & 1, sp = lane >> 1;
    const int64_t base = (int64_t)blockIdx.x * kLpChunk + warp * kLpSamples;   // first sample of this warp
    if (base >= n) return;
    const int nlive = (int)min((int64_t)kLpSamples, n - base);
    // lanes past the end recompute the last sample (never flushed): no predicates in the level loop
    const int64_t i = min(base + sp, n - 1);
    double t[3];
    load_unit_coords<3>(coords, i, t);
    if (dx) s_row[sp] = perm ? (long long)__ldg(perm + i) : (long long)i;
    __syncwarp();
    const int LF = L * F, LC = L * C;
    float* my_ft = s_tile + sp * WF;
    float* my_zt = s_ztile + sp * WZ;
    for (int l0 = 0; l0 < L; l0 += kLpFlush) {
        const int lw = min(kLpFlush, L - l0);   // levels in this flush
        int l1 = 0;
        for (; l1 + kLpLv <= lw; l1 += kLpLv)
            lp_fwd_levels<C, F, kLpLv>(t, lp, l0 + l1, dx, per_level, round_flag, latents, dec_A, s_shift, my_ft + l1 * F,
                                       my_zt + l1 * C);
        for (; l1 < lw; ++l1)
            lp_fwd_levels<C, F, 1>(t, lp, l0 + l1, dx, per_level, round_flag, latents, dec_A, s_shift, my_ft + l1 * F,
                                   my_zt + l1 * C);
        __syncwarp();
        // flush `lw` levels of the live samples: consecutive lanes write consecutive 16-byte chunks of a row piece
        {
            const int wf = lw * F;
            if ((wf & 3) == 0 && (LF & 3) == 0) {
                const int per = wf >> 2;
                int s = 0, c4 = lane;
                while (c4 >= per) { c4 -= per; ++s; }
                while (s < nlive) {
                    const float4 val = *reinterpret_cast<const float4*>(s_tile + s * WF + 4 * c4);
                    *reinterpret_cast<float4*>(feats + s_row[s] * LF + l0 * F + 4 * c4) = val;
                    c4 += 32;
                    while (c4 >= per) { c4 -= per; ++s; }
                }
            } else {
                for (int u = lane; u < nlive * wf; u += 32) {
                    const int s = u / wf, e = u - s * wf;
                    feats[s_row[s] * LF + l0 * F + e] = s_tile[s * WF + e];
                }
            }
            if (zsave) {   // rows in the order of `coords`: the warp's 16 rows are contiguous
                const int wz = lw * C;
                float* zb = zsave + base * LC + l0 * C;
                if ((wz & 3) == 0 && (LC & 3) == 0) {
                    const int per = wz >> 2;
                    int s = 0, c4 = lane;
                    while (c4 >= per) { c4 -= per; ++s; }
                    while (s < nlive) {
                        *reinterpret_cast<float4*>(zb + (int64_t)s * LC + 4 * c4) =
                            *reinterpret_cast<const float4*>(s_ztile + s * WZ + 4 * c4);
                        c4 += 32;
                        while (c4 >= per) { c4 -= per; ++s; }
                    }
                } else {
                    for (int u = lane; u < nlive * wz; u += 32) {
                        const int s = u / wz, e = u - s * wz;
                        zb[(int64_t)s * LC + e] = s_ztile[s * WZ + e];
                    }
                }
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------------------------
// backward, lane pairs. Persistent CTAs: each pass a warp stages the upstream-gradient rows (and saved z rows) of its
// 16 samples in shared memory with whole-line loads, then both lanes of a sample scatter their side of the cell --
// the two x-neighbour corners of 16 samples side by side in every `red`. Decoder gradients are COLUMN sums of the
// staged tile (lane = column; no shuffles), kept in registers over the CTA's passes and reduced once per CTA.
// skip_mask: levels whose scatter another kernel does (tile-staged coarse levels); level_mask: levels of this launch.
// ------------------------------------------------------------------------------------------------------------------
template <int C, int F>
struct LpBwdLayout {
    static int wg(int L) { return L * F + 4; }   // gradient tile row stride
    static int wz(int L) { return L * C + 4; }
    static int warp_floats(int L, bool dec) { return kLpSamples * (wg(L) + (dec ? wz(L) : 0)); }
    static size_t bytes(int L, int nA, bool dec) {
        return sizeof(float) * (size_t)(lp_dec_floats(nA, C, F) + lp_dec_floats(L, C, F) + kLpWarps * warp_floats(L, dec));
    }
};

template <int C, int F>
__global__ void __launch_bounds__(kLpBlock, (C * F <= 4) ? 4 : 2)
latent_bwd3d_lp_kernel(const float* __restrict__ coords, const int32_t* __restrict__ perm, int64_t n,
                       const float* __restrict__ grad_out, const float* __restrict__ zsave,
                       const __grid_constant__ LevelParams lp, const float* __restrict__ A, int per_level,
                       uint32_t skip_mask, uint32_t level_mask, float* __restrict__ grad_latents,
                       float* __restrict__ grad_A, float* __restrict__ grad_shift) {
    extern __shared__ __align__(16) float s_dyn[];
    const int L = lp.num_lods;
    const int nA = per_level ? L : 1;
    const bool want_dec = (grad_A != nullptr) || (grad_shift != nullptr);
    const bool have_z = want_dec && zsave != nullptr;
    const int LF = L * F, LC = L * C;
    const int WG = LF + 4, WZ = LC + 4;
    float* s_A = s_dyn;                                   // [nA][C][F]
    float* s_gA = s_dyn + lp_dec_floats(nA, C, F);        // [L][C][F]
    float* s_gS = s_gA + L * C * F;                       // [L][F]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_g = s_gA + lp_dec_floats(L, C, F) + warp * (kLpSamples * (WG + (want_dec ? WZ : 0)));   // [16][WG]
    float* s_z = s_g + kLpSamples * WG;                                                              // [16][WZ]
    if (A)
        for (int e = threadIdx.x; e < nA * C * F; e += kLpBlock) s_A[e] = A[e];
    for (int e = threadIdx.x; e < L * (C * F + F); e += kLpBlock) s_gA[e] = 0.0f;
    __syncthreads();
    const int dx = lane & 1, sp = lane >> 1;
    const uint32_t scatter_mask = level_mask & ~skip_mask;
    const float* my_g = s_g + sp * WG;
    // decoder-gradient columns of this lane: col = lane + 32 k (< L*F), k < F (L <= 32)
    float accS[F], accA[F][C];
#pragma unroll
    for (int k = 0; k < F; ++k) {
        accS[k] = 0.0f;
#pragma unroll
        for (int ch = 0; ch < C; ++ch) accA[k][ch] = 0.0f;
    }
    const int64_t nchunks = (n + kLpChunk - 1) / kLpChunk;
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const int64_t base = chunk * kLpChunk + warp * kLpSamples;
        if (base >= n) continue;   // warp-uniform
        const int nlive = (int)min((int64_t)kLpSamples, n - base);
        const bool live = base + sp < n;
        const int64_t i = min(base + sp, n - 1);
        double t[3];
        load_unit_coords<3>(coords, i, t);
        // stage the gradient rows: lane pair s holds the row index of sample s; whole 16-byte chunks, whole lines
        const long long my_row = perm ? (long long)__ldg(perm + i) : (long long)i;
        __syncwarp();
        if ((LF & 3) == 0) {
            const int per = LF >> 2;
            int s = 0, c4 = lane;
            while (c4 >= per) { c4 -= per; ++s; }
            const int iters = (kLpSamples * per + 31) >> 5;   // warp-uniform trip count (the shuffle needs every lane)
            for (int it = 0; it < iters; ++it) {
                const bool in = s < kLpSamples;
                const long long r = __shfl_sync(0xffffffffu, my_row, in ? 2 * s : 0);
                if (in) {
                    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (s < nlive) val = __ldg(reinterpret_cast<const float4*>(grad_out + r * LF) + c4);
                    *reinterpret_cast<float4*>(s_g + s * WG + 4 * c4) = val;
                }
                c4 += 32;
                while (c4 >= per) { c4 -= per; ++s; }
            }
        } else {
            for (int u0 = 0; u0 < kLpSamples * LF; u0 += 32) {
                const int u = u0 + lane;
                const int s = u / LF, e = u - s * LF;
                const long long r = __shfl_sync(0xffffffffu, my_row, (s < kLpSamples ? s : 0) * 2);
                if (s < kLpSamples) s_g[s * WG + e] = (s < nlive) ? __ldg(grad_out + r * LF + e) : 0.0f;
            }
        }
        if (want_dec) {
            const float* zb = have_z ? zsave + base * LC : nullptr;   // rows in the order of `coords`
            for (int u = lane; u < kLpSamples * LC; u += 32) {
                const int s = u / LC, e = u - s * LC;
                s_z[s * WZ + e] = (zb && s < nlive) ? __ldg(zb + (int64_t)s * LC + e) : 0.0f;
            }
        }
        __syncwarp();
        // scatter
#pragma unroll 2
        for (int l = 0; l < L; ++l) {
            if (!((scatter_mask >> l) & 1u)) continue;
            Side3 sd;
            side3(t, lp, l, dx, sd);
            const float* Ap = s_A + (per_level ? l : 0) * C * F;
            float g[F];
#pragma unroll
            for (int jf = 0; jf < F; ++jf) g[jf] = my_g[l * F + jf];
            float gz[C];
            if (C == F && A == nullptr) {   // plain table: the gradient rows are the row gradients (2d_cuda.cu:203-205)
#pragma unroll
                for (int ch = 0; ch < C; ++ch) gz[ch] = g[ch < F ? ch : 0];
            } else {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) {
                    float acc = 0.0f;
#pragma unroll
                    for (int jf = 0; jf < F; ++jf) acc = __fmaf_rn(g[jf], Ap[ch * F + jf], acc);
                    gz[ch] = acc;
                }
            }
            if (live) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float gv[C];
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) gv[ch] = __fmul_rn(gz[ch], sd.w[j]);
                    red_add_row<C>(grad_latents + (int64_t)sd.idx[j] * C, gv);
                }
            }
        }
        // decoder gradients: column sums over the warp's samples
        if (want_dec) {
#pragma unroll
            for (int k = 0; k < F; ++k) {
                const int col = lane + 32 * k;
                if (col < LF && ((level_mask >> (col / F)) & 1u)) {
                    const int lc = (col / F) * C;
                    float sS = 0.0f, sA[C];
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) sA[ch] = 0.0f;
#pragma unroll 4
                    for (int s = 0; s < kLpSamples; ++s) {
                        const float gv = s_g[s * WG + col];
                        sS += gv;
#pragma unroll
                        for (int ch = 0; ch < C; ++ch) sA[ch] = __fmaf_rn(s_z[s * WZ + lc + ch], gv, sA[ch]);
                    }
                    accS[k] += sS;
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) accA[k][ch] += sA[ch];
                }
            }
        }
        __syncwarp();
    }
    if (want_dec) {
#pragma unroll
        for (int k = 0; k < F; ++k) {
            const int col = lane + 32 * k;
            if (col < LF) {
                const int l = col / F, jf = col - l * F;
                atomicAdd(&s_gS[col], accS[k]);
#pragma unroll
                for (int ch = 0; ch < C; ++ch) atomicAdd(&s_gA[(l * C + ch) * F + jf], accA[k][ch]);
            }
        }
        __syncthreads();
        if (grad_A)
            for (int e = threadIdx.x; e < L * C * F; e += kLpBlock)
                if (s_gA[e] != 0.0f) red_add(grad_A + e, s_gA[e]);
        if (grad_shift)
            for (int e = threadIdx.x; e < L * F; e += kLpBlock)
                if (s_gS[e] != 0.0f) red_add(grad_shift + e, s_gS[e]);
    }
}

}  // namespace shacira
