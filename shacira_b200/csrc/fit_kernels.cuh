// fit_kernels.cuh -- the image-fit step's grid forward, decoder MLP + MSE and grid backward as ONE tile-resident
// kernel (SURVEY section 8 row f-1 as written: "features never leave the SM").
//
// Reference path this replaces, per training step of app/image:
//   feats = grid.interpolate(coords)          wisp/models/grids/latent_grid.py:340-382
//   rgb   = decoder_color(feats)              wisp/models/nefs/image.py:109-120,152
//   loss  = ((rgb - gt) ** 2).mean()          wisp/trainers/image_trainer.py:298-300
//   loss.backward()                           hashgrid_interpolate2d_cuda.cu:133-232 (scatter-add), autograd MLP
// and, in this repository, the three launches latent_fwd_tiled_kernel -> mlp16_tc_step_kernel -> latent_bwd_tiled_kernel
// that exchange feats[N,16] and grad_feats[N,16] through HBM (2 x 2 x 25 MB per step at the Kodak shape).
//
// One persistent CTA (4 warps) walks the plan's tiles. Per tile: stage the tile's nodes of all levels in shared memory
// (rounded latents, node table from the plan), then in passes of 64 points
//   * every lane interpolates ITS OWN entries of the mma.sync A fragment -- lane (g, t) of a warp owns points
//     g, g+8 of the warp's 16-point tile and the four levels {2t, 2t+1, 8+2t, 8+2t+1} -- so the 16 features of a point
//     are born in the register layout the first layer's tensor-core product consumes (no transposition, no staging);
//   * the warp runs the 16 -> 16 -> 16 -> 3 MLP, the MSE and its backward on the tensor cores (3xTF32, the building
//     blocks of mlp_tc_common.cuh), weight gradients accumulate in registers across the whole kernel;
//   * the feature gradient comes out in the same fragment layout: the lane scatters its 2 points x 4 levels into the
//     tile's fixed-point node accumulators (shared-memory integer atomics, lane-replicated on coarse levels) with the
//     cell / weights it kept from the forward.
// The fixed-point scale of a level needs max |gradient| over the tile, which is only known when the tile's last pass
// has run the MLP: the scale follows a RUNNING maximum (`headroom` bits of slack) and, when a later pass outgrows it, the
// accumulators of that level are shifted right once (exact up to one rounding per shift). After the last pass every
// touched node is flushed with one float RED, decoder gradients (scale / shift of the affine latent decoder) are
// applied per node there, as in latent_bwd_tiled_kernel's scatter-g mode.
//
// Shapes: 2D, latent_dim = feature_dim = 1, one affine decoder, 16 levels that all fit the tile's node box, rows in the
// plan's sorted order (shacira_plan_set_sorted_io). Everything else keeps the three-kernel path.
//
// fit_render_kernel (end of file): the same tile walk, staging and lerp, forward only -- a model of this shape into pixels
// and the integer SSE of its clamped PSNR (shacira_fit_render).
#pragma once
#include "mlp_tc_common.cuh"
#include "tiled_kernels.cuh"

namespace shacira {

constexpr int kFitWarps = 4;
static_assert(kFitWarps * 32 == kTileThreads, "the staging helpers stride by kTileThreads");
constexpr int kFitPts = 16 * kFitWarps;                                   // points per pass
constexpr int kFitParams = 16 * 16 + 16 + 16 * 16 + 16 + 3 * 16 + 3;      // W1 | b1 | W2 | b2 | W3 | b3 (packed order)
constexpr int kExpUnset = 127, kExpNan = -128;
#ifndef SHACIRA_FIT_MIN_CTAS
#define SHACIRA_FIT_MIN_CTAS 4
#endif

struct FitSmem {
    uint4 wf[20][32];                          // weight fragments (tc_build_fragments)
    float rows[kFitWarps][3][16][kTcStride];   // per warp: three rotating staging buffers for the weight gradients
    float dy[kFitWarps][16][8];
    double resd[16];                           // level constants (lane-dependent level index: shared, not c[bank])
    float hi[16];
    float b1[16], b2[16], b3[4];
    float g[kFitParams + 1];                   // block reduction of the MLP gradients
    unsigned pmax[2][16];                      // running max |feature gradient| per level of this tile (bit patterns)
    float inv[16];                             // 2^-exponent of the level's fixed-point scale (flush)
    double loss;
    float gA, gS;
};

// one point, one level: cell, weights' fractions and the first corner's slot (offp + x + y * w0)
__device__ __forceinline__ void fit_locate(double t0, double t1, double resd, float hi, int offp, int w0, int& slot,
                                           float& f0, float& f1) {
    float x = __double2float_rn(__dmul_rn(resd, t0)), y = __double2float_rn(__dmul_rn(resd, t1));
    x = fmaxf(0.0f, fminf(hi, x));
    y = fmaxf(0.0f, fminf(hi, y));
    int cx, cy;
    float fx, fy;
    floor_cell(x, cx, fx);
    floor_cell(y, cy, fy);
    f0 = __fsub_rn(x, fx);
    f1 = __fsub_rn(y, fy);
    slot = offp + cx + cy * w0;
}

// This lane's entries of the first layer's A fragment: its 2 points x 4 levels lerped from the tile's staged nodes, with
// the cell / weights of each kept for a backward scatter. Lane (g, t) owns points g, g+8 of its warp's 16 and the levels
// lev[j] = 8 (j >> 1) + 2 t + (j & 1), i.e. fragment entry [j >> 1][2 hh + (j & 1)].
__device__ __forceinline__ void fit_lerp(const double* resd_s, const float* hi_s, const TileGeom<2>& tg,
                                         const int (&lev)[4], const double (&tu)[2][2], const float* s_nodes,
                                         float Aval, float Sval, float (&X)[1][2][4], int (&slot)[2][4],
                                         float (&f0)[2][4], float (&f1)[2][4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int l = lev[j];
        const double resd = resd_s[l];
        const float hi = hi_s[l];
        const int offp = tg.offp[l], w0 = tg.w[l][0];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            fit_locate(tu[hh][0], tu[hh][1], resd, hi, offp, w0, slot[hh][j], f0[hh][j], f1[hh][j]);
            const float g0 = __fsub_rn(1.0f, f0[hh][j]), g1 = __fsub_rn(1.0f, f1[hh][j]);
            const int sb = slot[hh][j];
            const float v0 = s_nodes[sb], v1 = s_nodes[sb + w0], v2 = s_nodes[sb + 1], v3 = s_nodes[sb + w0 + 1];
            // corner order and contraction order of the tiled forward (stencil(), lerp_rows())
            float z = __fmul_rn(v1, __fmul_rn(g0, f1[hh][j]));
            z = __fmaf_rn(v0, __fmul_rn(g0, g1), z);
            z = __fmaf_rn(v2, __fmul_rn(f0[hh][j], g1), z);
            z = __fmaf_rn(v3, __fmul_rn(f0[hh][j], f1[hh][j]), z);
            X[0][j >> 1][2 * hh + (j & 1)] = __fmaf_rn(z, Aval, Sval);
        }
    }
}

__global__ void __launch_bounds__(kTileThreads, SHACIRA_FIT_MIN_CTAS)
fit_tile_kernel(const PlanView pv, const float* __restrict__ latents, const __grid_constant__ LevelParams lp,
                const float* __restrict__ A, const float* __restrict__ shift, int round_flag,
                const float* __restrict__ target, const float* __restrict__ W1, const float* __restrict__ b1,
                const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ W3,
                const float* __restrict__ b3, float grad_scale, float* __restrict__ grad_latents,
                float* __restrict__ grad_A, float* __restrict__ grad_shift, double* __restrict__ loss_sum,
                float* __restrict__ grad_params, int cap, int cap_acc, int headroom) {
    constexpr int H = 16, OUT = 3, L = 16;
    constexpr int oW1 = 0, ob1 = oW1 + 256, oW2 = ob1 + H, ob2 = oW2 + 256, oW3 = ob2 + H, ob3 = oW3 + OUT * H;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ TileGeom<2> tg;
    FitSmem& S = *reinterpret_cast<FitSmem*>(s_raw);
    float* s_nodes = reinterpret_cast<float*>(s_raw + sizeof(FitSmem));   // [cap] rounded latents of the tile's nodes
    int* s_acc = reinterpret_cast<int*>(s_nodes + cap);                   // [cap_acc] fixed-point node sums
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;

    tc_build_fragments(S.wf, W1, W2, W3, tid, kTileThreads);
    for (int e = tid; e < kFitParams + 1; e += kTileThreads) S.g[e] = 0.0f;
    if (tid < 16) {
        S.b1[tid] = b1[tid];
        S.b2[tid] = b2[tid];
        S.resd[tid] = lp.resd[tid];
        S.hi[tid] = lp.hi[tid];
    }
    if (tid < 4) S.b3[tid] = tid < OUT ? b3[tid] : 0.0f;
    if (tid == 0) { S.loss = 0.0; S.gA = 0.0f; S.gS = 0.0f; }
    __syncthreads();   // (a CTA whose tiles are all empty goes straight to the final reduction)
    const float Aval = __ldg(A), Sval = shift ? __ldg(shift) : 0.0f;
    // this lane's levels: j -> 8 (j >> 1) + 2 t + (j & 1), i.e. fragment entry [ks = j >> 1][2 hh + (j & 1)]
    int lev[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) lev[j] = 8 * (j >> 1) + 2 * t + (j & 1);

    float accW1[2][4], accW2[2][4], accW3[1][4], accb1[2][2], accb2[2][2], accb3[2] = {0.0f, 0.0f};
#pragma unroll
    for (int a = 0; a < 2; ++a) {
#pragma unroll
        for (int b = 0; b < 4; ++b) { accW1[a][b] = 0.0f; accW2[a][b] = 0.0f; }
        accb1[a][0] = accb1[a][1] = accb2[a][0] = accb2[a][1] = 0.0f;
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) accW3[0][b] = 0.0f;
    float my_loss = 0.0f, pS = 0.0f, pA = 0.0f;
    float (*bufA)[kTcStride] = S.rows[warp][0];
    float (*bufB)[kTcStride] = S.rows[warp][1];
    float (*bufC)[kTcStride] = S.rows[warp][2];
    float (*sdy)[8] = S.dy[warp];

    for (int tile = blockIdx.x; tile < pv.ntiles; tile += gridDim.x) {
        const int beg = pv.tile_off[tile], end = pv.tile_off[tile + 1];
        if (beg == end) continue;   // uniform over the CTA
        const int ti[2] = {tile % pv.g, tile / pv.g};
        const int2* tab = pv.node_tab + (size_t)tile * pv.node_stride;
        int pre[kPre];
        prefetch_rows(tab, pv.node_stride, pre);
        __syncthreads();   // the previous tile's flush is done with tg / s_nodes / s_acc (and the setup above is visible)
        tile_geometry<2>(tg, lp, ti, pv.g, cap, cap_acc, cap_acc - cap);
        stage_nodes_prefetched<2, 1>(tg, tab, pre, latents, round_flag, s_nodes);
        {
            const int n4 = (tg.acc_total + 3) >> 2;
            int4* z4 = reinterpret_cast<int4*>(s_acc);
            for (int e = tid; e < n4; e += kTileThreads) z4[e] = make_int4(0, 0, 0, 0);
        }
        if (tid < 32) S.pmax[tid >> 4][tid & 15] = 0u;
        int my_exp = kExpUnset, pb = 0;   // lane l < 16 (of every warp): exponent of level l's fixed-point scale
        int kbits = 0;
        while ((1 << kbits) < (end - beg)) ++kbits;
        __syncthreads();

        // this lane's two points of a pass: coordinates and targets are requested one pass ahead (software pipeline)
        float2 cN[2];
        float TN[4];
        auto request = [&](int p0) {
            const int base = p0 + warp * 16;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                // rows past the tile's end take the tile's last point: every slot they form is valid, their loss gradient is
                // zero (row < end below), so they add zeros -- no liveness branches in the lerp and the scatter
                const int j = min(base + g + 8 * hh, end - 1);
                cN[hh] = __ldg(reinterpret_cast<const float2*>(pv.coords_sorted) + j);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int col = 2 * t + (r & 1);
                const int row = base + g + 8 * (r >> 1);
                TN[r] = (col < OUT && row < end) ? __ldg(target + (int64_t)row * OUT + col) : 0.0f;
            }
        };
        request(beg);
        for (int p0 = beg; p0 < end; p0 += kFitPts) {
            const int base = p0 + warp * 16;
            double tu[2][2];
            float T[4];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                tu[hh][0] = unit_coord(cN[hh].x);
                tu[hh][1] = unit_coord(cN[hh].y);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) T[r] = TN[r];
            // ---- grid forward: the A fragment of the first layer, entry by entry -------------------------------------
            float X[1][2][4];
            int slot[2][4];
            float f0[2][4], f1[2][4];
            fit_lerp(S.resd, S.hi, tg, lev, tu, s_nodes, Aval, Sval, X, slot, f0, f1);
            // ---- MLP forward ------------------------------------------------------------------------------------------
            __syncwarp();   // the previous pass's weight-gradient reads of bufA are done
            tc_stage<1>(bufA, g, t, X);
            float h1[1][2][4], h2[1][2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b1[8 * nt + 2 * t]);
                h1[0][nt][0] = h1[0][nt][2] = bb.x;
                h1[0][nt][1] = h1[0][nt][3] = bb.y;
            }
            tc_layer<2, 2, 1>(S.wf, F_L1, lane, X, h1);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b2[8 * nt + 2 * t]);
#pragma unroll
                for (int r = 0; r < 4; ++r) h1[0][nt][r] = fmaxf(h1[0][nt][r], 0.0f);
                h2[0][nt][0] = h2[0][nt][2] = bb.x;
                h2[0][nt][1] = h2[0][nt][3] = bb.y;
            }
            tc_stage<1>(bufB, g, t, h1);
            tc_layer<2, 2, 1>(S.wf, F_L2, lane, h1, h2);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) h2[0][nt][r] = fmaxf(h2[0][nt][r], 0.0f);
            tc_stage<1>(bufC, g, t, h2);
            float Y[4];
            {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b3[(2 * t) & 3]);
                Y[0] = Y[2] = (t < 2) ? bb.x : 0.0f;
                Y[1] = Y[3] = (t < 2) ? bb.y : 0.0f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint4 f = S.wf[F_L3 + ks][lane];
                    uint32_t ahi[4], alo[4];
                    tile_to_a(h2[0][ks], ahi, alo);
                    mma3(Y, ahi, alo, f.x, f.y, f.z, f.w);
                }
            }
            // ---- loss and its gradient (columns 2t, 2t+1 < 3 are real) -------------------------------------------------
            float DY[1][2][4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int col = 2 * t + (r & 1);
                const int row = base + g + 8 * (r >> 1);
                float d = 0.0f;
                if (col < OUT && row < end) {
                    const float e = Y[r] - T[r];
                    my_loss = fmaf(e, e, my_loss);
                    d = e * grad_scale;
                }
                DY[0][0][r] = d;
                DY[0][1][r] = 0.0f;
            }
            *reinterpret_cast<float2*>(&sdy[g][2 * t]) = make_float2(DY[0][0][0], DY[0][0][1]);
            *reinterpret_cast<float2*>(&sdy[g + 8][2 * t]) = make_float2(DY[0][0][2], DY[0][0][3]);
            accb3[0] += DY[0][0][0] + DY[0][0][2];
            accb3[1] += DY[0][0][1] + DY[0][0][3];
            __syncwarp();
            tc_wgrad<1, 8, 1>(bufC, sdy, g, t, accW3);           // dW3^T[j][k] = sum_p h2[p][j] dy[p][k]
            // ---- backward to the features ----------------------------------------------------------------------------------
            float D[1][2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) D[0][nt][r] = 0.0f;
            tc_layer<1, 2, 1>(S.wf, B_D2, lane, DY, D);           // d2 = dy W3
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int r = 0; r < 4; ++r) D[0][nt][r] = h2[0][nt][r] > 0.0f ? D[0][nt][r] : 0.0f;
                accb2[nt][0] += D[0][nt][0] + D[0][nt][2];
                accb2[nt][1] += D[0][nt][1] + D[0][nt][3];
            }
            __syncwarp();   // bufC (h2) has been read by every lane
            tc_stage<1>(bufC, g, t, D);                           // bufC := d2
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) h2[0][nt][r] = 0.0f;  // h2 is dead: reuse as d1
            tc_layer<2, 2, 1>(S.wf, B_D1, lane, D, h2);           // d1 = d2 W2
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    h2[0][nt][r] = h1[0][nt][r] > 0.0f ? h2[0][nt][r] : 0.0f;
                    D[0][nt][r] = 0.0f;
                }
                accb1[nt][0] += h2[0][nt][0] + h2[0][nt][2];
                accb1[nt][1] += h2[0][nt][1] + h2[0][nt][3];
            }
            __syncwarp();
            tc_wgrad<2, kTcStride, 1>(bufC, bufB, g, t, accW2);   // dW2[j][i] = sum_p d2[p][j] h1[p][i]
            __syncwarp();   // bufB (h1) has been read
            tc_stage<1>(bufB, g, t, h2);                          // bufB := d1
            tc_layer<2, 2, 1>(S.wf, B_GX, lane, h2, D);           // gx = d1 W1: D[0][nt][2 hh + e] <-> level 8 nt + 2 t + e
            __syncwarp();
            tc_wgrad<2, kTcStride, 1>(bufB, bufA, g, t, accW1);   // dW1[i][m] = sum_p d1[p][i] x[p][m]
            // the next pass's coordinates and targets: requested here, where the MLP's registers are dead, and in flight
            // behind the maxima, the barrier and the scatter (requested at the top of the pass they cost 8 registers
            // across the whole MLP: spills, measured slower)
            if (p0 + kFitPts < end) request(p0 + kFitPts);

            // ---- running per-level maximum of |gx| over the tile (this warp's 16 points) -----------------------------------
            // Two copies of the maxima, used by alternating passes: a warp that is already in the next pass adds to the
            // other copy, so after this pass's barrier every warp reads the SAME values and takes the same decision
            // without a second barrier (lane l < 16 of every warp tracks level l's exponent in a register).
            unsigned* pm = S.pmax[pb];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float m = nan_max(fabsf(D[0][j >> 1][j & 1]), fabsf(D[0][j >> 1][2 + (j & 1)]));
                unsigned mb = __float_as_uint(m);
                mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 4));
                mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 8));
                mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, 16));
                if (g == 0 && mb > pm[lev[j]]) atomicMax(&pm[lev[j]], mb);
            }
            __syncthreads();
            int sh = 0;
            {
                const unsigned mb = pm[lane & 15];
                const float m = __uint_as_float(mb);
                if (warp == 0 && lane < L && mb != 0u) atomicMax(&S.pmax[pb ^ 1][lane], mb);   // the running maximum carries over
                const int old = my_exp;
                if (m != m || mb >= 0x7f800000u) {
                    my_exp = kExpNan;   // Inf / NaN upstream: the level's nodes of this tile are poisoned at flush time
                } else if (mb != 0u && old != kExpNan) {
                    const int ex = (int)((mb >> 23) & 0xffu) - 126;   // m < 2^ex
                    const int need = max(-126, min(min(30 - kbits, 21) - ex, 126));
                    if (old == kExpUnset) {
                        my_exp = max(-126, need - headroom);   // accumulators still zero: nothing to shift
                    } else if (need < old) {
                        my_exp = max(-126, need - headroom);
                        sh = old - my_exp;
                    }
                }
            }
            pb ^= 1;
            if (__any_sync(0xffffffffu, sh > 0)) {   // uniform over the CTA: every warp evaluated the same numbers
                // a level outgrew its scale: shift its accumulators (round to nearest), then go on at the new scale
                for (int l = 0; l < L; ++l) {
                    const int shl = __shfl_sync(0xffffffffu, sh, l);
                    if (shl <= 0) continue;
                    const int a0 = tg.acc_off[l], a1 = (l + 1 < L) ? tg.acc_off[l + 1] : tg.acc_total;
                    for (int e = a0 + tid; e < a1; e += kTileThreads) {
                        const int v = s_acc[e];
                        s_acc[e] = shl >= 31 ? 0 : ((v + (1 << (shl - 1))) >> shl);
                    }
                }
                __syncthreads();
            }
            // ---- scatter: this lane's 2 points x 4 levels into the tile's node accumulators ---------------------------------
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int l = lev[j];
                const int ej = __shfl_sync(0xffffffffu, my_exp, l);
                const float sc = (ej == kExpNan || ej == kExpUnset) ? 0.0f : __int_as_float((127 + ej) << 23);
                const int amul = tg.acc_mul[l], w0 = tg.w[l][0];
                const int abase = tg.acc_off[l] + (amul == 32 ? lane : 0) - tg.off[l] * amul;
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const float gs = __fmul_rn(D[0][j >> 1][2 * hh + (j & 1)], sc);   // power-of-two scale: exact
                    const float a0 = f0[hh][j], a1 = f1[hh][j];
                    const float g0 = __fsub_rn(1.0f, a0), g1 = __fsub_rn(1.0f, a1);
                    const int sb = slot[hh][j];
                    atomicAdd(&s_acc[sb * amul + abase], fixed_rn(__fmul_rn(gs, __fmul_rn(g0, g1))));
                    atomicAdd(&s_acc[(sb + w0) * amul + abase], fixed_rn(__fmul_rn(gs, __fmul_rn(g0, a1))));
                    atomicAdd(&s_acc[(sb + 1) * amul + abase], fixed_rn(__fmul_rn(gs, __fmul_rn(a0, g1))));
                    atomicAdd(&s_acc[(sb + w0 + 1) * amul + abase], fixed_rn(__fmul_rn(gs, __fmul_rn(a0, a1))));
                }
            }
        }   // passes of this tile

        // ---- flush: one float RED per touched node; decoder gradients per node ---------------------------------------------
        constexpr int kFlushPre = 8;
        int2 fpre[kFlushPre];
#pragma unroll
        for (int u = 0; u < kFlushPre; ++u) {
            const int e = tid + u * kTileThreads;
            fpre[u] = (e < tg.total) ? __ldg(tab + e) : make_int2(0, 0);
        }
        if (tid < L) {
            const int e = my_exp;
            S.inv[tid] = (e == kExpNan) ? __int_as_float(0x7fc00000) : ((e == kExpUnset) ? 0.0f : __int_as_float((127 - e) << 23));
        }
        __syncthreads();
        auto flush_node = [&](int e, int2 ent) {
            const int l = ent.y & 0xff;
            const int nloc = e - tg.off[l];
            const float inv = S.inv[l];
            int qv = 0;
            if (tg.acc_mul[l] == 32) {
                const int* a = s_acc + tg.acc_off[l] + nloc * 32;
#pragma unroll 8
                for (int jj = 0; jj < 32; ++jj) qv += a[(lane + jj) & 31];
            } else {
                qv = s_acc[tg.acc_off[l] + nloc];
            }
            float gv = (float)qv * inv;
            bool any = qv != 0;
            if (inv != inv) { any = true; gv = inv; }
            if (!any || (ent.y & kNodeInvalid)) return;
            red_add(grad_latents + ent.x, gv * Aval);
            pA = __fmaf_rn(s_nodes[e], gv, pA);
            pS += gv;
        };
        {
            int e = tid;
#pragma unroll
            for (int u = 0; u < kFlushPre; ++u, e += kTileThreads)
                if (e < tg.total) flush_node(e, fpre[u]);
            for (; e < tg.total; e += kTileThreads) flush_node(e, __ldg(tab + e));
        }
    }   // tiles

    // ---- block reduction in shared memory, then one global add per CTA and value ------------------------------------------
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
    const float wl = warp_sum(my_loss), wA = warp_sum(pA), wS = warp_sum(pS);
    if (lane == 0) {
        atomicAdd(&S.loss, (double)wl);
        atomicAdd(&S.gA, wA);
        atomicAdd(&S.gS, wS);
    }
    __syncthreads();
    for (int e = tid; e < kFitParams; e += kTileThreads) red_add(grad_params + e, S.g[e]);
    if (tid == 0) {
        atomicAdd(loss_sum, S.loss);
        // one shared decoder: only the SUM over the L rows is defined (the caller adds them): spread the CTAs over the rows
        const int dl = blockIdx.x % L;
        if (grad_A && S.gA != 0.0f) red_add(grad_A + dl, S.gA);
        if (grad_shift && S.gS != 0.0f) red_add(grad_shift + dl, S.gS);
    }
}

// ---- forward only: grid -> MLP -> RGB (and the uint8 SSE against a target) ------------------------------------------------
// fit_tile_kernel's tile walk, staging and lerp (fit_lerp) with rounding on -- the stored model is integers -- followed by
// the 16 -> 16 -> 16 -> 3 forward on the tensor cores; nothing is staged for a backward. Rows follow the plan's convention
// (original index, or tile order on a sorted-I/O plan). With `target`, every real output adds
// (q(rgb) - q(target))^2 with q(v) = (uint8)(clamp(v, 0, 1) * 255) (torch's .to(torch.uint8) truncates): an integer sum,
// exact in any order.
struct RenderSmem {
    uint4 wf[20][32];
    double resd[16];
    float hi[16];
    float b1[16], b2[16], b3[4];
};

__device__ __forceinline__ int quantize_u8(float v) { return (int)__fmul_rn(fminf(fmaxf(v, 0.0f), 1.0f), 255.0f); }

__global__ void __launch_bounds__(kTileThreads, SHACIRA_FIT_MIN_CTAS)
fit_render_kernel(const PlanView pv, const float* __restrict__ latents, const __grid_constant__ LevelParams lp,
                  const float* __restrict__ A, const float* __restrict__ shift, const float* __restrict__ W1,
                  const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                  const float* __restrict__ W3, const float* __restrict__ b3, float* __restrict__ rgb,
                  const float* __restrict__ target, unsigned long long* __restrict__ sse_u8, int cap) {
    constexpr int OUT = 3;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ TileGeom<2> tg;
    RenderSmem& S = *reinterpret_cast<RenderSmem*>(s_raw);
    float* s_nodes = reinterpret_cast<float*>(s_raw + sizeof(RenderSmem));   // [cap] rounded latents of the tile's nodes
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;

    tc_build_fragments(S.wf, W1, W2, W3, tid, kTileThreads);
    if (tid < 16) {
        S.b1[tid] = b1[tid];
        S.b2[tid] = b2[tid];
        S.resd[tid] = lp.resd[tid];
        S.hi[tid] = lp.hi[tid];
    }
    if (tid < 4) S.b3[tid] = tid < OUT ? b3[tid] : 0.0f;
    __syncthreads();
    const float Aval = __ldg(A), Sval = shift ? __ldg(shift) : 0.0f;
    int lev[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) lev[j] = 8 * (j >> 1) + 2 * t + (j & 1);
    unsigned long long my_sse = 0ull;

    for (int tile = blockIdx.x; tile < pv.ntiles; tile += gridDim.x) {
        const int beg = pv.tile_off[tile], end = pv.tile_off[tile + 1];
        if (beg == end) continue;   // uniform over the CTA
        const int ti[2] = {tile % pv.g, tile / pv.g};
        const int2* tab = pv.node_tab + (size_t)tile * pv.node_stride;
        int pre[kPre];
        prefetch_rows(tab, pv.node_stride, pre);
        __syncthreads();   // the previous tile's passes are done with tg / s_nodes
        tile_geometry<2>(tg, lp, ti, pv.g, cap);
        stage_nodes_prefetched<2, 1>(tg, tab, pre, latents, 1, s_nodes);
        __syncthreads();
        for (int p0 = beg; p0 < end; p0 += kFitPts) {
            const int base = p0 + warp * 16;
            double tu[2][2];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                // rows past the tile's end take the tile's last point (valid slots); their outputs are dropped below
                const float2 c = __ldg(reinterpret_cast<const float2*>(pv.coords_sorted) + min(base + g + 8 * hh, end - 1));
                tu[hh][0] = unit_coord(c.x);
                tu[hh][1] = unit_coord(c.y);
            }
            float X[1][2][4];
            int slot[2][4];
            float f0[2][4], f1[2][4];
            fit_lerp(S.resd, S.hi, tg, lev, tu, s_nodes, Aval, Sval, X, slot, f0, f1);
            float h1[1][2][4], h2[1][2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b1[8 * nt + 2 * t]);
                h1[0][nt][0] = h1[0][nt][2] = bb.x;
                h1[0][nt][1] = h1[0][nt][3] = bb.y;
            }
            tc_layer<2, 2, 1>(S.wf, F_L1, lane, X, h1);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b2[8 * nt + 2 * t]);
#pragma unroll
                for (int r = 0; r < 4; ++r) h1[0][nt][r] = fmaxf(h1[0][nt][r], 0.0f);
                h2[0][nt][0] = h2[0][nt][2] = bb.x;
                h2[0][nt][1] = h2[0][nt][3] = bb.y;
            }
            tc_layer<2, 2, 1>(S.wf, F_L2, lane, h1, h2);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int r = 0; r < 4; ++r) h2[0][nt][r] = fmaxf(h2[0][nt][r], 0.0f);
            float Y[4];
            {
                const float2 bb = *reinterpret_cast<const float2*>(&S.b3[(2 * t) & 3]);
                Y[0] = Y[2] = (t < 2) ? bb.x : 0.0f;
                Y[1] = Y[3] = (t < 2) ? bb.y : 0.0f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint4 f = S.wf[F_L3 + ks][lane];
                    uint32_t ahi[4], alo[4];
                    tile_to_a(h2[0][ks], ahi, alo);
                    mma3(Y, ahi, alo, f.x, f.y, f.z, f.w);
                }
            }
            // Y[r]: point base + g + 8 (r >> 1), column 2 t + (r & 1); columns < 3 are real
            if (t < 2) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int col = 2 * t + (r & 1);
                    const int row = base + g + 8 * (r >> 1);
                    if (col < OUT && row < end) {
                        const int64_t o = (int64_t)(pv.perm ? __ldg(pv.perm + row) : row) * OUT + col;
                        if (rgb) rgb[o] = Y[r];
                        if (target) {
                            const int d = quantize_u8(Y[r]) - quantize_u8(__ldg(target + o));
                            my_sse += (unsigned long long)(d * d);
                        }
                    }
                }
            }
        }
    }
    if (target) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_sse += __shfl_xor_sync(0xffffffffu, my_sse, o);
        if (lane == 0 && my_sse) atomicAdd(sse_u8, my_sse);
    }
}

}  // namespace shacira
