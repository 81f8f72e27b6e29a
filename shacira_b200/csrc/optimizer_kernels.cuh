// optimizer_kernels.cuh -- the whole optimizer side of the image-fit step as ONE launch (SURVEY section 8 row f-4).
//
// Reference: optimizer.step() over the parameter groups of base_trainer.py:206-266 (image_trainer.py:321-359) and, at the
// start of the next step, the SGA sample of the latents (basic_latent_decoder.py:183-191). Here:
//   CTAs [0, S.num)      Adam over the ~20 small tensors (decoder MLP, latent decoder, density model) with their chain
//                        rules, exactly multi_adam_kernel's per-CTA work;
//   the remaining CTAs   one pass over the latent table: optionally the bit-rate loss of the latents before their update
//                        (latent_grid.py:122-136: entropy_kernel's math and noise stream, latent_dim 1), Adam (gradient =
//                        grid gradient x d w_hat / d w + (lambda / rows) x bit-rate gradient, adam_step_sum_kernel's math)
//                        and, with SGA on, the NEXT step's sample of the freshly updated latents (w_hat, d w_hat / d w)
//                        while they are still in registers -- the table is read and written once per step instead of four
//                        times (bit-rate kernel, SGA kernel, Adam kernel) and three launches go away;
//   the last CTA         (arrival ticket) reduces the bit-rate partial sums, runs the density model's Adam segments that
//                        wait for them, advances the step counters and the draw counters.
#pragma once
#include "entropy_kernels.cuh"
#include "sga_kernels.cuh"

namespace shacira {

struct TableAdam {
    float* p;                 // latents [n]
    float* g;                 // grid gradient (cleared after use)
    const float* gmul;        // d w_hat / d w of THIS step's sample (SGA) or NULL
    const float* g2;          // bit-rate gradient or NULL
    const float* scale2;      // device scalar lambda or NULL
    float mul2;               // 1 / rows
    float* m;
    float* v;
    int64_t n;
    float lr, weight_decay;
    // next step's SGA sample (w_hat == NULL: off)
    const float* temperature;
    int diff_sampling;
    unsigned long long seed;
    unsigned long long* rng_step;   // index of the next draw; advanced by the last CTA
    float* w_hat;
    float* dw;
    // the bit-rate loss of the table evaluated in the same pass (ent_params == NULL: off; latent_dim = 1 only): the
    // latents' bit-rate gradient never goes through memory, the density model's gradients are reduced by the last CTA,
    // which then runs the density model's Adam segments (they are skipped by their own CTAs)
    const float* ent_params;        // [4][3][1] = {f1..f4} x {h, b, a}
    int ent_layers;
    const float* ent_noise;         // injected U(-1/2, 1/2) draws [n], or NULL: drawn in the kernel
    unsigned long long ent_seed;
    unsigned long long* ent_rng_step;
    float* ent_partials;            // scratch [table CTAs][13]
    double* bits;                   // [1] total bits
    float* g_prob;                  // [4][3][1] gradients w.r.t. the raw parameters (written by the last CTA)
};
constexpr int kOptEnt = 13;   // bits | {d softplus(h), d b, d tanh(a)} x 4 layers

// kSnap: best-state selection (shacira_fit_snapshot_t). The parameters are in registers right before their update, and
// the arrival ticket orders every CTA's read of best_loss before the last CTA's write of it; kSnap = false compiles to
// the kernel without it.
template <bool kSnap>
__global__ void __launch_bounds__(256)
fit_optimizer_kernel(const __grid_constant__ AdamSegs S, const __grid_constant__ TableAdam Tb, float beta1, float beta2,
                     float eps, float* __restrict__ step_small, float* __restrict__ step_table,
                     const float* __restrict__ scale, const float* __restrict__ div, float* __restrict__ A_out, int C, int F,
                     unsigned* __restrict__ ticket, const __grid_constant__ shacira_fit_snapshot_t snap) {
    // this step's loss, bit for bit what ImageFitStep.rgb_loss() returns, against the best so far (NaN is never taken)
    bool take = false;
    float loss_t = 0.0f;
    if constexpr (kSnap) {
        loss_t = (float)(*snap.sse / (double)snap.count);
        take = loss_t < *snap.best_loss;
    }
    if ((int)blockIdx.x < S.num) {
        const float t = *step_small + 1.0f;
        const float bc1 = 1.0f - powf(beta1, t), inv_sqrt_bc2 = rsqrtf(1.0f - powf(beta2, t));
        const shacira_adam_seg_t& sg = S.seg[blockIdx.x];
        const float gs = sg.grad_mul * (sg.grad_scale ? *sg.grad_scale : 1.0f);
        const float step_size = sg.lr / bc1;
        // density-model segments wait for the bit-rate reduction when it runs in this launch (last CTA, below)
        const bool deferred = Tb.ent_params && sg.grad >= Tb.g_prob && sg.grad < Tb.g_prob + 12;
        float* keep = nullptr;
        if constexpr (kSnap) {
            if (take) keep = snap.seg_param[blockIdx.x];
            if (take && sg.param == scale) {   // the A this step's forward used, and the div it was made with
                for (int e = threadIdx.x; e < C * F; e += 256) snap.A[e] = A_out[e];
                for (int e = threadIdx.x; e < C; e += 256) snap.div[e] = div[e];
            }
        }
        for (int i = threadIdx.x; i < (deferred ? 0 : sg.n); i += 256) {
            float g = 0.0f;
            for (int r = 0; r < sg.grad_rows; ++r) g += sg.grad[(size_t)r * sg.grad_row_stride + i];
            if (sg.zero_grad != 0.0f)
                for (int r = 0; r < sg.grad_rows; ++r) const_cast<float*>(sg.grad)[(size_t)r * sg.grad_row_stride + i] = 0.0f;
            g *= gs;
            if (sg.grad_div) g /= sg.grad_div[i / sg.div_group];
            const float p = sg.param[i];
            if constexpr (kSnap) {
                if (keep) keep[i] = p;
            }
            const float gk = fmaf(sg.weight_decay, p, g);
            const float mk = fmaf(beta1, sg.exp_avg[i], (1.0f - beta1) * gk);
            const float vk = fmaf(beta2, sg.exp_avg_sq[i], (1.0f - beta2) * gk * gk);
            sg.exp_avg[i] = mk;
            sg.exp_avg_sq[i] = vk;
            sg.param[i] = p - step_size * mk / (sqrtf(vk) * inv_sqrt_bc2 + eps);
        }
        __syncthreads();
        if (A_out && sg.param == scale)
            for (int e = threadIdx.x; e < C * F; e += 256) A_out[e] = scale[e] / div[e / F];
    } else {
        __shared__ float s_bc[2];   // bias corrections: two powf per CTA instead of per thread
        if (threadIdx.x == 0) {
            const float t = *step_table + 1.0f;
            s_bc[0] = 1.0f - powf(beta1, t);
            s_bc[1] = rsqrtf(1.0f - powf(beta2, t));
        }
        __syncthreads();
        const float bc1 = s_bc[0], inv_sqrt_bc2 = s_bc[1];
        const float step_size = Tb.lr / bc1;
        const float s2 = Tb.g2 ? (Tb.scale2 ? *Tb.scale2 * Tb.mul2 : Tb.mul2) : 0.0f;
        const bool sga = Tb.w_hat != nullptr;
        float tau = 1.0f;
        uint32_t base = 0u;
        if (sga) {
            tau = __ldg(Tb.temperature);
            base = sga_rng_base(Tb.rng_step ? *Tb.rng_step : 0ull, Tb.seed);
        }
        const bool ent = Tb.ent_params != nullptr;
        __shared__ float e_sp[4], e_b[4], e_ta[4], e_acc[kOptEnt];
        uint32_t ent_base = 0u;
        if (ent) {
            if (threadIdx.x < 4) {
                const float h = Tb.ent_params[threadIdx.x * 3 + 0], a = Tb.ent_params[threadIdx.x * 3 + 2];
                e_sp[threadIdx.x] = (h > 20.0f) ? h : log1pf(expf(h));     // F.softplus: beta 1, threshold 20
                e_b[threadIdx.x] = Tb.ent_params[threadIdx.x * 3 + 1];
                e_ta[threadIdx.x] = (threadIdx.x < 3) ? tanhf(a) : 0.0f;
            }
            if (threadIdx.x < kOptEnt) e_acc[threadIdx.x] = 0.0f;
            if (!Tb.ent_noise) {
                const unsigned long long st = Tb.ent_rng_step ? *Tb.ent_rng_step : 0ull;   // entropy_kernel's stream
                ent_base = (uint32_t)st * 0x9E3779B9u + (uint32_t)(st >> 32) * 0x7F4A7C15u +
                           (uint32_t)Tb.ent_seed * 0x85EBCA6Bu + (uint32_t)(Tb.ent_seed >> 32) * 0xC2B2AE35u;
            }
            __syncthreads();
        }
        const int64_t i4 = ((int64_t)(blockIdx.x - S.num) * 256 + threadIdx.x) * 4;
        const int cnt = (int)max((int64_t)0, min((int64_t)4, Tb.n - i4));
        const bool vec = cnt == 4 && ((reinterpret_cast<uintptr_t>(Tb.p) | reinterpret_cast<uintptr_t>(Tb.g) |
                                       reinterpret_cast<uintptr_t>(Tb.g2) | reinterpret_cast<uintptr_t>(Tb.m) |
                                       reinterpret_cast<uintptr_t>(Tb.v) | reinterpret_cast<uintptr_t>(Tb.gmul) |
                                       reinterpret_cast<uintptr_t>(Tb.w_hat) | reinterpret_cast<uintptr_t>(Tb.dw)) & 15) == 0;
        float P[4], M[4], V[4], G[4], Q[4], H[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { P[k] = M[k] = V[k] = G[k] = H[k] = 0.0f; Q[k] = 1.0f; }
        if (vec) {
            *reinterpret_cast<float4*>(P) = *reinterpret_cast<const float4*>(Tb.p + i4);
            *reinterpret_cast<float4*>(M) = *reinterpret_cast<const float4*>(Tb.m + i4);
            *reinterpret_cast<float4*>(V) = *reinterpret_cast<const float4*>(Tb.v + i4);
            *reinterpret_cast<float4*>(G) = *reinterpret_cast<const float4*>(Tb.g + i4);
            if (Tb.gmul) *reinterpret_cast<float4*>(Q) = *reinterpret_cast<const float4*>(Tb.gmul + i4);
            if (Tb.g2) *reinterpret_cast<float4*>(H) = *reinterpret_cast<const float4*>(Tb.g2 + i4);
        } else {
            for (int k = 0; k < cnt; ++k) {
                P[k] = Tb.p[i4 + k]; M[k] = Tb.m[i4 + k]; V[k] = Tb.v[i4 + k]; G[k] = Tb.g[i4 + k];
                if (Tb.gmul) Q[k] = Tb.gmul[i4 + k];
                if (Tb.g2) H[k] = Tb.g2[i4 + k];
            }
        }
        if constexpr (kSnap) {
            if (take) {   // the continuous latents theta_t (under SGA the forward saw their sample)
                if (vec) *reinterpret_cast<float4*>(snap.table + i4) = *reinterpret_cast<const float4*>(P);
                else for (int k = 0; k < cnt; ++k) snap.table[i4 + k] = P[k];
            }
        }
        float s2e = s2;
        if (ent) {
            // bit-rate value and gradients of this thread's (up to) four latents: four independent chains
            s2e = Tb.scale2 ? *Tb.scale2 * Tb.mul2 : Tb.mul2;
            const int m = min(Tb.ent_layers, 4) - 1;
            const float inv_ln2 = 1.0f / 0.6931471805599453f;
            float d_sp[4] = {0, 0, 0, 0}, d_b[4] = {0, 0, 0, 0}, d_ta[4] = {0, 0, 0, 0};
            float my_bits = 0.0f;
            // two latents at a time, layer by layer: four independent CDF chains (x +- 1/2 of both) share every basic
            // block, so their transcendental latencies overlap (one latent at a time left the launch latency bound)
#pragma unroll
            for (int k0 = 0; k0 < 4; k0 += 2) {
                float xs[2], nzv[2];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int64_t e = min(i4 + k0 + q, Tb.n - 1);   // clamped: dead lanes compute on a valid entry, masked below
                    if (Tb.ent_noise) {
                        nzv[q] = Tb.ent_noise[e];
                    } else {
                        uint32_t h = (uint32_t)e + ent_base;      // lowbias32 finaliser (as entropy_kernel)
                        h ^= h >> 16; h *= 0x7feb352du; h ^= h >> 15; h *= 0x846ca68bu; h ^= h >> 16;
                        h += (uint32_t)(e >> 32) * 0x9E3779B9u;
                        nzv[q] = (float)(h >> 8) * 5.9604644775390625e-08f - 0.5f;
                    }
                    xs[q] = P[k0 + q] + nzv[q];
                }
                CdfTrace tr[4];                                   // [2 q + 0] upper, [2 q + 1] lower
                float xc[4] = {xs[0] + 0.5f, xs[0] - 0.5f, xs[1] + 0.5f, xs[1] - 0.5f};
#pragma unroll
                for (int l = 0; l < 3; ++l) {
                    if (l < m) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            tr[c].xin[l] = xc[c];
                            const float u = fmaf(xc[c], e_sp[l], e_b[l]);
                            const float th = fast_tanh(u);
                            tr[c].th[l] = th;
                            xc[c] = fmaf(th, e_ta[l], u);
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    tr[c].xf = xc[c];
                    tr[c].F = fast_sigmoid(fmaf(xc[c], e_sp[3], e_b[3]));
                }
                float gp[2];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const bool livek = k0 + q < cnt;
                    const float pr = tr[2 * q].F - tr[2 * q + 1].F;
                    const float raw = -logf(pr + 1e-10f) * inv_ln2;
                    my_bits += livek ? fminf(fmaxf(raw, 0.0f), 50.0f) : 0.0f;
                    const float g_raw = (livek && raw >= 0.0f && raw <= 50.0f) ? 1.0f : 0.0f;
                    gp[q] = -g_raw * inv_ln2 / (pr + 1e-10f);
                }
                // reverse sweeps of the four chains, layer by layer
                float gx[4], gv[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float G = (c & 1) ? -gp[c >> 1] : gp[c >> 1];
                    gv[c] = G * tr[c].F * (1.0f - tr[c].F);
                    d_sp[3] += gv[c] * tr[c].xf;
                    d_b[3] += gv[c];
                    gx[c] = gv[c] * e_sp[3];
                }
#pragma unroll
                for (int l = 2; l >= 0; --l) {
                    if (l < m) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float th = tr[c].th[l];
                            d_ta[l] += gx[c] * th;
                            const float gu = gx[c] * fmaf(1.0f - th * th, e_ta[l], 1.0f);
                            d_sp[l] += gu * tr[c].xin[l];
                            d_b[l] += gu;
                            gx[c] = gu * e_sp[l];
                        }
                    }
                }
                H[k0] = gx[0] + gx[1];
                H[k0 + 1] = gx[2] + gx[3];
            }
            float red[kOptEnt];
            red[0] = my_bits;
#pragma unroll
            for (int k = 0; k < 4; ++k) { red[1 + 3 * k] = d_sp[k]; red[2 + 3 * k] = d_b[k]; red[3 + 3 * k] = d_ta[k]; }
#pragma unroll
            for (int q = 0; q < kOptEnt; ++q) {
                const float v = warp_sum(red[q]);
                if ((threadIdx.x & 31) == 0) atomicAdd(&e_acc[q], v);
            }
        }
        float WH[4], DW[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float gi = Tb.gmul ? G[k] * Q[k] : G[k];
            if (ent) gi = fmaf(s2e, H[k], gi);
            else if (Tb.g2) gi = fmaf(s2, H[k], gi);
            const float gk = fmaf(Tb.weight_decay, P[k], gi);
            M[k] = fmaf(beta1, M[k], (1.0f - beta1) * gk);
            V[k] = fmaf(beta2, V[k], (1.0f - beta2) * gk * gk);
            P[k] -= step_size * M[k] / (sqrtf(V[k]) * inv_sqrt_bc2 + eps);
            WH[k] = DW[k] = 0.0f;
            if (sga && k < cnt) {
                const int64_t i = i4 + k;
                sga_sample(P[k], sga_uniform((uint32_t)(2 * i), base), sga_uniform((uint32_t)(2 * i + 1), base), tau,
                           Tb.diff_sampling, WH[k], DW[k]);
            }
        }
        if (vec) {
            *reinterpret_cast<float4*>(Tb.p + i4) = *reinterpret_cast<float4*>(P);
            *reinterpret_cast<float4*>(Tb.m + i4) = *reinterpret_cast<float4*>(M);
            *reinterpret_cast<float4*>(Tb.v + i4) = *reinterpret_cast<float4*>(V);
            *reinterpret_cast<float4*>(Tb.g + i4) = make_float4(0.f, 0.f, 0.f, 0.f);
            if (sga) {
                *reinterpret_cast<float4*>(Tb.w_hat + i4) = *reinterpret_cast<float4*>(WH);
                if (Tb.dw) *reinterpret_cast<float4*>(Tb.dw + i4) = *reinterpret_cast<float4*>(DW);
            }
        } else {
            for (int k = 0; k < cnt; ++k) {
                Tb.p[i4 + k] = P[k]; Tb.m[i4 + k] = M[k]; Tb.v[i4 + k] = V[k]; Tb.g[i4 + k] = 0.0f;
                if (sga) { Tb.w_hat[i4 + k] = WH[k]; if (Tb.dw) Tb.dw[i4 + k] = DW[k]; }
            }
        }
        if (ent) {   // this CTA's bit-rate partial sums
            __syncthreads();
            if (threadIdx.x < kOptEnt) Tb.ent_partials[(size_t)(blockIdx.x - S.num) * kOptEnt + threadIdx.x] = e_acc[threadIdx.x];
        }
    }
    // every CTA has read the counters when the last one arrives: it advances them
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (Tb.ent_params) {
        // the last CTA: reduce the table CTAs' partial rows in a fixed order, chain to the raw parameters, then run the
        // density model's Adam segments that waited for it
        __shared__ float tot[kOptEnt];
        const int nb = (int)gridDim.x - S.num, lane = threadIdx.x & 31;
        for (int v = threadIdx.x >> 5; v < kOptEnt; v += 8) {
            double sum = 0.0;
            for (int b = lane; b < nb; b += 32) sum += (double)Tb.ent_partials[(size_t)b * kOptEnt + v];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            if (lane == 0) {
                tot[v] = (float)sum;
                if (v == 0) *Tb.bits = sum;
            }
        }
        __syncthreads();
        if (threadIdx.x < 4) {
            const int k = threadIdx.x;
            const float h = Tb.ent_params[k * 3 + 0], a = Tb.ent_params[k * 3 + 2];
            const float ta = (k < 3) ? tanhf(a) : 0.0f;
            Tb.g_prob[k * 3 + 0] = tot[1 + 3 * k] * (1.0f / (1.0f + expf(-h)));   // d softplus / dh
            Tb.g_prob[k * 3 + 1] = tot[2 + 3 * k];
            Tb.g_prob[k * 3 + 2] = (k < 3) ? tot[3 + 3 * k] * (1.0f - ta * ta) : 0.0f;
        }
        __syncthreads();
        if (threadIdx.x < S.num) {
            const shacira_adam_seg_t& sg = S.seg[threadIdx.x];
            if (sg.grad >= Tb.g_prob && sg.grad < Tb.g_prob + 12) {
                const float t = *step_small + 1.0f;
                const float bc1 = 1.0f - powf(beta1, t), inv_sqrt_bc2 = rsqrtf(1.0f - powf(beta2, t));
                const float gs = sg.grad_mul * (sg.grad_scale ? *sg.grad_scale : 1.0f);
                float* keep = nullptr;
                if constexpr (kSnap) {
                    if (take) keep = snap.seg_param[threadIdx.x];
                }
                for (int i = 0; i < sg.n; ++i) {
                    float g = 0.0f;
                    for (int r = 0; r < sg.grad_rows; ++r) g += sg.grad[(size_t)r * sg.grad_row_stride + i];
                    g *= gs;
                    if (sg.grad_div) g /= sg.grad_div[i / sg.div_group];
                    const float p = sg.param[i];
                    if constexpr (kSnap) {
                        if (keep) keep[i] = p;
                    }
                    const float gk = fmaf(sg.weight_decay, p, g);
                    const float mk = fmaf(beta1, sg.exp_avg[i], (1.0f - beta1) * gk);
                    const float vk = fmaf(beta2, sg.exp_avg_sq[i], (1.0f - beta2) * gk * gk);
                    sg.exp_avg[i] = mk;
                    sg.exp_avg_sq[i] = vk;
                    sg.param[i] = p - (sg.lr / bc1) * mk / (sqrtf(vk) * inv_sqrt_bc2 + eps);
                }
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if constexpr (kSnap) {
            if (take) {
                *snap.best_loss = loss_t;
                *snap.best_step = (int64_t)*step_small;
            }
        }
        *step_small += 1.0f;
        *step_table += 1.0f;
        if (Tb.w_hat && Tb.rng_step) *Tb.rng_step += 1ull;
        if (Tb.ent_params && !Tb.ent_noise && Tb.ent_rng_step) *Tb.ent_rng_step += 1ull;
        *ticket = 0u;
    }
}

}  // namespace shacira
