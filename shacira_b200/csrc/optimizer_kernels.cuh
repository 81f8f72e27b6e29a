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

// The training schedule of the fit (shacira_fit_schedule_t), evaluated on the device: lambda and the SGA temperature
// BEFORE step `it` (0-based), in double and in the host formula's operation order (no FMA contraction), so that the
// float the kernel stores is the one a host fill_ of the same Python expression stores.
__device__ __forceinline__ float sched_lambda(const shacira_fit_schedule_t& sc, int64_t it) {
    if (sc.lambda_kind == SHACIRA_LAMBDA_FIX) return (float)sc.lambda_start;
    // end + 0.5 * (start - end) * (1 + cos(pi * it / num_epochs))        (utils/schedulers.py, 'cosine')
    const double c = cos(__ddiv_rn(__dmul_rn(3.141592653589793, (double)it), (double)sc.num_epochs));
    return (float)__dadd_rn(sc.lambda_end,
                            __dmul_rn(__dmul_rn(0.5, __dadd_rn(sc.lambda_start, -sc.lambda_end)), __dadd_rn(1.0, c)));
}
__device__ __forceinline__ float sched_temperature(const shacira_fit_schedule_t& sc, int64_t it) {
    // max(end, exp(-ln(1 / end) * (it + 1) / num_epochs / decay_period))  (DecayScheduler 'exp', start 1)
    const double x = __ddiv_rn(__ddiv_rn(__dmul_rn(-log(__ddiv_rn(1.0, sc.temperature_end)), (double)(it + 1)),
                                         (double)sc.num_epochs), sc.decay_period);
    return (float)fmax(sc.temperature_end, exp(x));
}

// kSnap: best-state selection (shacira_fit_snapshot_t). The parameters are in registers right before their update, and
// the arrival ticket orders every CTA's read of best_loss before the last CTA's write of it; kSnap = false compiles to
// the kernel without it.
template <bool kSnap>
__global__ void __launch_bounds__(256)
fit_optimizer_kernel(const __grid_constant__ AdamSegs S, const __grid_constant__ TableAdam Tb, float beta1, float beta2,
                     float eps, float* __restrict__ step_small, float* __restrict__ step_table,
                     const float* __restrict__ scale, const float* __restrict__ div, float* __restrict__ A_out, int C, int F,
                     unsigned* __restrict__ ticket, const __grid_constant__ shacira_fit_snapshot_t snap) {
#define SHACIRA_FIT_OPT_SCHED 0
#include "fit_optimizer_body.inl"
#undef SHACIRA_FIT_OPT_SCHED
}

// The scheduled form (shacira_fit_optimizer_step_sched): the last CTA appends this step's record to the log and writes
// the NEXT step's lambda (*Tb.scale2) and temperature (*Tb.temperature). Every CTA that reads them (table CTAs,
// density-model segments) does so before the arrival ticket, the deferred density-model segments inside the last CTA
// before its thread 0 writes them; the next step's SGA sample drawn in this launch used this step's temperature, as
// with the host-side hooks.
template <bool kSnap>
__global__ void __launch_bounds__(256)
fit_optimizer_sched_kernel(const __grid_constant__ AdamSegs S, const __grid_constant__ TableAdam Tb, float beta1,
                           float beta2, float eps, float* __restrict__ step_small, float* __restrict__ step_table,
                           const float* __restrict__ scale, const float* __restrict__ div, float* __restrict__ A_out,
                           int C, int F, unsigned* __restrict__ ticket,
                           const __grid_constant__ shacira_fit_snapshot_t snap,
                           const __grid_constant__ shacira_fit_schedule_t sc, const double* __restrict__ bits) {
#define SHACIRA_FIT_OPT_SCHED 1
#include "fit_optimizer_body.inl"
#undef SHACIRA_FIT_OPT_SCHED
}

}  // namespace shacira
