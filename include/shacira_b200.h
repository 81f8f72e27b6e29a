/*
 * shacira_b200.h -- C ABI of the B200-native latent hash-grid hot path.
 *
 * One shared library (shacira_b200/libshacira_b200.so, built by shacira_b200/build.py with
 * nvcc for sm_100a) exports exactly these symbols. There are no torch types in any
 * signature: plain device pointers, sizes and a CUDA stream handle. The Python host side
 * (shacira_b200/_lib.py) binds them with ctypes; INTEGRATION.md shows the binding a
 * maintainer of the reference would add.
 *
 * Every entry point
 *   - returns 0 on success or a negative SHACIRA_ERR_* code (never throws, never aborts);
 *     shacira_last_error() returns the message of the last failure on the calling thread;
 *   - launches asynchronously on `stream` (NULL = legacy default stream) on the CURRENT
 *     device, like the reference (`at::cuda::getCurrentCUDAStream()`,
 *     wisp/csrc/ops/hashgrid_interpolate2d_cuda.cu:116-118), and is re-entrant;
 *   - takes `coords` as float32 [n, dim] row-major in [-1, 1], `resolutions` and
 *     `first_idx` as HOST int32[num_lods] (the reference passes first_idx as a device
 *     tensor and dereferences it in-kernel; the torch shim caches the host copy);
 *   - computes in fp32 (the graded path; kodak.yaml disables AMP).
 *
 * Level l of the table holds min(2^bitwidth, res_l^dim) rows starting at row first_idx[l]
 * (wisp/models/grids/latent_grid.py:100-112). Corner index, weights and summation follow
 * wisp/csrc/ops/hashgrid_interpolate{,2d}_cuda.cu; see DESIGN.md for the exact arithmetic.
 */
#ifndef SHACIRA_B200_H_
#define SHACIRA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHACIRA_ABI_VERSION 1
#define SHACIRA_MAX_LEVELS 32

#define SHACIRA_OK 0
#define SHACIRA_ERR_INVALID_ARGUMENT (-1) /* null pointer, bad dim/size/bitwidth ...            */
#define SHACIRA_ERR_UNSUPPORTED (-2)      /* channel combination without a compiled kernel      */
#define SHACIRA_ERR_CUDA (-3)             /* a CUDA runtime call or launch failed               */
#define SHACIRA_ERR_Q2_WINDOW (-4)        /* level where the reference's int32 dense predicate  */
                                          /* overflows (res^3 wraps): behaviour undefined there */
#define SHACIRA_ERR_NO_DEVICE (-5)        /* no CUDA device visible                             */

typedef void* shacira_stream_t; /* cudaStream_t */

/* ---- library info ------------------------------------------------------------------- */
int shacira_abi_version(void);
const char* shacira_last_error(void);
/* Number of kernels launched by this library since load (process-wide, all threads). */
int64_t shacira_launch_count(void);
/* sm count / L2 bytes / max persisting L2 bytes of the current device. */
int shacira_device_info(int32_t* sm_count, int64_t* l2_bytes, int64_t* l2_persist_max);
/* Pin [base, base+bytes) in L2 for kernels subsequently launched on `stream`
 * (cudaStreamAttributeAccessPolicyWindow, hitRatio clipped to the persisting carve-out).
 * bytes == 0 clears the window. */
int shacira_l2_pin(const void* base, int64_t bytes, shacira_stream_t stream);

/* ---- plain hash grid: replaces wisp._C.ops.hashgrid_interpolate{,2d}_cuda ------------- */
/* hashgrid_interpolate.h:18-23 (3D) and :35-40 (2D); host loops hashgrid_interpolate.cpp:44-66,
 * 130-152. ALL levels in one launch. feats[n, num_lods*feature_dim], element
 * [i, lod*feature_dim + j]. feature_dim in {1,2,4,8}. */
int shacira_hashgrid_forward(int32_t dim, const float* coords, int64_t n, const float* codebook,
                             const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                             int32_t codebook_bitwidth, int32_t feature_dim, float* feats, shacira_stream_t stream);

/* hashgrid_interpolate.h:25-33, :42-50; host loops hashgrid_interpolate.cpp:68-100,154-186.
 * grad_codebook[table_rows, feature_dim] is zero-filled by this call when zero_first != 0
 * (the reference allocates zeros_like, .cpp:81,167) and accumulated into otherwise.
 * The reference's grad_coords output is computed with wrong indices and discarded
 * (SURVEY Q6); it is not provided. */
int shacira_hashgrid_backward(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                              const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                              int32_t codebook_bitwidth, int32_t feature_dim, int64_t table_rows, int32_t zero_first,
                              float* grad_codebook, shacira_stream_t stream);

/* Level-local corner indices idx[n, num_lods, 2^dim] (int32) and weights w[n, num_lods, 2^dim]
 * exactly as the forward/backward kernels use them (bit-exactness tests, debugging). */
int shacira_hashgrid_corners(int32_t dim, const float* coords, int64_t n, const int32_t* resolutions,
                             int32_t num_lods, int32_t codebook_bitwidth, int32_t* idx, float* w,
                             shacira_stream_t stream);

/* ---- fused latent grid: replaces latent_dec(codebook) + hashgrid*() ------------------ */
/* LatentGrid.interpolate (wisp/models/grids/latent_grid.py:340-382) with an affine latent
 * decoder (LatentDecoder / HierarchicalLatentDecoder with num_layers_dec = 0,
 * wisp/models/latent_decoders/basic_latent_decoder.py:85-95,182-198):
 *   q      = round_flag ? rint(latents) : latents           (StraightThrough, :28-36)
 *   z[i,l] = sum_k w_k * q[first_idx[l] + idx_k]             (latent_dim channels)
 *   feats[i, l*F + f] = sum_c z[i,l,c] * A[la,c,f] + shift[la,f]
 * with A = scale / div[:,None] prepared by the caller ([1|L, C, F] row-major; la = l when
 * per_level != 0 else 0) and shift [1|L, F] or NULL. Interpolating before the affine map
 * equals the reference's decode-then-interpolate because the weights sum to 1 (DESIGN.md).
 * zsave (nullable) receives z[n, L*C] for the backward pass.
 * latent_dim C in {1,2,4}, feature_dim F in {1,2,4,8}. */
int shacira_latent_forward(int32_t dim, const float* coords, int64_t n, const float* latents,
                           const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                           int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, int32_t round_flag,
                           const float* A, const float* shift, int32_t per_level, float* feats, float* zsave,
                           shacira_stream_t stream);

/* Backward of the above. grad_latents[table_rows, C] += w_k * sum_f g[i,l,f] * A[la,c,f]
 * (straight-through: the rounding passes gradients unchanged); grad_A[L, C, F] and
 * grad_shift[L, F] are ACCUMULATED into (caller zero-fills); either may be NULL. With
 * per_level != 0 row l is level l's gradient; with one shared decoder (per_level == 0) only
 * the SUM over the L rows is defined (the caller adds them; a kernel may put it all in row 0). zsave is the forward's
 * z[n, L*C] (required when grad_A != NULL). */
int shacira_latent_backward(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                            const float* zsave, const int32_t* first_idx, const int32_t* resolutions,
                            int32_t num_lods, int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                            const float* A, int32_t per_level, int64_t table_rows, int32_t zero_first,
                            float* grad_latents, float* grad_A, float* grad_shift, shacira_stream_t stream);
/* The same restricted to the levels whose bit is set in `level_mask` (bit l = level l): gradients of the other
 * levels' rows and decoder slots are left untouched. The rows of a level are a contiguous range of the table, so a
 * data-parallel caller can run the backward in a few level chunks and start the all-reduce of one chunk's rows while
 * the next chunk computes (benchmarks/nerf_dp.py --chunks). zero_first clears the WHOLE table: pass it with the first
 * chunk only. */
int shacira_latent_backward_levels(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                                   const float* zsave, const int32_t* first_idx, const int32_t* resolutions,
                                   int32_t num_lods, int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                                   const float* A, int32_t per_level, int64_t table_rows, int32_t zero_first,
                                   uint32_t level_mask, float* grad_latents, float* grad_A, float* grad_shift,
                                   shacira_stream_t stream);


/* ---- tiled fast path: spatial plan + planned fused forward / backward ----------------- */
/* A plan bins the points of ONE coordinate set into power-of-two spatial tiles (about
 * tile_points per tile; 0 = default) and keeps the permutation and a sorted copy of the
 * coordinates on the device. It depends only on the coordinates, not on the levels, and is
 * reusable for every forward/backward over those coordinates (an image fit uses the same
 * coordinates for tens of thousands of steps). Creation is asynchronous on `stream`.
 * The planned kernels give one CTA per tile, stage the grid nodes the tile touches in shared
 * memory (forward) or accumulate into them in fixed point (backward); DESIGN.md "tiled path".
 * Results follow the same arithmetic as the unplanned entry points; outputs are in the
 * ORIGINAL point order. */
typedef struct shacira_plan shacira_plan_t;
int shacira_plan_create(int32_t dim, const float* coords, int64_t n, int32_t tile_points, shacira_stream_t stream,
                        shacira_plan_t** plan);
/* Re-bin `plan` for a new coordinate set, reusing its device allocation when large enough
 * (workloads whose coordinates change every step, e.g. NeRF samples). */
int shacira_plan_rebuild(shacira_plan_t* plan, int32_t dim, const float* coords, int64_t n, int32_t tile_points,
                         shacira_stream_t stream);
int shacira_plan_destroy(shacira_plan_t* plan);
int shacira_plan_info(const shacira_plan_t* plan, int64_t* n, int32_t* dim, int32_t* tiles_per_axis,
                      int32_t* ntiles);
/* Device pointers of the plan's arrays (perm[n], coords_sorted[n,dim], tile_off[ntiles+1]) for tests. */
int shacira_plan_debug(const shacira_plan_t* plan, const int32_t** perm, const float** coords_sorted,
                       const int32_t** tile_off);
/* sorted_io != 0: the planned forward writes row j of `feats`, and the planned backward reads row j of
 * `grad_output`, for the point at SORTED position j (perm[j] of shacira_plan_debug is its original index) instead of
 * at the original index. A consumer that is order independent -- a per-point MLP with a mean loss over a static
 * coordinate set, its targets permuted once -- then exchanges contiguous, tile-ordered rows with the grid, and the
 * kernels lose the perm -> row dependent load. Off by default (reference semantics). */
int shacira_plan_set_sorted_io(shacira_plan_t* plan, int32_t sorted_io);
/* Same contract as shacira_latent_forward (no zsave: the backward recomputes the interpolation). */
int shacira_latent_forward_planned(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                                   const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth,
                                   int32_t latent_dim, int32_t feature_dim, int32_t round_flag, const float* A,
                                   const float* shift, int32_t per_level, float* feats, shacira_stream_t stream);
/* Same contract as shacira_latent_backward; `latents` (+ round_flag) replace zsave and are needed
 * only when grad_A / grad_shift are requested. */
int shacira_latent_backward_planned(const shacira_plan_t* plan, const float* grad_output, const float* latents,
                                    const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                                    int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                                    int32_t round_flag, const float* A, int32_t per_level, int64_t table_rows,
                                    int32_t zero_first, float* grad_latents, float* grad_A, float* grad_shift,
                                    shacira_stream_t stream);
/* The same with `level_max` (device, [num_lods * feature_dim], may be NULL): upper bounds of |grad_output| per
 * column, e.g. reduced by the kernel that produced the rows (shacira_mlp_mse_step_bounded). The tiled backward
 * accumulates in fixed point and otherwise finds the bound itself with an extra pass over every tile's gradient rows;
 * with the bound that second read of grad_output is skipped. The fixed-point step is then 2^-19 of the GLOBAL
 * per-level bound instead of the tile's own maximum. A bound that is too small is an error of the caller (sums wrap). */
int shacira_latent_backward_planned_bounded(const shacira_plan_t* plan, const float* grad_output,
                                            const float* latents, const int32_t* first_idx, const int32_t* resolutions,
                                            int32_t num_lods, int32_t codebook_bitwidth, int32_t latent_dim,
                                            int32_t feature_dim, int32_t round_flag, const float* A, int32_t per_level,
                                            int64_t table_rows, int32_t zero_first, float* grad_latents, float* grad_A,
                                            float* grad_shift, const float* level_max, shacira_stream_t stream);

/* 3D plans (NeRF samples, new coordinates every step: shacira_plan_rebuild per step). The planned 3D kernels run one
 * thread per sample over the plan's tile-sorted samples -- neighbouring lanes share the cache lines of the coarse
 * and middle levels -- fetch the two x-neighbour corners of a cell with ONE aligned 16-byte load (forward) / add to
 * them with ONE vector red (backward), and accumulate the coarse levels per tile in shared memory (fixed point) on a
 * forked stream. `zsave` [n, L*C] is scratch private to this pair of calls (rows in the plan's sorted order): the
 * forward writes the interpolated latents, the backward reads them for grad_A. Other arguments as
 * shacira_latent_forward / shacira_latent_backward. latent_dim in {1, 2}; tables 16-byte aligned. */
int shacira_latent_forward_planned_z(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                                     const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth,
                                     int32_t latent_dim, int32_t feature_dim, int32_t round_flag, const float* A,
                                     const float* shift, int32_t per_level, float* feats, float* zsave,
                                     shacira_stream_t stream);
int shacira_latent_backward_planned_z(const shacira_plan_t* plan, const float* grad_output, const float* zsave,
                                      const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                                      int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, const float* A,
                                      int32_t per_level, int64_t table_rows, int32_t zero_first, float* grad_latents,
                                      float* grad_A, float* grad_shift, shacira_stream_t stream);

/* ---- factorized-density bit-rate estimate -------------------------------------------- */
/* LatentGrid.ent_loss (latent_grid.py:122-136) + BitEstimator/Bitparm
 * (wisp/models/prob_models/bit_estimator.py:9-65), forward and backward in one pass:
 *   x = latents + noise (noise != NULL)  or  rint(latents) (noise == NULL, the is_val branch)
 *   p = CDF(x + .5) - CDF(x - .5);  bits = clamp(-log(p + 1e-10) / ln 2, 0, 50)
 * num_layers in 1..4 selects f1..f(num_layers-1) then f4 (bit_estimator.py:58-65).
 * params: float32 [4, 3, C] = {f1,f2,f3,f4} x {h,b,a} x channel (f4.a unused).
 * Outputs (all nullable except bits): bits[1 + num_lods] double = total, then per level;
 * grad_latents[T, C] = d total / d latents (written, not accumulated; zero when noise==NULL);
 * grad_params[4, 3, C] float32 = d total / d params (written).
 * first_idx (host, nullable with num_lods = 0) gives the per-level reduction. */
int shacira_entropy_bits(const float* latents, const float* noise, int64_t table_rows, int32_t latent_dim,
                         const float* params, int32_t num_layers, const int32_t* first_idx, int32_t num_lods,
                         double* bits, float* grad_latents, float* grad_params, void* scratch, int64_t scratch_bytes,
                         shacira_stream_t stream);
/* Device scratch for the block partials of shacira_entropy_bits: zero-fill it ONCE, then reuse it for every call
 * on the same stream (the kernel leaves it ready). scratch == NULL makes the call allocate from the stream's
 * memory pool instead (more launch overhead). */
/* The same in training mode with the U(-0.5, 0.5) noise (latent_grid.py:128-132) drawn INSIDE the kernel from a
 * counter-based hash of (element, *rng_step, seed) instead of read from a buffer: no RNG kernel, no noise tensor,
 * and a captured CUDA graph draws fresh noise on every replay because the call advances *rng_step (device uint64)
 * itself. `scratch` (shacira_entropy_scratch_bytes, zero-initialised once) is mandatory here. The reference's
 * torch.rand stream cannot be reproduced by any device generator; parity runs inject the noise through
 * shacira_entropy_bits. */
int shacira_entropy_bits_rng(const float* latents, uint64_t seed, uint64_t* rng_step, int64_t table_rows,
                             int32_t latent_dim, const float* params, int32_t num_layers, const int32_t* first_idx,
                             int32_t num_lods, double* bits, float* grad_latents, float* grad_params, void* scratch,
                             int64_t scratch_bytes, shacira_stream_t stream);
int64_t shacira_entropy_scratch_bytes(int32_t latent_dim, int32_t num_lods);

/* ---- symbols / histogram for LatentGrid.size() --------------------------------------- */
/* latent_grid.py:138-153: per channel q = rint(latents[:,c]); symbols[T, C] (int16,
 * nullable) = q, minmax[2*C] (int32) = {min_c, max_c}. Values must fit int16
 * (the reference casts to int16 for torchac, latent_grid.py:170). */
int shacira_quantize_symbols(const float* latents, int64_t table_rows, int32_t latent_dim, int16_t* symbols,
                             int32_t* minmax, shacira_stream_t stream);
/* counts[C, num_bins] (int64, ACCUMULATED) of rint(latents[:,c]) - lo[c]; lo is HOST int32[C]. */
int shacira_symbol_histogram(const float* latents, int64_t table_rows, int32_t latent_dim, const int32_t* lo,
                             int32_t num_bins, int64_t* counts, shacira_stream_t stream);

/* ---- fused decoder MLP + image loss (SURVEY section 8, row f-1) ----------------------- */
/* The reference's NeuralImage decoder (BasicDecoder: Linear(in,16) ReLU Linear(16,16) ReLU Linear(16,3), bias;
 * wisp/models/nefs/image.py:109-120, wisp/models/decoders/basic_decoders.py:60-100) applied to the grid
 * features, the loss ((pred - target)^2).mean() (wisp/trainers/image_trainer.py:298-300), and ALL gradients in
 * one pass: grad_features[n, in_dim] = dL/dfeatures (feed it to shacira_latent_backward*), pred[n, 3] (nullable).
 * Weights use the torch.nn.Linear layout W[out][in]. `out` is a device buffer of
 * 8 + 4*(16*in + 16 + 256 + 16 + 48 + 3) bytes, written by the call:
 *   double sum of squared errors (loss = sum / (3 n)) | float dL/dW1 | db1 | dW2 | db2 | dW3 | db3.
 * in_dim in {16, 24, 32}, hidden_dim = 16, out_dim = 3. */
int shacira_mlp_mse_step(const float* features, const float* target, int64_t n, int32_t in_dim, int32_t hidden_dim,
                         int32_t out_dim, const float* W1, const float* b1, const float* W2, const float* b2,
                         const float* W3, const float* b3, float* grad_features, float* pred, void* out,
                         shacira_stream_t stream);

/* The same, also reducing max |grad_features[:, j]| per input column j into grad_feature_absmax (device,
 * [in_dim], written by the call) for shacira_latent_backward_planned_bounded. in_dim = 16 only. */
int shacira_mlp_mse_step_bounded(const float* features, const float* target, int64_t n, int32_t in_dim,
                                 int32_t hidden_dim, int32_t out_dim, const float* W1, const float* b1, const float* W2,
                                 const float* b2, const float* W3, const float* b3, float* grad_features, float* pred,
                                 void* out, float* grad_feature_absmax, shacira_stream_t stream);

/* ---- grid forward + decoder MLP + MSE + grid backward in ONE tile-resident kernel (row f-1 as written) ----------
 * Replaces, for the static-coordinate image fit, the sequence shacira_latent_forward_planned ->
 * shacira_mlp_mse_step_bounded -> shacira_latent_backward_planned_bounded (reference: latent_grid.py:340-382 ->
 * nefs/image.py:109-120,152 -> image_trainer.py:298-300 and their autograd backward): the [n, 16] feature rows and
 * their gradient never leave the SM. `plan`: 2D, sorted-I/O mode (shacira_plan_set_sorted_io); `target_sorted`
 * [n, 3] in the plan's sorted order; latent_dim = feature_dim = 1, ONE affine decoder (A [1], shift [1] or NULL),
 * 16 levels that all fit a tile's shared-memory node box (else SHACIRA_ERR_UNSUPPORTED: use the three calls).
 * Weights in the torch.nn.Linear layout (W1 [16,16], W2 [16,16], W3 [3,16]). Outputs: grad_latents [table_rows]
 * (ACCUMULATED into), grad_A [16] / grad_shift [16] (accumulated; only the sum over the 16 rows is defined),
 * mlp_out as shacira_mlp_mse_step writes it (double SSE | dW1 | db1 | dW2 | db2 | dW3 | db3; cleared by the call). */
int shacira_fit_tile_step(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                          const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth, int32_t round_flag,
                          const float* A, const float* shift, const float* target_sorted, const float* W1,
                          const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                          int64_t table_rows, float* grad_latents, float* grad_A, float* grad_shift, void* mlp_out,
                          shacira_stream_t stream);

/* The forward-only sibling of shacira_fit_tile_step: turns a model of that shape into pixels (the final PSNR of a fit,
 * a decoded codec model, a render at another resolution) without writing the [n, 16] feature rows. Reference:
 * mlp(grid.interpolate(coords)) with STE rounding (latent_grid.py:340-382, nefs/image.py:109-120,152). Same shapes as
 * shacira_fit_tile_step; the latents are always rounded. `plan`: 2D, any mode; rows of `rgb` [n, 3] and `target` [n, 3]
 * follow the plan's convention (original point index, or tile order on a sorted-I/O plan). With target != NULL,
 * *sse_u8 (cleared by the call) receives sum (q(rgb) - q(target))^2 over all n x 3 values with
 * q(v) = (uint8)(clamp(v, 0, 1) * 255) -- the integer SSE behind the clamped PSNR of wisp/ops/image/metrics.py:39-57;
 * rgb may then be NULL (PSNR without writing the image). */
int shacira_fit_render(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                       const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth, const float* A,
                       const float* shift, const float* W1, const float* b1, const float* W2, const float* b2,
                       const float* W3, const float* b3, float* rgb, const float* target, uint64_t* sse_u8,
                       shacira_stream_t stream);

/* ---- fused Adam over the latent table (SURVEY section 8, row f-4) ------------------------ */
/* torch.optim.Adam semantics (L2 weight decay added to the gradient, bias correction, eps outside the sqrt) for
 * ONE float32 tensor in place; `step` is a device float counter (starts at 0) that the call advances, so the
 * launch is CUDA-graph capturable. zero_grad != 0 also clears the gradient. */
int shacira_adam_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                      float beta2, float eps, float weight_decay, float* step, int32_t zero_grad,
                      shacira_stream_t stream);

/* Same update with the gradient taken as grad + (*scale2 * scale2_mul) * grad2: the image fit adds the bit-rate
 * gradient (lambda / rows, lambda a device scalar that changes every step) to the grid gradient without a pass of
 * its own (wisp/trainers/image_trainer.py:298-319). grad2 / scale2 may be NULL. With advance == 0 the step counter
 * is left to a later shacira_multi_adam_step (extra_step), saving the one-thread launch. zero_grad != 0 clears `grad`
 * after use (the next backward then accumulates into it without a memset of its own). */
int shacira_adam_step_sum(float* param, const float* grad, const float* grad2, const float* scale2, float scale2_mul,
                          float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2, float eps,
                          float weight_decay, float* step, int32_t advance, int32_t zero_grad, shacira_stream_t stream);

/* The same with the grid gradient multiplied element-wise by grad_mul first (NULL: 1): the chain rule of a table-side
 * quantiser, i.e. d w_hat / d w of shacira_sga_quantize -- the SGA backward costs no pass of its own. */
int shacira_adam_step_sum_mul(float* param, const float* grad, const float* grad_mul, const float* grad2,
                              const float* scale2, float scale2_mul, float* exp_avg, float* exp_avg_sq, int64_t n,
                              float lr, float beta1, float beta2, float eps, float weight_decay, float* step,
                              int32_t advance, int32_t zero_grad, shacira_stream_t stream);

/* ---- stochastic Gumbel annealing (SGA): the reference's quantiser for the first `decay_period` of training -------- */
/* LatentDecoder.forward with use_sga (wisp/models/latent_decoders/basic_latent_decoder.py:183-191, torch's
 * RelaxedOneHotCategorical): w_hat = floor(w) * s_0 + (floor(w) + 1) * s_1 with (s_0, s_1) a Gumbel-softmax sample at
 * `temperature` (device float: the trainer's schedule changes it every epoch, image_trainer.py:131-133) over the
 * logits -tanh(w - floor w) / T, -tanh(floor w + 1 - w) / T. Element-wise over `count` = rows * latent_dim values.
 * uniforms [count, 2]: the U(0,1) draws (parity runs inject the reference's torch.rand); NULL = drawn in the kernel
 * from a counter-based hash of (element, *rng_step, seed), *rng_step (device uint64, may be NULL) advanced by the call.
 * w_hat feeds shacira_latent_forward* with round_flag = 0. dw (nullable) receives d w_hat / d w: the rsample
 * derivative when diff_sampling != 0, else s_0 + s_1 (straight-through floor, sample() not differentiated). */
int shacira_sga_quantize(const float* latents, const float* uniforms, int64_t count, const float* temperature,
                         int32_t diff_sampling, uint64_t seed, uint64_t* rng_step, float* w_hat, float* dw,
                         shacira_stream_t stream);

/* Adam over MANY small tensors in ONE single-CTA launch (the reference's trainer steps ~20 tensors of 1..256
 * elements: decoder MLP, latent-decoder scale/shift, density-model h/b/a; wisp/trainers/base_trainer.py:206-266
 * builds their parameter groups). Per segment the gradient is
 *     (sum_{r < grad_rows} grad[r * grad_row_stride + i]) * grad_mul * (grad_scale ? *grad_scale : 1)
 *                                                         / (grad_div ? grad_div[i / div_group] : 1)
 * which covers the chain rules of this path without extra kernels: latent-decoder scale = A * div (sum of the
 * per-level dA rows, divided by div), shift (sum of per-level rows), density parameters (lambda / rows).
 * After the update, if A_out != NULL: A_out[c * F + f] = scale[c * F + f] / div[c] for the next step's kernels
 * (`scale` must then be the `param` of one of the segments). One launch, one CTA per segment; `ticket` is a device
 * uint32 the caller zero-initialises once per optimizer (the kernel leaves it at 0), so that independent optimizers
 * may run concurrently on different streams.
 * `step` (device float) is advanced by the call, and so is `extra_step` when not NULL. At most
 * SHACIRA_MAX_ADAM_SEGS segments. */
#define SHACIRA_MAX_ADAM_SEGS 32
typedef struct {
    float* param;
    const float* grad;
    float* exp_avg;
    float* exp_avg_sq;
    const float* grad_scale; /* device scalar or NULL */
    const float* grad_div;   /* device [ceil(n / div_group)] or NULL */
    int32_t n;
    int32_t grad_rows;
    int32_t grad_row_stride;
    int32_t div_group;
    float lr;
    float weight_decay;
    float grad_mul;
    float zero_grad; /* != 0: clear the gradient rows after use (they are accumulated into by the next step) */
} shacira_adam_seg_t;
int shacira_multi_adam_step(const shacira_adam_seg_t* segs, int32_t num_segs, float beta1, float beta2, float eps,
                            float* step, float* extra_step, const float* scale, const float* div, float* A_out,
                            int32_t latent_dim, int32_t feature_dim, uint32_t* ticket, shacira_stream_t stream);

/* ---- packed exponential integration along rays (SURVEY section 8, row f-3) ----------------- */
/* What the reference's tracer calls right after the grid and its decoders
 * (wisp/tracers/packed_rf_tracer.py:136-153: spc_render.exponential_integration(color, tau, boundary, exclusive=True)
 * and spc_render.sum_reduce(transmittance, boundary); kaolin 0.13.0, absent -- published algorithm restated, parity
 * with kaolin unpinned). Samples are packed ray after ray: ray r owns [ray_start[r], ray_start[r+1]) (device int32,
 * num_rays + 1 entries; the shim derives them from the reference's boolean `boundary`).
 *   weights[i]   = exp(-sum_{j<i in ray} tau[j]) * (1 - exp(-tau[i]))
 *   ray_feats[r] = sum_i weights[i] * feats[i, :]      ray_alpha[r] = sum_i weights[i]   (may be NULL)
 * backward: grad_feats (may be NULL) and grad_tau from grad_ray_feats and, optionally, a gradient reaching the
 * per-sample weights directly (grad_weights: alpha and depth terms). num_feats in {1, 3, 4, 8}. */
int shacira_integrate_forward(const float* feats, const float* tau, const int32_t* ray_start, int32_t num_rays,
                              int32_t num_feats, float* weights, float* ray_feats, float* ray_alpha,
                              shacira_stream_t stream);
int shacira_integrate_backward(const float* feats, const float* tau, const float* weights, const int32_t* ray_start,
                               int32_t num_rays, int32_t num_feats, const float* grad_ray_feats,
                               const float* grad_weights, float* grad_feats, float* grad_tau, shacira_stream_t stream);

/* Samples inside the intersected cells: everything OctreeAS._raymarch_voxel does after the ray/cell intersection
 * (wisp/accelstructs/octree_as.py:195-228; sample_from_depth_intervals / expand_pack_boundary,
 * wisp/ops/spc/sampling.py:35-71) in one pass. Nuggets are packed ray after ray: ridx[m] (int32) and
 * depth[m] = {entry, exit}; num_samples per nugget; jitter[m, k] in [0, 1) is the reference's rand_like draw,
 * injected. Outputs for e = m * num_samples + k: ridx_out (int64, may be NULL), samples [., 3], depth_samples,
 * deltas, boundary (uint8, 1 at the first sample of every ray). depth_samples / deltas / boundary are bit-exact
 * with the reference's own functions (tests/golden/sampling_ref.npz). */
int shacira_voxel_samples(const float* origins, const float* dirs, const int32_t* ridx, const float* depth,
                          const float* jitter, int64_t num_nuggets, int32_t num_samples, int64_t* ridx_out,
                          float* samples, float* depth_samples, float* deltas, uint8_t* boundary,
                          shacira_stream_t stream);

/* Ray / occupied-cell intersections against a dense occupancy grid (res^3 uint8 cells over [-1,1]^3, cell (x,y,z) at
 * (x*res + y)*res + z): stands in for kaolin's unbatched_raytrace(..., return_depth=True, with_exit=True) as called
 * by OctreeAS.raytrace (wisp/accelstructs/octree_as.py:148-170) on the dense / pruned grid of the hash-grid NeRFs.
 * From-scratch 3D-DDA, parity with kaolin unpinned. Two calls: _count fills count[num_rays]; the caller turns the
 * counts into exclusive offsets (int64 [num_rays]) and sizes the outputs; _fill writes the nuggets packed ray after
 * ray, sorted by depth: ridx / pidx (int32 [M]) and depth [M, 2] = {entry, exit}. */
int shacira_raytrace_dense_count(const uint8_t* occupancy, int32_t res, const float* origins, const float* dirs,
                                 int32_t num_rays, int32_t* count, shacira_stream_t stream);
int shacira_raytrace_dense_fill(const uint8_t* occupancy, int32_t res, const float* origins, const float* dirs,
                                int32_t num_rays, const int64_t* offset, int32_t* ridx, int32_t* pidx, float* depth,
                                shacira_stream_t stream);

/* Occupancy pruning on the dense grid (NeuralRadianceField.prune, wisp/models/nefs/nerf.py:150-185), cell layout of
 * shacira_raytrace_dense_*. _samples: one jittered sample per cell, ((cell + jitter) / res) * 2 - 1 (jitter [res^3, 3]
 * in [0, 1), the reference's torch.rand, injected). _update: occupancy = max(density, occupancy * decay) in place and
 * mask = occupancy > min_density (uint8, the grid the ray tracer reads). The caller evaluates the density at the
 * samples in between (its own network). */
int shacira_prune_samples(int32_t res, const float* jitter, float* samples, shacira_stream_t stream);
int shacira_prune_update(int64_t cells, const float* density, float decay, float min_density, float* occupancy,
                         uint8_t* mask, shacira_stream_t stream);

/* ---- latent bitstream (host side) ---------------------------------------------------- */
/* Static arithmetic coder over dense symbol ranks 0..num_symbols-1 with 16-bit cumulative
 * frequencies cdf[num_symbols+1] (cdf[0] = 0, strictly increasing, cdf[num_symbols] = 65536).
 * Stands in for torchac.encode_float_cdf (latent_grid.py:170), whose length is all the
 * reference uses; byte parity with torchac is unpinned (package absent), round trip is exact.
 * encode returns the number of bytes written or a negative error; both run on the host. */
int64_t shacira_ac_encode(const int16_t* symbols, int64_t n, const uint32_t* cdf, int32_t num_symbols,
                          uint8_t* out, int64_t out_capacity);
int shacira_ac_decode(const uint8_t* in, int64_t nbytes, const uint32_t* cdf, int32_t num_symbols,
                      int16_t* symbols, int64_t n);

/* ---- host-buffer entry (end-to-end measurement, non-torch hosts) --------------------- */
/* One fused latent fwd+bwd step with every buffer in HOST memory (pinned or pageable):
 * copies coords, latents, grad_output, A, shift to the device, runs shacira_latent_forward
 * + shacira_latent_backward, copies feats and grad_latents back, synchronises. Device
 * scratch is cached per thread between calls. */
int shacira_latent_step_host(int32_t dim, const float* coords, int64_t n, const float* latents, int64_t table_rows,
                             const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                             int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, int32_t round_flag,
                             const float* A, const float* shift, int32_t per_level, const float* grad_output,
                             float* feats, float* grad_latents);

/* Host-buffer SESSION: the same step for a caller that runs many steps over ONE coordinate set (an image fit:
 * static coordinates, image_trainer.py:234-266), pipelined two steps deep. The coordinates and their spatial plan stay
 * on the device (set_coords: upload + binning, once); the table and decoder are uploaded when the host changed them
 * (set_table, ordered after the kernels in flight that read the old values); step_async enqueues
 *   upload(grad_output) | forward -> download(feats) | backward -> download(grad_latents, grad_A, grad_shift)
 * on three streams over two slots of device buffers and returns at once with the slot it used: the upload of step
 * i+1 and the downloads of step i use both PCIe directions at the same time. The host buffers of a slot (ideally
 * pinned) are complete after session_wait(slot) and must not be reused before. grad_A [L, C, F] / grad_shift [L, F]
 * (nullable) as in shacira_latent_backward_planned (2D tiled path; with one shared decoder only the sum over the L
 * rows is defined). */
typedef struct shacira_host_session shacira_host_session_t;
int shacira_host_session_create(int32_t dim, int64_t n, int64_t table_rows, const int32_t* first_idx,
                                const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth,
                                int32_t latent_dim, int32_t feature_dim, int32_t per_level,
                                shacira_host_session_t** session);
int shacira_host_session_destroy(shacira_host_session_t* session);
int shacira_host_session_set_coords(shacira_host_session_t* session, const float* coords);
int shacira_host_session_set_table(shacira_host_session_t* session, const float* latents, const float* A,
                                   const float* shift, int32_t round_flag);
int shacira_host_session_step_async(shacira_host_session_t* session, const float* grad_output, float* feats,
                                    float* grad_latents, float* grad_A, float* grad_shift, int32_t* slot);
int shacira_host_session_wait(shacira_host_session_t* session, int32_t slot);

/* The optimizer side of the image-fit step as ONE launch: shacira_multi_adam_step's segments (one CTA each), the latent
 * table's shacira_adam_step_sum_mul (gradient cleared after use) and -- when w_hat != NULL -- the NEXT step's SGA sample
 * of the updated latents (shacira_sga_quantize's math with the draw index *rng_step, advanced by the call; dw may be NULL).
 * Both step counters advance by one. With ent_params != NULL (latent_dim 1; grad2 must be NULL) the table pass also
 * evaluates the bit-rate loss of the latents BEFORE their update (shacira_entropy_bits' math and noise stream: ent_noise
 * [n] injected, or NULL = drawn in the kernel from (ent_seed, *ent_rng_step), advanced by the call): bits[0] = total bits,
 * the latents' bit-rate gradient goes straight into the table's Adam (scaled by *scale2 x scale2_mul), the density model's
 * gradients grad_ent_params[4][3] are reduced by the last CTA, which then runs the segments whose gradient lives there.
 * ent_scratch: at least 52 bytes per 1024 table entries. Reference: optimizer.step() over the groups of
 * base_trainer.py:206-266, latent_grid.py:122-136, and basic_latent_decoder.py:183-191 at the start of the next step. */
int shacira_fit_optimizer_step(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                               const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                               float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay, float beta1,
                               float beta2, float eps, float* step_small, float* step_table, const float* scale,
                               const float* div, float* A_out, int32_t latent_dim, int32_t feature_dim,
                               const float* temperature, int32_t diff_sampling, uint64_t seed, uint64_t* rng_step,
                               float* w_hat, float* dw, const float* ent_params, int32_t ent_layers,
                               const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step, double* bits,
                               float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes, uint32_t* ticket,
                               shacira_stream_t stream);

/* Best-state selection inside that launch (the reference's ImageTrainer keeps the state of the lowest rgb_loss and
 * reports PSNR / bpp from it, image_trainer.py:173-178,305-310,471-502). Every CTA evaluates
 * loss_t = (float)(*sse / count) -- the SSE the fit kernel wrote for this step's parameters, count = n x 3 -- and, when
 * loss_t < *best_loss (strict: the first minimum wins, NaN never), stores the PRE-update values of the parameters it
 * owns: the latent table into `table`, segment i's param into seg_param[i] (NULL: not stored), div [latent_dim] and
 * A [latent_dim * feature_dim] (the A this step's forward used) by the CTA of the `scale` segment. Only the last CTA
 * writes *best_loss / *best_step (the step index: *step_small before the call advances it), after every CTA has
 * evaluated the predicate. Initialise *best_loss to +inf. */
typedef struct {
    const double* sse;
    int64_t count;
    float* best_loss;
    int64_t* best_step;
    float* table;
    float* seg_param[SHACIRA_MAX_ADAM_SEGS];
    float* div;
    float* A;
} shacira_fit_snapshot_t;
/* shacira_fit_optimizer_step with the snapshot above (snap != NULL). */
int shacira_fit_optimizer_step_best(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                                    const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                                    float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay,
                                    float beta1, float beta2, float eps, float* step_small, float* step_table,
                                    const float* scale, const float* div, float* A_out, int32_t latent_dim,
                                    int32_t feature_dim, const float* temperature, int32_t diff_sampling, uint64_t seed,
                                    uint64_t* rng_step, float* w_hat, float* dw, const float* ent_params,
                                    int32_t ent_layers, const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step,
                                    double* bits, float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes,
                                    uint32_t* ticket, const shacira_fit_snapshot_t* snap, shacira_stream_t stream);

/* The trainer's schedules advanced by that launch (image_trainer.py:113-193; utils/schedulers.py). Before step `it`
 * (0-based, = *step_small):
 *   lambda(it) = lambda_end + 0.5 * (lambda_start - lambda_end) * (1 + cos(pi * it / num_epochs))   (COSINE)
 *              = lambda_start                                                                      (FIX)
 *   T(it)      = max(temperature_end, exp(-ln(1 / temperature_end) * (it + 1) / num_epochs / decay_period))
 * evaluated in double and rounded to float. */
#define SHACIRA_LAMBDA_FIX 0
#define SHACIRA_LAMBDA_COSINE 1
typedef struct {
    int32_t num_epochs;          /* >= 1 */
    int32_t lambda_kind;         /* SHACIRA_LAMBDA_COSINE or SHACIRA_LAMBDA_FIX */
    double lambda_start, lambda_end;
    double temperature_end;      /* > 0 */
    double decay_period;         /* in (0, 1] */
    const double* sse;           /* this step's rgb_loss = (float)(*sse / count), as for the snapshot */
    int64_t count;
    float* log;                  /* [log_capacity][4]: rgb_loss, total bits (NaN without bits), lambda, temperature */
    int64_t log_capacity;
} shacira_fit_schedule_t;
/* shacira_fit_optimizer_step(_best) (snap may be NULL) that also advances the schedule: the last CTA appends record
 * *step_small to sched->log (dropped when it is >= log_capacity) -- the step's rgb_loss, (float)bits[0] (the folded
 * bit-rate loss of this launch, or what shacira_entropy_bits wrote before it), and the lambda (*scale2) and temperature
 * (*temperature) the step used -- and then writes lambda(it + 1) into *scale2 and T(it + 1) into *temperature. Every
 * reader of those scalars in the launch reads them first; the next step's SGA sample, drawn here, uses T(it). scale2
 * and temperature must not be NULL. */
int shacira_fit_optimizer_step_sched(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                                     const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                                     float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay,
                                     float beta1, float beta2, float eps, float* step_small, float* step_table,
                                     const float* scale, const float* div, float* A_out, int32_t latent_dim,
                                     int32_t feature_dim, const float* temperature, int32_t diff_sampling, uint64_t seed,
                                     uint64_t* rng_step, float* w_hat, float* dw, const float* ent_params,
                                     int32_t ent_layers, const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step,
                                     double* bits, float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes,
                                     uint32_t* ticket, const shacira_fit_snapshot_t* snap,
                                     const shacira_fit_schedule_t* sched, shacira_stream_t stream);

/* ---- exchange step of the ray-batch data-parallel path over NVLink / NVSwitch peer memory (SURVEY 8e) ------------
 * north_star: "NeRF ray batches are data-parallel, with the hash-table/latent gradient allreduced ... over NVLink".
 * The reference is single-GPU (no counterpart file); the NCCL form is shacira_b200.dp.GradArena.allreduce.
 * One process per GPU. Every rank allocates its gradient arena with shacira_peer_alloc (cudaMalloc: bytes rounded up to
 * 256 + a 256-byte flag block at shacira_peer_flags_offset(bytes), all zero), exports it (64-byte CUDA IPC handle,
 * exchanged by the host: torch.distributed.all_gather_object in shacira_b200/peer.py) and maps every other rank's
 * arena with shacira_peer_open. Inside ONE process that drives several GPUs the pointers are used directly after
 * shacira_peer_enable_access. */
int64_t shacira_peer_flags_offset(int64_t bytes);
int shacira_peer_alloc(int64_t bytes, void** ptr);
int shacira_peer_free(void* ptr);
int shacira_peer_export(void* ptr, void* handle64);
int shacira_peer_open(const void* handle64, void** ptr);
int shacira_peer_close(void* ptr);
int shacira_peer_enable_access(int32_t device, int32_t peer_device);
/* SUM all-reduce of `numel` floats (multiple of 4) in place over `world` in {2, 4, 8} arenas: bufs[p] = rank p's arena as
 * mapped into this process (bufs[rank] = the local one). ONE kernel per rank: cross-GPU barrier, rank r reduces slice r
 * from all arenas in rank order and stores the sum into all arenas, cross-GPU barrier. Every rank must make the same
 * sequence of calls; the result is bit-identical on all ranks. Stream-ordered and CUDA-graph capturable (the barrier
 * epoch lives on the device). */
int shacira_peer_allreduce(void* const* bufs, int64_t flags_offset, int32_t rank, int32_t world, int64_t numel,
                           shacira_stream_t stream);
/* The cross-GPU barriers give up after ~4 s of polling (a peer that died must not hang this GPU) and raise an error word
 * in the local flag block: *timed_out = 1 if any exchange on `buf` (the LOCAL arena / flag buffer) has timed out since it
 * was allocated. Synchronises the device. */
int shacira_peer_status(const void* buf, int64_t flags_offset, int32_t* timed_out);
/* The same pass with the latent table's Adam step inside (reduce-scatter + sharded optimizer state + all-gather): the
 * first `table_numel` floats of the arena are the table's gradient; the owner of a slice applies torch.optim.Adam's
 * update to params[rank] there (exp_avg / exp_avg_sq: this rank's slice-sized state, passed as pointers already offset
 * so that element i of the table is exp_avg[i]; `step` = device float, steps taken so far, advanced by the caller),
 * stores the updated parameters into every rank's table params[p] and clears the gradient slots. The rest of the arena
 * (decoder / density-model gradients) is all-reduced as above. */
int shacira_peer_allreduce_adam(void* const* bufs, int64_t flags_offset, int32_t rank, int32_t world, int64_t numel,
                                void* const* params, int64_t table_numel, float* exp_avg, float* exp_avg_sq,
                                const float* step, float lr, float beta1, float beta2, float eps, float weight_decay,
                                shacira_stream_t stream);

/* The all-reduce through the NVSwitch multicast object (NVLS): `multicast_ptr` = multicast address of the arena (every
 * rank's copy bound to one CUDA multicast object; shacira_b200/peer.py maps it with torch's symmetric-memory allocator),
 * flag_bufs[p] + flags_offset = rank p's 256-byte flag block in plain peer memory (a shacira_peer_alloc buffer). The sum
 * is formed inside the switch (multimem.ld_reduce) and stored to all copies (multimem.st): one arena's worth of bytes per
 * GPU and direction instead of 2 (N-1)/N. Same call discipline as shacira_peer_allreduce. */
int shacira_peer_allreduce_multimem(void* multicast_ptr, void* const* flag_bufs, int64_t flags_offset, int32_t rank,
                                    int32_t world, int64_t numel, shacira_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SHACIRA_B200_H_ */
