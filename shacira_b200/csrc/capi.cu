// capi.cu -- the extern "C" surface declared in include/shacira_b200.h: argument validation,
// level metadata, template dispatch and launches. No torch, no exceptions across the ABI.

#include "arith_coder.inl"
#include "capi_internal.h"
#include "coarse_kernels.cuh"
#include "entropy_kernels.cuh"
#include "hashgrid_kernels.cuh"
#include "mlp_kernels.cuh"
#include "render_kernels.cuh"
#include "sga_kernels.cuh"
#include "optimizer_kernels.cuh"

using namespace shacira;

namespace shacira {

char* last_error_buffer() {
    thread_local char buf[512] = "";
    return buf;
}
std::atomic<int64_t>& launch_counter() {
    static std::atomic<int64_t> c{0};
    return c;
}

int build_levels(int32_t dim, const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                 int32_t bitwidth, LevelParams& lp) {
    if (dim != 2 && dim != 3) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "dim must be 2 or 3, got %d", dim);
    if (!resolutions) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "resolutions is NULL");
    if (num_lods < 1 || num_lods > SHACIRA_MAX_LEVELS)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "num_lods must be in [1, %d], got %d", SHACIRA_MAX_LEVELS, num_lods);
    if (bitwidth < 1 || bitwidth > 30)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "codebook_bitwidth must be in [1, 30], got %d", bitwidth);
    memset(&lp, 0, sizeof(lp));
    const int64_t T = (int64_t)1 << bitwidth;
    lp.num_lods = num_lods;
    lp.hash_mask = (uint32_t)(T - 1);
    int64_t running = 0;
    for (int l = 0; l < num_lods; ++l) {
        const int64_t r = resolutions[l];
        if (r < 2 || r > (1 << 22))
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "resolution[%d] = %lld out of range [2, 2^22]", l, (long long)r);
        // the reference's predicate, with its int32 wrap-around (hashgrid_interpolate_cuda.cu:27-29)
        const int32_t r32 = (int32_t)r;
        const int32_t rr32 = (int32_t)((uint32_t)r32 * (uint32_t)r32);
        const int32_t rrr32 = (int32_t)((uint32_t)rr32 * (uint32_t)r32);
        const bool ref_dense = r32 < T && rr32 < T && (dim == 2 || rrr32 < T);
        // the same predicate in 64-bit
        const int64_t pts = (dim == 2) ? r * r : r * r * r;
        const bool dense = r < T && r * r < T && pts < T;
        if (ref_dense != dense)
            return fail(SHACIRA_ERR_Q2_WINDOW,
                        "level %d (res %lld, 2^%d rows): the reference's int32 dense predicate overflows here and "
                        "indexes outside the table; parity is undefined (SURVEY Q2)", l, (long long)r, bitwidth);
        if (dense) lp.dense_mask |= (1u << l);
        lp.res[l] = r32;
        lp.resd[l] = (double)r32;
        lp.rows[l] = (int32_t)(pts < T ? pts : T);
        lp.hi[l] = (float)((double)(r32 - 1) - 1e-5);
        lp.first[l] = first_idx ? first_idx[l] : (int32_t)running;
        if (lp.first[l] < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "first_idx[%d] is negative", l);
        running += lp.rows[l];
    }
    return SHACIRA_OK;
}

int check_points(const float* coords, int64_t n) {
    if (n < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "n is negative");
    if (n > 0 && !coords) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "coords is NULL");
    if (n > ((int64_t)1 << 31) * (int64_t)kBlock / 2) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "n too large");
    return SHACIRA_OK;
}

}  // namespace shacira

namespace {

inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

template <int D, int F>
int launch_plain_fwd(const float* coords, int64_t n, const float* table, const LevelParams& lp, float* feats,
                     cudaStream_t s) {
    if (D == 3 && grid3d_supported(F, F, table))   // lane pairs, identity decoder
        return launch_fwd3d(F, F, coords, nullptr, n, table, lp, nullptr, nullptr, 0, 0, feats, nullptr, s);
    hashgrid_fwd_kernel<D, F><<<grid_for(n, kBlock), kBlock, 0, s>>>(coords, n, table, lp, feats);
    LAUNCHED();
    return SHACIRA_OK;
}
// Coarse dense levels go through shared memory (coarse_kernels.cuh) when the batch is large enough for their
// same-address global adds to serialise. One slab per level: measured at the NeRF shape, whole-level jobs pay,
// slabbed levels do not.
constexpr int kCoarseMaxSlabs = 1;
inline int join_side(cudaStream_t s) {
    SideStream* ss = nullptr;
    if (int rc = side_stream(&ss)) return rc;
    CUDA_OK(cudaStreamWaitEvent(s, ss->join, 0));
    return SHACIRA_OK;
}
template <int D, int C, int F, bool LATENT>
int launch_coarse_bwd(const float* coords, int64_t n, const float* g, const LevelParams& lp, const float* A,
                      int per_level, float* gt, cudaStream_t s, uint32_t& mask, bool& pending_join,
                      uint32_t level_mask = 0xffffffffu) {
    mask = 0;
    pending_join = false;
    if (n < 65536) return SHACIRA_OK;
    CoarseJobs jobs;
    constexpr int NV = LATENT ? C : F;
    const uint32_t m = plan_coarse_jobs(D, lp, NV, n, sm_count(), kCoarseMaxSlabs, jobs, level_mask);
    if (!m) return SHACIRA_OK;
    const size_t smem = coarse_smem_bytes(jobs, NV);
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(coarse_bwd_kernel<D, C, F, LATENT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(sizeof(float) * kCoarseBudgetFloats)));
    // The coarse kernel is bound by shared-memory CAS, the point-parallel kernel by L2 atomics: fork a side stream so
    // that both run at once (one coarse CTA per SM is placed first, the other kernel fills the rest of the SM).
    // Event fork/join composes with stream capture (the side stream joins the caller's capture).
    SideStream* ssp = nullptr;
    if (int rc = side_stream(&ssp)) return rc;
    SideStream& ss = *ssp;
    CUDA_OK(cudaEventRecord(ss.fork, s));
    CUDA_OK(cudaStreamWaitEvent(ss.stream, ss.fork, 0));
    coarse_bwd_kernel<D, C, F, LATENT><<<coarse_total_ctas(jobs), kCoarseThreads, smem, ss.stream>>>(
        coords, n, g, lp, jobs, A, per_level, gt);
    LAUNCHED();
    CUDA_OK(cudaEventRecord(ss.join, ss.stream));
    pending_join = true;
    mask = m;
    return SHACIRA_OK;
}
template <int D, int F>
int launch_plain_bwd(const float* coords, int64_t n, const float* g, const LevelParams& lp, float* gt,
                     cudaStream_t s) {
    uint32_t skip = 0;
    bool join = false;
    int rc = launch_coarse_bwd<D, F, F, false>(coords, n, g, lp, nullptr, 0, gt, s, skip, join);
    if (rc) return rc;
    if (D == 3 && grid3d_supported(F, F, gt)) {   // lane pairs, identity decoder
        rc = launch_bwd3d(F, F, coords, nullptr, n, g, nullptr, lp, nullptr, 0, skip, 0xffffffffu, gt, nullptr, nullptr, s);
        if (rc) return rc;
        return join ? join_side(s) : SHACIRA_OK;
    }
    hashgrid_bwd_kernel<D, F><<<grid_for(n, kBlock), kBlock, 0, s>>>(coords, n, g, lp, skip, gt);
    LAUNCHED();
    return join ? join_side(s) : SHACIRA_OK;
}
template <int D, int C, int F>
int launch_latent_fwd(const float* coords, int64_t n, const float* lat, const LevelParams& lp, const float* A,
                      const float* shift, int per_level, int round_flag, float* feats, float* zsave,
                      cudaStream_t s) {
    if (D == 3 && grid3d_supported(C, F, lat))   // lane pairs (grid3d_kernels.cuh)
        return launch_fwd3d(C, F, coords, nullptr, n, lat, lp, A, shift, per_level, round_flag, feats, zsave, s);
    const int nA = per_level ? lp.num_lods : 1;
    const size_t smem = sizeof(float) * (size_t)(nA * C * F + nA * F);
    latent_fwd_kernel<D, C, F><<<grid_for(n, kBlock), kBlock, smem, s>>>(coords, n, lat, lp, A, shift, per_level,
                                                                          round_flag, feats, zsave);
    LAUNCHED();
    return SHACIRA_OK;
}
template <int D, int C, int F>
int launch_latent_bwd(const float* coords, int64_t n, const float* g, const float* zsave, const LevelParams& lp,
                      const float* A, int per_level, float* gl, float* gA, float* gS, cudaStream_t s,
                      uint32_t level_mask = 0xffffffffu) {
    const int nA = per_level ? lp.num_lods : 1;
    const size_t smem = sizeof(float) * (size_t)(nA * C * F + lp.num_lods * C * F + lp.num_lods * F);
    uint32_t skip = 0;
    bool join = false;
    int rc = launch_coarse_bwd<D, C, F, true>(coords, n, g, lp, A, per_level, gl, s, skip, join, level_mask);
    if (rc) return rc;
    if (D == 3 && grid3d_supported(C, F, gl)) {   // lane pairs (grid3d_kernels.cuh)
        rc = launch_bwd3d(C, F, coords, nullptr, n, g, zsave, lp, A, per_level, skip, level_mask, gl, gA, gS, s);
        if (rc) return rc;
        return join ? join_side(s) : SHACIRA_OK;
    }
    latent_bwd_kernel<D, C, F><<<grid_for(n, kBlock), kBlock, smem, s>>>(coords, n, g, zsave, lp, A, per_level, skip,
                                                                          level_mask, gl, gA, gS);
    LAUNCHED();
    return join ? join_side(s) : SHACIRA_OK;
}

#define DISPATCH_F(D_, F_, CALL)                                                                   \
    switch (F_) {                                                                                  \
        case 1: { constexpr int kF = 1; return CALL; }                                             \
        case 2: { constexpr int kF = 2; return CALL; }                                             \
        case 4: { constexpr int kF = 4; return CALL; }                                             \
        case 8: { constexpr int kF = 8; return CALL; }                                             \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "feature_dim %d not in {1,2,4,8}", (int)F_); \
    }

#define DISPATCH_CF(C_, F_, CALL)                                                                        \
    switch (C_) {                                                                                        \
        case 1: { constexpr int kC = 1; DISPATCH_F(0, F_, CALL) }                                        \
        case 2: { constexpr int kC = 2; DISPATCH_F(0, F_, CALL) }                                        \
        case 4: { constexpr int kC = 4; DISPATCH_F(0, F_, CALL) }                                        \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d not in {1,2,4}", (int)C_);          \
    }

}  // namespace

namespace {
// IN = 16 on the tensor cores (mlp16_tc_step_kernel: mma.sync TF32 with 3xTF32 compensation). Two m16 tiles per warp
// iteration, 6 warps x 2 CTAs per SM: the configuration chosen by measurement (mlp_kernels.cuh).
int launch_mlp_tc(const float* x, const float* gt, int64_t n, const float* W1, const float* b1, const float* W2,
                  const float* b2, const float* W3, const float* b3, float* gx, float* pred, void* out, float* absmax,
                  cudaStream_t s) {
    constexpr int MT = 2, WARPS = 6, MINB = 2;
    using Smem = MlpTcSmem<MT, WARPS>;
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(mlp16_tc_step_kernel<MT, WARPS, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)sizeof(Smem)));
    const size_t out_bytes = 8 + sizeof(float) * kMlp16Params;
    if (absmax && (char*)absmax == (char*)out + out_bytes) {   // caller keeps the bound behind `out`: one memset node
        CUDA_OK(cudaMemsetAsync(out, 0, out_bytes + sizeof(float) * 16, s));
    } else {
        CUDA_OK(cudaMemsetAsync(out, 0, out_bytes, s));
        if (absmax) CUDA_OK(cudaMemsetAsync(absmax, 0, sizeof(float) * 16, s));
    }
    const int64_t groups = (n + 16 * MT - 1) / (16 * MT);
    int64_t blocks = (groups + WARPS - 1) / WARPS;
    const int64_t cap = (int64_t)sm_count() * MINB;  // persistent CTAs
    if (blocks > cap) blocks = cap;
    const float scale = (float)(2.0 / ((double)n * 3.0));
    mlp16_tc_step_kernel<MT, WARPS, MINB><<<(int)blocks, WARPS * 32, sizeof(Smem), s>>>(
        x, gt, n, W1, b1, W2, b2, W3, b3, scale, gx, pred, (double*)out, (float*)((char*)out + 8), (unsigned*)absmax);
    LAUNCHED();
    return SHACIRA_OK;
}

template <int IN>
int launch_mlp(const float* x, const float* gt, int64_t n, const float* W1, const float* b1, const float* W2,
               const float* b2, const float* W3, const float* b3, float* gx, float* pred, void* out, cudaStream_t s) {
    using Smem = MlpSmem<IN, 16, 3>;
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(mlp_mse_step_kernel<IN, 16, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)sizeof(Smem)));
    const int sms = sm_count();
    const size_t out_bytes = 8 + sizeof(float) * (16 * IN + 16 + 16 * 16 + 16 + 3 * 16 + 3);
    CUDA_OK(cudaMemsetAsync(out, 0, out_bytes, s));
    int64_t warps = (n + 31) / 32;
    int64_t blocks = (warps + kMlpWarps - 1) / kMlpWarps;
    const int64_t cap = (int64_t)sms * 2;  // persistent: 2 CTAs per SM fit the shared memory
    if (blocks > cap) blocks = cap;
    const float scale = (float)(2.0 / ((double)n * 3.0));
    mlp_mse_step_kernel<IN, 16, 3><<<(int)blocks, kMlpThreads, sizeof(Smem), s>>>(
        x, gt, n, W1, b1, W2, b2, W3, b3, scale, gx, pred, (double*)out, (float*)((char*)out + 8));
    LAUNCHED();
    return SHACIRA_OK;
}
}  // namespace


extern "C" {

int shacira_abi_version(void) { return SHACIRA_ABI_VERSION; }
const char* shacira_last_error(void) { return last_error_buffer(); }
int64_t shacira_launch_count(void) { return launch_counter().load(); }

int shacira_device_info(int32_t* sm_count, int64_t* l2_bytes, int64_t* l2_persist_max) {
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    CUDA_OK(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (l2_bytes) *l2_bytes = p.l2CacheSize;
    if (l2_persist_max) *l2_persist_max = p.persistingL2CacheMaxSize;
    return SHACIRA_OK;
}

int shacira_l2_pin(const void* base, int64_t bytes, shacira_stream_t stream) {
    cudaStream_t s = (cudaStream_t)stream;
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    CUDA_OK(cudaGetDeviceProperties(&p, dev));
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (bytes > 0 && base) {
        size_t carve = (size_t)p.persistingL2CacheMaxSize;
        if ((size_t)bytes < carve) carve = (size_t)bytes;
        CUDA_OK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
        size_t win = (size_t)bytes;
        if (win > (size_t)p.accessPolicyMaxWindowSize) win = (size_t)p.accessPolicyMaxWindowSize;
        attr.accessPolicyWindow.base_ptr = const_cast<void*>(base);
        attr.accessPolicyWindow.num_bytes = win;
        attr.accessPolicyWindow.hitRatio = win <= carve ? 1.0f : (float)carve / (float)win;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    } else {
        attr.accessPolicyWindow.num_bytes = 0;
    }
    CUDA_OK(cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &attr));
    if (!(bytes > 0 && base)) {
        // clearing: give the carve-out back as well (measured: a 24 MB carve-out left behind costs an unpinned 3D step 13 %)
        CUDA_OK(cudaCtxResetPersistingL2Cache());
        CUDA_OK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0));
    }
    return SHACIRA_OK;
}

int shacira_hashgrid_forward(int32_t dim, const float* coords, int64_t n, const float* codebook,
                             const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                             int32_t codebook_bitwidth, int32_t feature_dim, float* feats, shacira_stream_t stream) {
    LevelParams lp;
    int rc = build_levels(dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if ((rc = check_points(coords, n))) return rc;
    if (n == 0) return SHACIRA_OK;
    if (!codebook || !feats) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "codebook/feats is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (dim == 2) { DISPATCH_F(2, feature_dim, (launch_plain_fwd<2, kF>(coords, n, codebook, lp, feats, s))) }
    DISPATCH_F(3, feature_dim, (launch_plain_fwd<3, kF>(coords, n, codebook, lp, feats, s)))
}

int shacira_hashgrid_backward(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                              const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                              int32_t codebook_bitwidth, int32_t feature_dim, int64_t table_rows, int32_t zero_first,
                              float* grad_codebook, shacira_stream_t stream) {
    LevelParams lp;
    int rc = build_levels(dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if ((rc = check_points(coords, n))) return rc;
    if (!grad_codebook) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_codebook is NULL");
    if ((rc = check_table(lp, table_rows))) return rc;
    if (feature_dim != 1 && feature_dim != 2 && feature_dim != 4 && feature_dim != 8)
        return fail(SHACIRA_ERR_UNSUPPORTED, "feature_dim %d not in {1,2,4,8}", feature_dim);
    cudaStream_t s = (cudaStream_t)stream;
    if (zero_first) CUDA_OK(cudaMemsetAsync(grad_codebook, 0, sizeof(float) * (size_t)table_rows * feature_dim, s));
    if (n == 0) return SHACIRA_OK;
    if (!grad_output) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_output is NULL");
    if (dim == 2) { DISPATCH_F(2, feature_dim, (launch_plain_bwd<2, kF>(coords, n, grad_output, lp, grad_codebook, s))) }
    DISPATCH_F(3, feature_dim, (launch_plain_bwd<3, kF>(coords, n, grad_output, lp, grad_codebook, s)))
}

int shacira_hashgrid_corners(int32_t dim, const float* coords, int64_t n, const int32_t* resolutions,
                             int32_t num_lods, int32_t codebook_bitwidth, int32_t* idx, float* w,
                             shacira_stream_t stream) {
    LevelParams lp;
    int rc = build_levels(dim, nullptr, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if ((rc = check_points(coords, n))) return rc;
    if (n == 0) return SHACIRA_OK;
    if (!idx || !w) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "idx/w is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (dim == 2) corners_kernel<2><<<grid_for(n, kBlock), kBlock, 0, s>>>(coords, n, lp, idx, w);
    else corners_kernel<3><<<grid_for(n, kBlock), kBlock, 0, s>>>(coords, n, lp, idx, w);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_latent_forward(int32_t dim, const float* coords, int64_t n, const float* latents,
                           const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                           int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, int32_t round_flag,
                           const float* A, const float* shift, int32_t per_level, float* feats, float* zsave,
                           shacira_stream_t stream) {
    LevelParams lp;
    int rc = build_levels(dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if ((rc = check_points(coords, n))) return rc;
    if (n == 0) return SHACIRA_OK;
    if (!latents || !feats || !A) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/feats/A is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (dim == 2) {
        DISPATCH_CF(latent_dim, feature_dim,
                    (launch_latent_fwd<2, kC, kF>(coords, n, latents, lp, A, shift, per_level, round_flag, feats,
                                                  zsave, s)))
    }
    DISPATCH_CF(latent_dim, feature_dim,
                (launch_latent_fwd<3, kC, kF>(coords, n, latents, lp, A, shift, per_level, round_flag, feats, zsave,
                                              s)))
}

int shacira_latent_backward_levels(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                                   const float* zsave, const int32_t* first_idx, const int32_t* resolutions,
                                   int32_t num_lods, int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                                   const float* A, int32_t per_level, int64_t table_rows, int32_t zero_first,
                                   uint32_t level_mask, float* grad_latents, float* grad_A, float* grad_shift,
                                   shacira_stream_t stream) {
    LevelParams lp;
    int rc = build_levels(dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if ((rc = check_points(coords, n))) return rc;
    if (!grad_latents || !A) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_latents/A is NULL");
    if ((rc = check_table(lp, table_rows))) return rc;
    if (grad_A && !zsave) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_A requested without zsave");
    if (latent_dim != 1 && latent_dim != 2 && latent_dim != 4)
        return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d not in {1,2,4}", latent_dim);
    cudaStream_t s = (cudaStream_t)stream;
    if (zero_first) CUDA_OK(cudaMemsetAsync(grad_latents, 0, sizeof(float) * (size_t)table_rows * latent_dim, s));
    if (n == 0) return SHACIRA_OK;
    if (!grad_output) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_output is NULL");
    if (dim == 2) {
        DISPATCH_CF(latent_dim, feature_dim,
                    (launch_latent_bwd<2, kC, kF>(coords, n, grad_output, zsave, lp, A, per_level, grad_latents,
                                                  grad_A, grad_shift, s, level_mask)))
    }
    DISPATCH_CF(latent_dim, feature_dim,
                (launch_latent_bwd<3, kC, kF>(coords, n, grad_output, zsave, lp, A, per_level, grad_latents, grad_A,
                                              grad_shift, s, level_mask)))
}

int shacira_latent_backward(int32_t dim, const float* coords, int64_t n, const float* grad_output,
                            const float* zsave, const int32_t* first_idx, const int32_t* resolutions,
                            int32_t num_lods, int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                            const float* A, int32_t per_level, int64_t table_rows, int32_t zero_first,
                            float* grad_latents, float* grad_A, float* grad_shift, shacira_stream_t stream) {
    return shacira_latent_backward_levels(dim, coords, n, grad_output, zsave, first_idx, resolutions, num_lods,
                                          codebook_bitwidth, latent_dim, feature_dim, A, per_level, table_rows,
                                          zero_first, 0xffffffffu, grad_latents, grad_A, grad_shift, stream);
}

static int entropy_bits_impl(const float* latents, const float* noise, int64_t table_rows, int32_t latent_dim,
                             const float* params, int32_t num_layers, const int32_t* first_idx, int32_t num_lods,
                             double* bits, float* grad_latents, float* grad_params, void* scratch,
                             int64_t scratch_bytes, uint64_t rng_seed, uint64_t* rng_step, shacira_stream_t stream) {
    if (!latents || !params || !bits) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/params/bits is NULL");
    if (table_rows < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "table_rows is negative");
    if (latent_dim < 1 || latent_dim > kMaxEntC || (latent_dim & (latent_dim - 1)))
        return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d must be a power of two <= %d", latent_dim, kMaxEntC);
    if (num_layers < 1) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "num_layers must be >= 1");
    if (num_lods < 0 || num_lods > SHACIRA_MAX_LEVELS || (num_lods > 0 && !first_idx))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "bad num_lods/first_idx");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t total = table_rows * latent_dim;
    if (total == 0) {
        CUDA_OK(cudaMemsetAsync(bits, 0, sizeof(double) * (size_t)(1 + num_lods), s));
        if (grad_params) CUDA_OK(cudaMemsetAsync(grad_params, 0, sizeof(float) * 12 * (size_t)latent_dim, s));
        return SHACIRA_OK;
    }
    LevelBounds lb;
    memset(&lb, 0, sizeof(lb));
    lb.num_lods = num_lods;
    for (int l = 0; l < num_lods; ++l) lb.first[l] = first_idx[l];
    lb.first[num_lods] = (int32_t)table_rows;
    const int sms = sm_count();
    int64_t blocks = (total + kEntBlock - 1) / kEntBlock;
    const int64_t cap = (int64_t)sms * 4;  // per-block prologue/epilogue (~500 instructions) vs parallelism: tuned on B200
    if (blocks > cap) blocks = cap;
    // scratch: [0, 256) arrival ticket, then the block partials. The ticket sits at a FIXED offset: one scratch serves
    // launches of any table size (a ticket behind the partials would be overwritten by a larger launch's rows). The
    // caller's scratch is zero-initialised once and reusable (the kernel leaves the ticket at 0); without one, a
    // stream-ordered pool allocation (3 more graph nodes per call)
    const int P = 1 + num_lods + 12 * latent_dim;
    const size_t part_bytes = ((sizeof(float) * (size_t)blocks * P) + 255) & ~(size_t)255;
    char* buf = (char*)scratch;
    const bool own = !buf || (size_t)scratch_bytes < part_bytes + 256;
    if (own) {
        buf = nullptr;
        CUDA_OK(cudaMallocAsync((void**)&buf, part_bytes + 256, s));
        CUDA_OK(cudaMemsetAsync(buf, 0, sizeof(unsigned), s));
    }
    unsigned* ticket = (unsigned*)buf;
    // validation mode (x = round(w)): per-integer table in shared memory instead of per-element CDF chains
    const bool val_mode = !noise && !rng_step;
    // (pays from ~1 M entries: every CTA builds the table first -- measured 22.9 vs 17.1 us at the image table's 375 k,
    // 51.6 vs 85.7 us at the NeRF table's 6.1 M with per-level sums)
    if (val_mode && latent_dim <= 4 && total >= (1 << 20)) {
        const size_t lut_bytes = sizeof(float) * (size_t)latent_dim * kLutK * kLutN;
        if (lut_bytes > 48 * 1024) {
            static unsigned long long configured = 0ull;
            if (needs_config(configured))
                CUDA_OK(cudaFuncSetAttribute(entropy_val_lut_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        }
        int64_t per_block = (total + blocks - 1) / blocks;
        per_block = (per_block + kEntBlock - 1) / kEntBlock * kEntBlock;   // multiple of 256 (and hence of latent_dim)
        entropy_val_lut_kernel<<<(int)blocks, kEntBlock, lut_bytes, s>>>(latents, total, latent_dim, params, num_layers, lb,
                                                                         bits, grad_latents, grad_params,
                                                                         (float*)(buf + 256), ticket, per_block);
    } else {
        entropy_kernel<<<(int)blocks, kEntBlock, 0, s>>>(latents, noise, total, latent_dim, params, num_layers, lb, bits,
                                                         grad_latents, grad_params, (float*)(buf + 256), ticket,
                                                         (unsigned long long)rng_seed, (unsigned long long*)rng_step);
    }
    launch_counter().fetch_add(1);
    const cudaError_t le = cudaGetLastError();
    if (own) cudaFreeAsync(buf, s);
    if (le != cudaSuccess) return fail(SHACIRA_ERR_CUDA, "entropy launch: %s", cudaGetErrorString(le));
    return SHACIRA_OK;
}

int shacira_entropy_bits(const float* latents, const float* noise, int64_t table_rows, int32_t latent_dim,
                         const float* params, int32_t num_layers, const int32_t* first_idx, int32_t num_lods,
                         double* bits, float* grad_latents, float* grad_params, void* scratch, int64_t scratch_bytes,
                         shacira_stream_t stream) {
    return entropy_bits_impl(latents, noise, table_rows, latent_dim, params, num_layers, first_idx, num_lods, bits,
                             grad_latents, grad_params, scratch, scratch_bytes, 0, nullptr, stream);
}

int shacira_entropy_bits_rng(const float* latents, uint64_t seed, uint64_t* rng_step, int64_t table_rows,
                             int32_t latent_dim, const float* params, int32_t num_layers, const int32_t* first_idx,
                             int32_t num_lods, double* bits, float* grad_latents, float* grad_params, void* scratch,
                             int64_t scratch_bytes, shacira_stream_t stream) {
    if (!rng_step) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "entropy_bits_rng: rng_step is NULL");
    if (!scratch) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "entropy_bits_rng: needs the caller's scratch");
    return entropy_bits_impl(latents, nullptr, table_rows, latent_dim, params, num_layers, first_idx, num_lods, bits,
                             grad_latents, grad_params, scratch, scratch_bytes, seed, rng_step, stream);
}

int64_t shacira_entropy_scratch_bytes(int32_t latent_dim, int32_t num_lods) {
    const int64_t blocks = (int64_t)sm_count() * 8;  // upper bound of the launch grid
    const int64_t P = 1 + num_lods + 12 * (int64_t)latent_dim;
    return ((4 * blocks * P + 255) & ~(int64_t)255) + 256;
}

int shacira_adam_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                      float beta2, float eps, float weight_decay, float* step, int32_t zero_grad,
                      shacira_stream_t stream) {
    if (!param || !grad || !exp_avg || !exp_avg_sq || !step) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "adam_step: NULL argument");
    if (n <= 0) return SHACIRA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t blocks = (n + 1023) / 1024;
    adam_step_kernel<<<(int)blocks, 256, 0, s>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                                                 step, zero_grad, grad);
    LAUNCHED();
    adam_advance_kernel<<<1, 1, 0, s>>>(step);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_adam_step_sum(float* param, const float* grad, const float* grad2, const float* scale2, float scale2_mul,
                          float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2, float eps,
                          float weight_decay, float* step, int32_t advance, int32_t zero_grad, shacira_stream_t stream) {
    return shacira_adam_step_sum_mul(param, grad, nullptr, grad2, scale2, scale2_mul, exp_avg, exp_avg_sq, n, lr, beta1,
                                     beta2, eps, weight_decay, step, advance, zero_grad, stream);
}

int shacira_adam_step_sum_mul(float* param, const float* grad, const float* grad_mul, const float* grad2,
                              const float* scale2, float scale2_mul, float* exp_avg, float* exp_avg_sq, int64_t n,
                              float lr, float beta1, float beta2, float eps, float weight_decay, float* step,
                              int32_t advance, int32_t zero_grad, shacira_stream_t stream) {
    if (!param || !grad || !exp_avg || !exp_avg_sq || !step)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "adam_step_sum: NULL argument");
    if (n <= 0) return SHACIRA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t blocks = (n + 1023) / 1024;
    adam_step_sum_kernel<<<(int)blocks, 256, 0, s>>>(param, grad, grad_mul, grad2, scale2, scale2_mul, exp_avg, exp_avg_sq,
                                                     n, lr, beta1, beta2, eps, weight_decay, step, zero_grad);
    LAUNCHED();
    if (advance) {
        adam_advance_kernel<<<1, 1, 0, s>>>(step);
        LAUNCHED();
    }
    return SHACIRA_OK;
}

int shacira_sga_quantize(const float* latents, const float* uniforms, int64_t count, const float* temperature,
                         int32_t diff_sampling, uint64_t seed, uint64_t* rng_step, float* w_hat, float* dw,
                         shacira_stream_t stream) {
    if (count < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "sga_quantize: count is negative");
    if (count == 0) return SHACIRA_OK;
    if (!latents || !temperature || !w_hat) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "sga_quantize: NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t blocks = (count + kSgaBlock - 1) / kSgaBlock;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    sga_quantize_kernel<<<(int)blocks, kSgaBlock, 0, s>>>(latents, uniforms, count, temperature, diff_sampling,
                                                          (unsigned long long)seed, (const unsigned long long*)rng_step,
                                                          w_hat, dw);
    LAUNCHED();
    if (!uniforms && rng_step) {
        sga_advance_kernel<<<1, 1, 0, s>>>((unsigned long long*)rng_step);
        LAUNCHED();
    }
    return SHACIRA_OK;
}

}  // extern "C"

namespace {

// shacira_fit_optimizer_step and its best-state form (snap != NULL): one validation, one launch
int fit_optimizer_launch(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                         const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                         float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay, float beta1,
                         float beta2, float eps, float* step_small, float* step_table, const float* scale,
                         const float* div, float* A_out, int32_t latent_dim, int32_t feature_dim,
                         const float* temperature, int32_t diff_sampling, uint64_t seed, uint64_t* rng_step,
                         float* w_hat, float* dw, const float* ent_params, int32_t ent_layers,
                         const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step, double* bits,
                         float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes, uint32_t* ticket,
                         const shacira_fit_snapshot_t* snap, const shacira_fit_schedule_t* sched,
                         shacira_stream_t stream) {
    if (!step_small || !step_table || !ticket || num_segs < 0 || (num_segs > 0 && !segs))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: NULL argument");
    if (num_segs > SHACIRA_MAX_ADAM_SEGS)
        return fail(SHACIRA_ERR_UNSUPPORTED, "fit_optimizer_step: %d segments (max %d)", num_segs, SHACIRA_MAX_ADAM_SEGS);
    if (!table || !grad || !exp_avg || !exp_avg_sq || n <= 0)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: table / grad / state is NULL");
    if (w_hat && !temperature) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: SGA needs the temperature");
    if (A_out && (!scale || !div || latent_dim < 1 || feature_dim < 1))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: A_out needs scale, div, latent_dim, feature_dim");
    AdamSegs S;
    memset(&S, 0, sizeof(S));
    S.num = num_segs;
    bool owner = false;
    for (int i = 0; i < num_segs; ++i) {
        const shacira_adam_seg_t& g = segs[i];
        if (!g.param || !g.grad || !g.exp_avg || !g.exp_avg_sq || g.n < 0 || g.grad_rows < 1 ||
            (g.grad_div && g.div_group < 1))
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: bad segment %d", i);
        S.seg[i] = g;
        owner |= (g.param == scale);
    }
    if (A_out && !owner) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: A_out needs `scale` among the segments");
    TableAdam Tb;
    memset(&Tb, 0, sizeof(Tb));
    Tb.p = table; Tb.g = grad; Tb.gmul = grad_mul; Tb.g2 = grad2; Tb.scale2 = scale2; Tb.mul2 = scale2_mul;
    Tb.m = exp_avg; Tb.v = exp_avg_sq; Tb.n = n; Tb.lr = lr; Tb.weight_decay = weight_decay;
    Tb.temperature = temperature; Tb.diff_sampling = diff_sampling; Tb.seed = seed;
    Tb.rng_step = (unsigned long long*)rng_step; Tb.w_hat = w_hat; Tb.dw = dw;
    if (ent_params) {
        if (latent_dim != 1) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_optimizer_step: the folded bit-rate loss needs latent_dim = 1");
        if (!bits || !grad_ent_params || !ent_scratch || ent_layers < 1)
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: bit-rate outputs / scratch are NULL");
        if (ent_scratch_bytes < (int64_t)sizeof(float) * kOptEnt * ((n + 1023) / 1024))
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: bit-rate scratch too small");
        if (grad2) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step: grad2 and the folded bit-rate loss exclude each other");
        Tb.ent_params = ent_params; Tb.ent_layers = ent_layers; Tb.ent_noise = ent_noise; Tb.ent_seed = ent_seed;
        Tb.ent_rng_step = (unsigned long long*)ent_rng_step; Tb.ent_partials = (float*)ent_scratch; Tb.bits = bits;
        Tb.g_prob = grad_ent_params;
    }
    shacira_fit_snapshot_t sn;
    memset(&sn, 0, sizeof(sn));
    if (snap) {
        if (!snap->sse || snap->count <= 0 || !snap->best_loss || !snap->best_step || !snap->table)
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_best: snapshot sse / count / best / table missing");
        if (!A_out || !snap->div || !snap->A)
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_best: the snapshot of div and A needs A_out, div and A");
        sn = *snap;
    }
    const int64_t blocks = num_segs + (n + 1023) / 1024;
    if (sched) {
        if (snap)
            fit_optimizer_sched_kernel<true><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
                S, Tb, beta1, beta2, eps, step_small, step_table, scale, div, A_out, latent_dim, feature_dim, ticket, sn,
                *sched, bits);
        else
            fit_optimizer_sched_kernel<false><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
                S, Tb, beta1, beta2, eps, step_small, step_table, scale, div, A_out, latent_dim, feature_dim, ticket, sn,
                *sched, bits);
    } else if (snap)
        fit_optimizer_kernel<true><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
            S, Tb, beta1, beta2, eps, step_small, step_table, scale, div, A_out, latent_dim, feature_dim, ticket, sn);
    else
        fit_optimizer_kernel<false><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
            S, Tb, beta1, beta2, eps, step_small, step_table, scale, div, A_out, latent_dim, feature_dim, ticket, sn);
    LAUNCHED();
    return SHACIRA_OK;
}

}  // namespace

extern "C" {

int shacira_fit_optimizer_step(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                               const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                               float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay, float beta1,
                               float beta2, float eps, float* step_small, float* step_table, const float* scale,
                               const float* div, float* A_out, int32_t latent_dim, int32_t feature_dim,
                               const float* temperature, int32_t diff_sampling, uint64_t seed, uint64_t* rng_step,
                               float* w_hat, float* dw, const float* ent_params, int32_t ent_layers,
                               const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step, double* bits,
                               float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes, uint32_t* ticket,
                               shacira_stream_t stream) {
    return fit_optimizer_launch(segs, num_segs, table, grad, grad_mul, grad2, scale2, scale2_mul, exp_avg, exp_avg_sq, n,
                                lr, weight_decay, beta1, beta2, eps, step_small, step_table, scale, div, A_out,
                                latent_dim, feature_dim, temperature, diff_sampling, seed, rng_step, w_hat, dw,
                                ent_params, ent_layers, ent_noise, ent_seed, ent_rng_step, bits, grad_ent_params,
                                ent_scratch, ent_scratch_bytes, ticket, nullptr, nullptr, stream);
}

int shacira_fit_optimizer_step_best(const shacira_adam_seg_t* segs, int32_t num_segs, float* table, float* grad,
                                    const float* grad_mul, const float* grad2, const float* scale2, float scale2_mul,
                                    float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float weight_decay,
                                    float beta1, float beta2, float eps, float* step_small, float* step_table,
                                    const float* scale, const float* div, float* A_out, int32_t latent_dim,
                                    int32_t feature_dim, const float* temperature, int32_t diff_sampling, uint64_t seed,
                                    uint64_t* rng_step, float* w_hat, float* dw, const float* ent_params,
                                    int32_t ent_layers, const float* ent_noise, uint64_t ent_seed, uint64_t* ent_rng_step,
                                    double* bits, float* grad_ent_params, void* ent_scratch, int64_t ent_scratch_bytes,
                                    uint32_t* ticket, const shacira_fit_snapshot_t* snap, shacira_stream_t stream) {
    if (!snap) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_best: snapshot descriptor is NULL");
    return fit_optimizer_launch(segs, num_segs, table, grad, grad_mul, grad2, scale2, scale2_mul, exp_avg, exp_avg_sq, n,
                                lr, weight_decay, beta1, beta2, eps, step_small, step_table, scale, div, A_out,
                                latent_dim, feature_dim, temperature, diff_sampling, seed, rng_step, w_hat, dw,
                                ent_params, ent_layers, ent_noise, ent_seed, ent_rng_step, bits, grad_ent_params,
                                ent_scratch, ent_scratch_bytes, ticket, snap, nullptr, stream);
}

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
                                     const shacira_fit_schedule_t* sched, shacira_stream_t stream) {
    if (!sched) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: schedule descriptor is NULL");
    if (!sched->log) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: the step log is NULL");
    if (sched->log_capacity < 0)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: log_capacity %lld < 0",
                    (long long)sched->log_capacity);
    if (!sched->sse || sched->count <= 0)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: sse / count missing");
    if (sched->num_epochs < 1)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: num_epochs %d < 1", sched->num_epochs);
    if (!(sched->decay_period > 0.0 && sched->decay_period <= 1.0))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: decay_period %g outside (0, 1]",
                    sched->decay_period);
    if (!(sched->temperature_end > 0.0))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: temperature_end %g <= 0",
                    sched->temperature_end);
    if (sched->lambda_kind != SHACIRA_LAMBDA_COSINE && sched->lambda_kind != SHACIRA_LAMBDA_FIX)
        return fail(SHACIRA_ERR_UNSUPPORTED, "fit_optimizer_step_sched: unknown lambda kind %d", sched->lambda_kind);
    if (!scale2 || !temperature)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: the lambda (scale2) and temperature scalars are NULL");
    if (reinterpret_cast<uintptr_t>(sched->log) & 15)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_optimizer_step_sched: the step log must be 16-byte aligned");
    return fit_optimizer_launch(segs, num_segs, table, grad, grad_mul, grad2, scale2, scale2_mul, exp_avg, exp_avg_sq, n,
                                lr, weight_decay, beta1, beta2, eps, step_small, step_table, scale, div, A_out,
                                latent_dim, feature_dim, temperature, diff_sampling, seed, rng_step, w_hat, dw,
                                ent_params, ent_layers, ent_noise, ent_seed, ent_rng_step, bits, grad_ent_params,
                                ent_scratch, ent_scratch_bytes, ticket, snap, sched, stream);
}

int shacira_multi_adam_step(const shacira_adam_seg_t* segs, int32_t num_segs, float beta1, float beta2, float eps,
                            float* step, float* extra_step, const float* scale, const float* div, float* A_out,
                            int32_t latent_dim, int32_t feature_dim, uint32_t* ticket, shacira_stream_t stream) {
    if (!step || !ticket || num_segs < 0 || (num_segs > 0 && !segs))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "multi_adam_step: NULL argument");
    if (num_segs > SHACIRA_MAX_ADAM_SEGS)
        return fail(SHACIRA_ERR_UNSUPPORTED, "multi_adam_step: %d segments (max %d)", num_segs, SHACIRA_MAX_ADAM_SEGS);
    if (A_out && (!scale || !div || latent_dim < 1 || feature_dim < 1))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "multi_adam_step: A_out needs scale, div, latent_dim, feature_dim");
    AdamSegs S;
    memset(&S, 0, sizeof(S));
    S.num = num_segs;
    for (int i = 0; i < num_segs; ++i) {
        const shacira_adam_seg_t& g = segs[i];
        if (!g.param || !g.grad || !g.exp_avg || !g.exp_avg_sq || g.n < 0 || g.grad_rows < 1 ||
            (g.grad_div && g.div_group < 1))
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "multi_adam_step: bad segment %d", i);
        S.seg[i] = g;
    }
    if (num_segs == 0) return SHACIRA_OK;
    if (A_out) {
        bool owner = false;
        for (int i = 0; i < num_segs; ++i) owner |= (segs[i].param == scale);
        if (!owner) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "multi_adam_step: A_out needs `scale` among the segments");
    }
    multi_adam_kernel<<<num_segs, 128, 0, (cudaStream_t)stream>>>(S, beta1, beta2, eps, step, extra_step, scale, div,
                                                                  A_out, latent_dim, feature_dim, ticket);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_quantize_symbols(const float* latents, int64_t table_rows, int32_t latent_dim, int16_t* symbols,
                             int32_t* minmax, shacira_stream_t stream) {
    if (!latents || !minmax) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/minmax is NULL");
    if (latent_dim < 1 || latent_dim > kMaxEntC || (latent_dim & (latent_dim - 1)))
        return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d must be a power of two <= %d", latent_dim, kMaxEntC);
    cudaStream_t s = (cudaStream_t)stream;
    init_minmax_kernel<<<1, 32, 0, s>>>(minmax, latent_dim);
    LAUNCHED();
    const int64_t total = table_rows * latent_dim;
    if (total <= 0) return SHACIRA_OK;
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    quantize_symbols_kernel<<<(int)blocks, 256, 0, s>>>(latents, total, latent_dim, symbols, minmax);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_symbol_histogram(const float* latents, int64_t table_rows, int32_t latent_dim, const int32_t* lo,
                             int32_t num_bins, int64_t* counts, shacira_stream_t stream) {
    if (!latents || !lo || !counts) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/lo/counts is NULL");
    if (latent_dim < 1 || latent_dim > kMaxEntC || (latent_dim & (latent_dim - 1)))
        return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d must be a power of two <= %d", latent_dim, kMaxEntC);
    if (num_bins < 1) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "num_bins must be >= 1");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t total = table_rows * latent_dim;
    if (total <= 0) return SHACIRA_OK;
    // lo travels as a kernel-visible device copy: tiny, staged through a stream-ordered allocation
    int32_t* d_lo = nullptr;
    CUDA_OK(cudaMallocAsync((void**)&d_lo, sizeof(int32_t) * latent_dim, s));
    CUDA_OK(cudaMemcpyAsync(d_lo, lo, sizeof(int32_t) * latent_dim, cudaMemcpyHostToDevice, s));
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 4) blocks = 148 * 4;
    symbol_histogram_kernel<<<(int)blocks, 256, 0, s>>>(latents, total, latent_dim, d_lo, num_bins,
                                                        (unsigned long long*)counts);
    launch_counter().fetch_add(1);
    cudaError_t le = cudaGetLastError();
    cudaFreeAsync(d_lo, s);
    if (le != cudaSuccess) return fail(SHACIRA_ERR_CUDA, "histogram launch: %s", cudaGetErrorString(le));
    return SHACIRA_OK;
}

// ---- fused decoder MLP + MSE (SURVEY 8 f-1) ------------------------------------------------------------
int shacira_mlp_mse_step_bounded(const float* features, const float* target, int64_t n, int32_t in_dim,
                                 int32_t hidden_dim, int32_t out_dim, const float* W1, const float* b1, const float* W2,
                                 const float* b2, const float* W3, const float* b3, float* grad_features, float* pred,
                                 void* out, float* grad_feature_absmax, shacira_stream_t stream) {
    if (!features || !target || !W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !grad_features || !out)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "mlp_mse_step: NULL argument");
    if (n <= 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "mlp_mse_step: n must be positive");
    if (hidden_dim != 16 || out_dim != 3)
        return fail(SHACIRA_ERR_UNSUPPORTED, "mlp_mse_step: hidden %d / out %d (compiled: 16 / 3)", hidden_dim, out_dim);
    cudaStream_t s = (cudaStream_t)stream;
    switch (in_dim) {
        case 16: return launch_mlp_tc(features, target, n, W1, b1, W2, b2, W3, b3, grad_features, pred, out,
                                      grad_feature_absmax, s);
        case 24: if (grad_feature_absmax) return fail(SHACIRA_ERR_UNSUPPORTED, "mlp_mse_step_bounded: in_dim 16 only");
                 return launch_mlp<24>(features, target, n, W1, b1, W2, b2, W3, b3, grad_features, pred, out, s);
        case 32: if (grad_feature_absmax) return fail(SHACIRA_ERR_UNSUPPORTED, "mlp_mse_step_bounded: in_dim 16 only");
                 return launch_mlp<32>(features, target, n, W1, b1, W2, b2, W3, b3, grad_features, pred, out, s);
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "mlp_mse_step: in_dim %d not in {16,24,32}", in_dim);
    }
}

int shacira_mlp_mse_step(const float* features, const float* target, int64_t n, int32_t in_dim, int32_t hidden_dim,
                         int32_t out_dim, const float* W1, const float* b1, const float* W2, const float* b2,
                         const float* W3, const float* b3, float* grad_features, float* pred, void* out,
                         shacira_stream_t stream) {
    return shacira_mlp_mse_step_bounded(features, target, n, in_dim, hidden_dim, out_dim, W1, b1, W2, b2, W3, b3,
                                        grad_features, pred, out, nullptr, stream);
}

// ---- packed exponential integration (SURVEY 8 f-3) ---------------------------------------------------
#define DISPATCH_NF(NF_, CALL)                                                                     \
    switch (NF_) {                                                                                 \
        case 1: { constexpr int kNF = 1; CALL; break; }                                            \
        case 3: { constexpr int kNF = 3; CALL; break; }                                            \
        case 4: { constexpr int kNF = 4; CALL; break; }                                            \
        case 8: { constexpr int kNF = 8; CALL; break; }                                            \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "num_feats %d not in {1,3,4,8}", (int)NF_);  \
    }

int shacira_integrate_forward(const float* feats, const float* tau, const int32_t* ray_start, int32_t num_rays,
                              int32_t num_feats, float* weights, float* ray_feats, float* ray_alpha,
                              shacira_stream_t stream) {
    if (num_rays < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "num_rays is negative");
    if (num_rays == 0) return SHACIRA_OK;
    if (!feats || !tau || !ray_start || !weights || !ray_feats)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "integrate_forward: NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = (num_rays + kRenderWarps - 1) / kRenderWarps;
    DISPATCH_NF(num_feats, (integrate_fwd_kernel<kNF><<<blocks, kRenderWarps * 32, 0, s>>>(
                               feats, tau, ray_start, num_rays, weights, ray_feats, ray_alpha)))
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_integrate_backward(const float* feats, const float* tau, const float* weights, const int32_t* ray_start,
                               int32_t num_rays, int32_t num_feats, const float* grad_ray_feats,
                               const float* grad_weights, float* grad_feats, float* grad_tau, shacira_stream_t stream) {
    if (num_rays < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "num_rays is negative");
    if (num_rays == 0) return SHACIRA_OK;
    if (!feats || !tau || !weights || !ray_start || !grad_ray_feats || !grad_tau)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "integrate_backward: NULL argument");
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = (num_rays + kRenderWarps - 1) / kRenderWarps;
    DISPATCH_NF(num_feats, (integrate_bwd_kernel<kNF><<<blocks, kRenderWarps * 32, 0, s>>>(
                               feats, tau, weights, ray_start, num_rays, grad_ray_feats, grad_weights, grad_feats,
                               grad_tau)))
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_voxel_samples(const float* origins, const float* dirs, const int32_t* ridx, const float* depth,
                          const float* jitter, int64_t num_nuggets, int32_t num_samples, int64_t* ridx_out,
                          float* samples, float* depth_samples, float* deltas, uint8_t* boundary,
                          shacira_stream_t stream) {
    if (num_nuggets < 0 || num_samples < 1) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "voxel_samples: bad sizes");
    if (num_nuggets == 0) return SHACIRA_OK;
    if (!origins || !dirs || !ridx || !depth || !jitter || !samples || !depth_samples || !deltas || !boundary)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "voxel_samples: NULL argument");
    const int64_t total = num_nuggets * num_samples;
    if (total > ((int64_t)1 << 38)) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "voxel_samples: too many samples");
    // 1.0 / num_samples as torch multiplies by it: a double scalar narrowed to float32 (sampling.py:52)
    const float inv_k = (float)(1.0 / (double)num_samples);
    voxel_samples_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        origins, dirs, ridx, depth, jitter, num_nuggets, num_samples, inv_k, ridx_out, samples, depth_samples, deltas,
        boundary);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_raytrace_dense_count(const uint8_t* occupancy, int32_t res, const float* origins, const float* dirs,
                                 int32_t num_rays, int32_t* count, shacira_stream_t stream) {
    if (res < 1 || res > 1024 || num_rays < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "raytrace_dense: bad res / num_rays");
    if (num_rays == 0) return SHACIRA_OK;
    if (!occupancy || !origins || !dirs || !count) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "raytrace_dense_count: NULL argument");
    raytrace_dense_kernel<false><<<(num_rays + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        occupancy, res, origins, dirs, num_rays, count, nullptr, nullptr, nullptr, nullptr);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_raytrace_dense_fill(const uint8_t* occupancy, int32_t res, const float* origins, const float* dirs,
                                int32_t num_rays, const int64_t* offset, int32_t* ridx, int32_t* pidx, float* depth,
                                shacira_stream_t stream) {
    if (res < 1 || res > 1024 || num_rays < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "raytrace_dense: bad res / num_rays");
    if (num_rays == 0) return SHACIRA_OK;
    if (!occupancy || !origins || !dirs || !offset || !ridx || !pidx || !depth)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "raytrace_dense_fill: NULL argument");
    raytrace_dense_kernel<true><<<(num_rays + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        occupancy, res, origins, dirs, num_rays, nullptr, offset, ridx, pidx, depth);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_prune_samples(int32_t res, const float* jitter, float* samples, shacira_stream_t stream) {
    if (res < 1 || res > 1024) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "prune_samples: bad res");
    if (!jitter || !samples) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "prune_samples: NULL argument");
    const int64_t cells = (int64_t)res * res * res;
    prune_samples_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, (cudaStream_t)stream>>>(res, jitter, samples);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_prune_update(int64_t cells, const float* density, float decay, float min_density, float* occupancy,
                         uint8_t* mask, shacira_stream_t stream) {
    if (cells < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "prune_update: cells is negative");
    if (cells == 0) return SHACIRA_OK;
    if (!density || !occupancy || !mask) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "prune_update: NULL argument");
    prune_update_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, (cudaStream_t)stream>>>(cells, density, decay,
                                                                                           min_density, occupancy, mask);
    LAUNCHED();
    return SHACIRA_OK;
}

// ---- latent bitstream (host) ---------------------------------------------------------------
int64_t shacira_ac_encode(const int16_t* symbols, int64_t n, const uint32_t* cdf, int32_t num_symbols, uint8_t* out,
                          int64_t out_capacity) {
    if (!symbols || !cdf || !out || n < 0 || num_symbols < 1) {
        fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_encode: bad argument");
        return SHACIRA_ERR_INVALID_ARGUMENT;
    }
    if (cdf[0] != 0 || cdf[num_symbols] != (1u << 16)) {
        fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_encode: cdf must run from 0 to 65536");
        return SHACIRA_ERR_INVALID_ARGUMENT;
    }
    for (int32_t k = 0; k < num_symbols; ++k)
        if (cdf[k + 1] <= cdf[k]) {
            fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_encode: cdf must be strictly increasing");
            return SHACIRA_ERR_INVALID_ARGUMENT;
        }
    const int64_t r = shacira_ac::encode(symbols, n, cdf, num_symbols, out, out_capacity);
    if (r == -1) {
        fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_encode: symbol out of range");
        return SHACIRA_ERR_INVALID_ARGUMENT;
    }
    if (r < -1) {
        fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_encode: output buffer too small (%lld bytes needed)", (long long)(-2 - r));
        return SHACIRA_ERR_INVALID_ARGUMENT;
    }
    return r;
}

int shacira_ac_decode(const uint8_t* in, int64_t nbytes, const uint32_t* cdf, int32_t num_symbols, int16_t* symbols,
                      int64_t n) {
    if (!in || !cdf || !symbols || n < 0 || num_symbols < 1)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "ac_decode: bad argument");
    return shacira_ac::decode(in, nbytes, cdf, num_symbols, symbols, n);
}

// ---- host-buffer step ------------------------------------------------------------------
namespace {
struct HostStepScratch {
    shacira_plan_t* plan = nullptr;
    void* ptr = nullptr;
    size_t bytes = 0;
    cudaStream_t stream[2] = {nullptr, nullptr};
    cudaEvent_t up_done = nullptr;
    int dev = -1;
};
thread_local HostStepScratch g_scratch;
}  // namespace

int shacira_latent_step_host(int32_t dim, const float* coords, int64_t n, const float* latents, int64_t table_rows,
                             const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                             int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, int32_t round_flag,
                             const float* A, const float* shift, int32_t per_level, const float* grad_output,
                             float* feats, float* grad_latents) {
    if (n <= 0 || table_rows <= 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "n and table_rows must be positive");
    if (!coords || !latents || !A || !grad_output || !feats || !grad_latents)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "NULL host buffer");
    if (dim != 2 && dim != 3) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "dim must be 2 or 3");
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    HostStepScratch& sc = g_scratch;
    const int nA = per_level ? num_lods : 1;
    const size_t LF = (size_t)num_lods * feature_dim;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_coords = al(sizeof(float) * n * dim), b_lat = al(sizeof(float) * table_rows * latent_dim);
    const size_t b_rows = al(sizeof(float) * n * LF), b_A = al(sizeof(float) * nA * latent_dim * feature_dim);
    const size_t b_shift = al(sizeof(float) * nA * feature_dim);
    const size_t need = b_coords + 2 * b_lat + 2 * b_rows + b_A + b_shift;
    if (sc.dev != dev || sc.bytes < need) {
        if (sc.ptr) cudaFree(sc.ptr);
        sc.ptr = nullptr;
        CUDA_OK(cudaMalloc(&sc.ptr, need));
        sc.bytes = need;
        if (sc.dev != dev) {
            for (int k = 0; k < 2; ++k) CUDA_OK(cudaStreamCreateWithFlags(&sc.stream[k], cudaStreamNonBlocking));
            CUDA_OK(cudaEventCreateWithFlags(&sc.up_done, cudaEventDisableTiming));
        }
        sc.dev = dev;
    }
    char* p = (char*)sc.ptr;
    float* d_coords = (float*)p; p += b_coords;
    float* d_lat = (float*)p; p += b_lat;
    float* d_glat = (float*)p; p += b_lat;
    float* d_feats = (float*)p; p += b_rows;
    float* d_gout = (float*)p; p += b_rows;
    float* d_A = (float*)p; p += b_A;
    float* d_shift = (float*)p;
    cudaStream_t s0 = sc.stream[0], s1 = sc.stream[1];
    // stream 0: table + coords up, forward, features down. stream 1: grad_output up (overlaps
    // the forward), then the backward once the forward's inputs are resident, gradient down.
    CUDA_OK(cudaMemcpyAsync(d_lat, latents, sizeof(float) * table_rows * latent_dim, cudaMemcpyHostToDevice, s0));
    CUDA_OK(cudaMemcpyAsync(d_A, A, sizeof(float) * nA * latent_dim * feature_dim, cudaMemcpyHostToDevice, s0));
    if (shift) CUDA_OK(cudaMemcpyAsync(d_shift, shift, sizeof(float) * nA * feature_dim, cudaMemcpyHostToDevice, s0));
    CUDA_OK(cudaMemcpyAsync(d_coords, coords, sizeof(float) * n * dim, cudaMemcpyHostToDevice, s0));
    CUDA_OK(cudaMemcpyAsync(d_gout, grad_output, sizeof(float) * n * LF, cudaMemcpyHostToDevice, s1));
    // the coordinates are new to the device every call: bin them (3 small kernels, allocation reused),
    // then run the tiled kernels; configurations the tiled path does not cover use the point-parallel ones
    const bool tiled = (num_lods % 4 == 0) && n >= 65536;   // crossover measured: profiles/r02h_crossover.jsonl
    int rc = SHACIRA_OK;
    if (tiled) {
        rc = sc.plan ? shacira_plan_rebuild(sc.plan, dim, d_coords, n, 0, s0)
                     : shacira_plan_create(dim, d_coords, n, 0, s0, &sc.plan);
        if (rc) return rc;
        rc = shacira_latent_forward_planned(sc.plan, d_lat, first_idx, resolutions, num_lods, codebook_bitwidth,
                                            latent_dim, feature_dim, round_flag, d_A, shift ? d_shift : nullptr,
                                            per_level, d_feats, s0);
    } else {
        rc = shacira_latent_forward(dim, d_coords, n, d_lat, first_idx, resolutions, num_lods, codebook_bitwidth,
                                    latent_dim, feature_dim, round_flag, d_A, shift ? d_shift : nullptr, per_level,
                                    d_feats, nullptr, s0);
    }
    if (rc) return rc;
    CUDA_OK(cudaEventRecord(sc.up_done, s0));  // plan + forward inputs resident
    CUDA_OK(cudaMemcpyAsync(feats, d_feats, sizeof(float) * n * LF, cudaMemcpyDeviceToHost, s0));
    CUDA_OK(cudaStreamWaitEvent(s1, sc.up_done, 0));
    if (tiled)
        rc = shacira_latent_backward_planned(sc.plan, d_gout, nullptr, first_idx, resolutions, num_lods,
                                             codebook_bitwidth, latent_dim, feature_dim, round_flag, d_A, per_level,
                                             table_rows, 1, d_glat, nullptr, nullptr, s1);
    else
        rc = shacira_latent_backward(dim, d_coords, n, d_gout, nullptr, first_idx, resolutions, num_lods,
                                     codebook_bitwidth, latent_dim, feature_dim, d_A, per_level, table_rows, 1, d_glat,
                                     nullptr, nullptr, s1);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(grad_latents, d_glat, sizeof(float) * table_rows * latent_dim, cudaMemcpyDeviceToHost, s1));
    CUDA_OK(cudaStreamSynchronize(s0));
    CUDA_OK(cudaStreamSynchronize(s1));
    return SHACIRA_OK;
}

}  // extern "C"
