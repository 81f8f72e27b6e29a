// grid3d_capi.cu -- launchers of the 3D lane-pair kernels (grid3d_kernels.cuh); declared in
// capi_internal.h and used by the unplanned (capi.cu) and planned (tiled_capi.cu) entry points.
#include "capi_internal.h"
#include "grid3d_kernels.cuh"

namespace shacira {

bool grid3d_supported(int latent_dim, int feature_dim, const void* table) {
    if (latent_dim != 1 && latent_dim != 2) return false;
    if (feature_dim != 1 && feature_dim != 2 && feature_dim != 4 && feature_dim != 8) return false;
    return ((uintptr_t)table & 15u) == 0;
}

namespace {
inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

inline bool needs_config(unsigned long long& done_mask) {   // cudaFuncSetAttribute is per device
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return true;
    if ((done_mask >> dev) & 1ull) return false;
    done_mask |= 1ull << dev;
    return true;
}

template <int C, int F>
int fwd3d(const float* coords, const int32_t* perm, int64_t n, const float* lat, const LevelParams& lp, const float* A,
          const float* shift, int per_level, int round_flag, float* feats, float* zsave, cudaStream_t s) {
    const int nA = per_level ? lp.num_lods : 1;
    if (!A && C != F) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "3D forward: A is NULL");
    const size_t smem = LpFwdLayout<C, F>::bytes(nA);
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(latent_fwd3d_lp_kernel<C, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    latent_fwd3d_lp_kernel<C, F><<<grid_for(n, kLpChunk), kLpBlock, smem, s>>>(coords, perm, n, lat, lp, A, shift,
                                                                                per_level, round_flag, feats, zsave);
    LAUNCHED();
    return SHACIRA_OK;
}

template <int C, int F>
int bwd3d(const float* coords, const int32_t* perm, int64_t n, const float* g, const float* zsave, const LevelParams& lp,
          const float* A, int per_level, uint32_t skip_mask, uint32_t level_mask, float* gl, float* gA, float* gS,
          cudaStream_t s, int ctas_per_sm) {
    const int nA = per_level ? lp.num_lods : 1;
    if (!A && C != F) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "3D backward: A is NULL");
    const bool dec = gA != nullptr || gS != nullptr;
    const size_t smem = LpBwdLayout<C, F>::bytes(lp.num_lods, nA, dec);
    if (smem > 200 * 1024) return fail(SHACIRA_ERR_UNSUPPORTED, "3D backward: %zu bytes of shared memory per CTA", smem);
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(latent_bwd3d_lp_kernel<C, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    int64_t blocks = (n + kLpChunk - 1) / kLpChunk;   // persistent CTAs
    const int64_t cap = (int64_t)sm_count() * ctas_per_sm;
    if (blocks > cap) blocks = cap;
    latent_bwd3d_lp_kernel<C, F><<<(int)blocks, kLpBlock, smem, s>>>(coords, perm, n, g, zsave, lp, A, per_level,
                                                                      skip_mask, level_mask, gl, gA, gS);
    LAUNCHED();
    return SHACIRA_OK;
}
}  // namespace

#define G3_DISPATCH(C_, F_, CALL)                                                                             \
    switch ((C_) * 16 + (F_)) {                                                                               \
        case 1 * 16 + 1: { constexpr int kC = 1, kF = 1; return CALL; }                                       \
        case 1 * 16 + 2: { constexpr int kC = 1, kF = 2; return CALL; }                                       \
        case 1 * 16 + 4: { constexpr int kC = 1, kF = 4; return CALL; }                                       \
        case 1 * 16 + 8: { constexpr int kC = 1, kF = 8; return CALL; }                                       \
        case 2 * 16 + 1: { constexpr int kC = 2, kF = 1; return CALL; }                                       \
        case 2 * 16 + 2: { constexpr int kC = 2, kF = 2; return CALL; }                                       \
        case 2 * 16 + 4: { constexpr int kC = 2, kF = 4; return CALL; }                                       \
        case 2 * 16 + 8: { constexpr int kC = 2, kF = 8; return CALL; }                                       \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "3D merged kernels: latent_dim %d / feature_dim %d",    \
                             (int)(C_), (int)(F_));                                                           \
    }

int launch_fwd3d(int C, int F, const float* coords, const int32_t* perm, int64_t n, const float* latents,
                 const LevelParams& lp, const float* A, const float* shift, int per_level, int round_flag, float* feats,
                 float* zsave, cudaStream_t s) {
    G3_DISPATCH(C, F, (fwd3d<kC, kF>(coords, perm, n, latents, lp, A, shift, per_level, round_flag, feats, zsave, s)))
}

int launch_bwd3d(int C, int F, const float* coords, const int32_t* perm, int64_t n, const float* grad_out,
                 const float* zsave, const LevelParams& lp, const float* A, int per_level, uint32_t skip_mask,
                 uint32_t level_mask, float* grad_latents, float* grad_A, float* grad_shift, cudaStream_t s,
                 int ctas_per_sm) {
    G3_DISPATCH(C, F, (bwd3d<kC, kF>(coords, perm, n, grad_out, zsave, lp, A, per_level, skip_mask, level_mask,
                                     grad_latents, grad_A, grad_shift, s, ctas_per_sm)))
}

}  // namespace shacira
