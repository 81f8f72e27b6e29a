// nerf_heads_capi.cu -- C entry points of the NeRF decoder heads on the tensor cores (nerf_heads_kernels.cuh).
#include "capi_internal.h"
#include "nerf_heads_kernels.cuh"

using namespace shacira;

namespace {

int check_shapes(int64_t n, int32_t in_dim, int32_t hidden_dim, int32_t num_rays, int32_t emb_dim, bool colour) {
    if (n < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads: num_samples is negative");
    if (in_dim != 64 && in_dim != 96)
        return fail(SHACIRA_ERR_UNSUPPORTED, "nerf_heads: in_dim %d has no kernel (64 or 96)", (int)in_dim);
    if (hidden_dim != heads::kH)
        return fail(SHACIRA_ERR_UNSUPPORTED, "nerf_heads: hidden_dim %d has no kernel (128)", (int)hidden_dim);
    if (!colour) return SHACIRA_OK;
    if (emb_dim < 0 || emb_dim > heads::kMaxE)
        return fail(SHACIRA_ERR_UNSUPPORTED, "nerf_heads: emb_dim %d has no kernel (0 .. %d)", (int)emb_dim,
                    heads::kMaxE);
    if (num_rays < 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads: num_rays is negative");
    return SHACIRA_OK;
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

template <typename K>
int configure(K kernel, size_t smem, unsigned long long& done) {
    if (needs_config(done)) CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return SHACIRA_OK;
}

int grid_for(int64_t n) {
    const int64_t tiles = (n + heads::kTile - 1) / heads::kTile;
    return (int)(tiles < sm_count() ? tiles : sm_count());
}

template <int IN, bool DENSITY_ONLY>
int launch_fwd(const heads::Params& p, cudaStream_t s) {
    static unsigned long long done = 0ull;
    auto kernel = heads::nerf_heads_fwd_kernel<IN, DENSITY_ONLY>;
    const size_t smem = heads::Smem<IN>::kDynamic;
    if (int rc = configure(kernel, smem, done)) return rc;
    kernel<<<grid_for(p.S), heads::kThreads, smem, s>>>(p);
    LAUNCHED();
    return SHACIRA_OK;
}

template <int IN>
int launch_bwd(const heads::Params& p, float* const* g, cudaStream_t s) {
    static unsigned long long done = 0ull;
    auto kernel = heads::nerf_heads_bwd_kernel<IN>;
    const size_t smem = heads::Smem<IN>::kDynamic;
    if (int rc = configure(kernel, smem, done)) return rc;
    const int ctas = grid_for(p.S);
    kernel<<<ctas, heads::kThreads, smem, s>>>(p);
    LAUNCHED();
    const int total = heads::kH * IN + heads::kD * heads::kH + heads::kH * (heads::kD + p.E) + heads::kH * heads::kH +
                      heads::kOut * heads::kH + heads::kH + heads::kD + heads::kH + heads::kH + heads::kOut;
    heads::nerf_heads_reduce_kernel<IN><<<(total + 255) / 256, 256, 0, s>>>(p.partial, ctas, p.E, g[0], g[1], g[2], g[3],
                                                                            g[4], g[5], g[6], g[7], g[8], g[9]);
    LAUNCHED();
    return SHACIRA_OK;
}

int64_t workspace_for(int32_t in_dim, int64_t ctas) {
    const int64_t per = in_dim == 96 ? heads::Partial<96>::kFloats : heads::Partial<64>::kFloats;
    return ctas * per * (int64_t)sizeof(float);
}

}  // namespace

extern "C" {

int64_t shacira_nerf_heads_workspace_bytes(int32_t in_dim) {
    if (in_dim != 64 && in_dim != 96) {
        fail(SHACIRA_ERR_UNSUPPORTED, "nerf_heads: in_dim %d has no kernel (64 or 96)", (int)in_dim);
        return -1;
    }
    return workspace_for(in_dim, sm_count());
}

int shacira_nerf_heads_forward(const float* feats, int64_t num_samples, int32_t in_dim, int32_t hidden_dim,
                               const float* vemb, int32_t num_rays, int32_t emb_dim, const int32_t* ridx,
                               const float* const* params, int32_t density_only, float* density, float* rgb,
                               shacira_stream_t stream) {
    const bool colour = density_only == 0;
    if (int rc = check_shapes(num_samples, in_dim, hidden_dim, num_rays, emb_dim, colour)) return rc;
    if (!params) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_forward: params is NULL");
    const int np = colour ? 10 : 4;
    for (int i = 0; i < np; ++i)
        if (!params[i]) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_forward: params[%d] is NULL", i);
    if (num_samples == 0) return SHACIRA_OK;
    if (!feats || !density) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_forward: NULL feats or density");
    if (colour && (!rgb || !ridx || (emb_dim > 0 && num_rays > 0 && !vemb)))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_forward: NULL rgb, ridx or vemb");
    if (!aligned16(feats)) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_forward: feats is not 16-byte aligned");
    heads::Params p{};
    p.X = feats; p.V = vemb; p.ridx = ridx; p.S = num_samples; p.R = num_rays; p.E = emb_dim;
    p.W1 = params[0]; p.b1 = params[1]; p.W2 = params[2]; p.b2 = params[3];
    if (colour) {
        p.W3 = params[4]; p.b3 = params[5]; p.W4 = params[6]; p.b4 = params[7]; p.W5 = params[8]; p.b5 = params[9];
    }
    p.density = density; p.rgb = rgb;
    cudaStream_t s = (cudaStream_t)stream;
    if (in_dim == 64) return colour ? launch_fwd<64, false>(p, s) : launch_fwd<64, true>(p, s);
    return colour ? launch_fwd<96, false>(p, s) : launch_fwd<96, true>(p, s);
}

int shacira_nerf_heads_backward(const float* feats, int64_t num_samples, int32_t in_dim, int32_t hidden_dim,
                                const float* vemb, int32_t num_rays, int32_t emb_dim, const int32_t* ridx,
                                const float* const* params, const float* grad_density, const float* grad_rgb,
                                float* grad_feats, float* const* grad_params, void* workspace, int64_t workspace_bytes,
                                shacira_stream_t stream) {
    if (int rc = check_shapes(num_samples, in_dim, hidden_dim, num_rays, emb_dim, true)) return rc;
    if (!params || !grad_params) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: params is NULL");
    for (int i = 0; i < 10; ++i) {
        if (!params[i]) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: params[%d] is NULL", i);
        if (!grad_params[i])
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: grad_params[%d] is NULL", i);
    }
    if (num_samples == 0) return SHACIRA_OK;
    if (!feats || !ridx || !grad_density || !grad_rgb || !grad_feats || (emb_dim > 0 && num_rays > 0 && !vemb))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: NULL argument");
    if (!aligned16(feats) || !aligned16(grad_feats))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: feats / grad_feats not 16-byte aligned");
    const int64_t need = workspace_for(in_dim, grid_for(num_samples));
    if (!workspace || workspace_bytes < need)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "nerf_heads_backward: workspace of %lld bytes, needs %lld",
                    (long long)workspace_bytes, (long long)need);
    heads::Params p{};
    p.X = feats; p.V = vemb; p.ridx = ridx; p.S = num_samples; p.R = num_rays; p.E = emb_dim;
    p.W1 = params[0]; p.b1 = params[1]; p.W2 = params[2]; p.b2 = params[3]; p.W3 = params[4];
    p.b3 = params[5]; p.W4 = params[6]; p.b4 = params[7]; p.W5 = params[8]; p.b5 = params[9];
    p.g_density = grad_density; p.g_rgb = grad_rgb; p.g_X = grad_feats; p.partial = (float*)workspace;
    cudaStream_t s = (cudaStream_t)stream;
    return in_dim == 64 ? launch_bwd<64>(p, grad_params, s) : launch_bwd<96>(p, grad_params, s);
}

}  // extern "C"
