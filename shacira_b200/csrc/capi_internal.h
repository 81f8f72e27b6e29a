// capi_internal.h -- error reporting, launch counting and level metadata shared by the C-ABI
// translation units (capi.cu, tiled_capi.cu). Internal; the public surface is include/shacira_b200.h.
#pragma once
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace shacira {

char* last_error_buffer();           // thread-local, 512 bytes
std::atomic<int64_t>& launch_counter();

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(last_error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_OK(expr)                                                                          \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver         \
                            ? SHACIRA_ERR_NO_DEVICE : SHACIRA_ERR_CUDA,                        \
                        "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

#define LAUNCHED()                            \
    do {                                      \
        launch_counter().fetch_add(1);        \
        CUDA_OK(cudaGetLastError());          \
    } while (0)

// Level metadata + the checks the reference does not make (SURVEY 8b "error convention").
int build_levels(int32_t dim, const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                 int32_t bitwidth, LevelParams& lp);
int check_points(const float* coords, int64_t n);
// every level must end inside a table of `table_rows` rows (a mismatched first_idx / bitwidth would scatter out of bounds)
inline int check_table(const LevelParams& lp, int64_t table_rows) {
    for (int l = 0; l < lp.num_lods; ++l)
        if ((int64_t)lp.first[l] + lp.rows[l] > table_rows)
            return fail(SHACIRA_ERR_INVALID_ARGUMENT, "level %d ends at row %lld, past table_rows %lld", l,
                        (long long)lp.first[l] + lp.rows[l], (long long)table_rows);
    return SHACIRA_OK;
}

// SM count of the CURRENT device (cached per device ordinal).
inline int sm_count() {
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return 148;
    int v = cache[dev].load(std::memory_order_relaxed);
    if (v <= 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cache[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

// cudaFuncSetAttribute is per DEVICE: remember which devices a kernel has been configured on (bit per ordinal),
// so a process that drives several GPUs configures each of them.
inline bool needs_config(unsigned long long& done_mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return true;
    if ((done_mask >> dev) & 1ull) return false;
    done_mask |= 1ull << dev;
    return true;
}

// A side stream per calling thread AND device for kernels that run beside the caller's stream (event fork / join:
// composes with stream capture). Created once per (thread, device) and kept until the thread exits.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
struct SideStreams {
    SideStream dev[64];
    ~SideStreams() {
        for (auto& d : dev) {   // best effort: the context may already be gone at thread exit
            if (d.fork) cudaEventDestroy(d.fork);
            if (d.join) cudaEventDestroy(d.join);
            if (d.stream) cudaStreamDestroy(d.stream);
        }
    }
};
inline int side_stream(SideStream** out) {
    thread_local SideStreams all;
    int d = 0;
    CUDA_OK(cudaGetDevice(&d));
    if (d < 0 || d > 63) return fail(SHACIRA_ERR_CUDA, "device ordinal %d out of range", d);
    SideStream& ss = all.dev[d];
    if (!ss.stream) {
        CUDA_OK(cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking));
        CUDA_OK(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
        CUDA_OK(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
    }
    *out = &ss;
    return SHACIRA_OK;
}

// 3D lane-pair kernels (grid3d_kernels.cuh, launched from grid3d_capi.cu). `perm` != NULL: `coords` is a plan's
// sorted copy and row i of feats / grad_output belongs to sample perm[i]; zsave rows follow `coords`.
// *_supported: latent_dim 1 or 2 and 16-byte aligned tables.
bool grid3d_supported(int latent_dim, int feature_dim, const void* table);
int launch_fwd3d(int latent_dim, int feature_dim, const float* coords, const int32_t* perm, int64_t n,
                 const float* latents, const LevelParams& lp, const float* A, const float* shift, int per_level,
                 int round_flag, float* feats, float* zsave, cudaStream_t s);
int launch_bwd3d(int latent_dim, int feature_dim, const float* coords, const int32_t* perm, int64_t n,
                 const float* grad_out, const float* zsave, const LevelParams& lp, const float* A, int per_level,
                 uint32_t skip_mask, uint32_t level_mask, float* grad_latents, float* grad_A, float* grad_shift,
                 cudaStream_t s, int ctas_per_sm = 4);

}  // namespace shacira
