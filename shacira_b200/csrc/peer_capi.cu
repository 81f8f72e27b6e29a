// peer_capi.cu -- extern "C" entry points of the peer-memory exchange step (declared in include/shacira_b200.h):
// allocation / CUDA-IPC export / mapping of the gradient arenas and the one-kernel all-reduce over NVLink.
#include "capi_internal.h"
#include "peer_kernels.cuh"

using namespace shacira;

namespace {

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
constexpr int kPeerBlocksPerSm = 2;   // persistent CTAs of the exchange kernels

int fill_view(PeerView& v, void* const* bufs, int64_t flags_offset, int rank, int world) {
    if (world < 2 || world > kPeerMax || (world & (world - 1)))
        return fail(SHACIRA_ERR_UNSUPPORTED, "peer exchange: world size %d not in {2, 4, 8}", world);
    if (rank < 0 || rank >= world || !bufs) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer exchange: bad rank / bufs");
    memset(&v, 0, sizeof(v));
    for (int p = 0; p < world; ++p) {
        if (!bufs[p]) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer exchange: arena of rank %d is NULL", p);
        v.buf[p] = (float*)bufs[p];
        v.flags[p] = (unsigned*)((char*)bufs[p] + flags_offset);
    }
    v.rank = rank;
    v.world = world;
    return SHACIRA_OK;
}

template <bool ADAM>
int launch_peer(const PeerView& v, int64_t numel4, const PeerAdam& ad, cudaStream_t s) {
    const int64_t per = (numel4 + v.world - 1) / v.world;
    int64_t blocks = (per + kPeerThreads - 1) / kPeerThreads;
    const int64_t cap = (int64_t)sm_count() * kPeerBlocksPerSm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    switch (v.world) {
        case 2: peer_allreduce_kernel<2, ADAM><<<(int)blocks, kPeerThreads, 0, s>>>(v, numel4, ad); break;
        case 4: peer_allreduce_kernel<4, ADAM><<<(int)blocks, kPeerThreads, 0, s>>>(v, numel4, ad); break;
        default: peer_allreduce_kernel<8, ADAM><<<(int)blocks, kPeerThreads, 0, s>>>(v, numel4, ad); break;
    }
    LAUNCHED();
    return SHACIRA_OK;
}

}  // namespace

extern "C" {

int64_t shacira_peer_flags_offset(int64_t bytes) { return (int64_t)align256((size_t)bytes); }

int shacira_peer_alloc(int64_t bytes, void** ptr) {
    if (!ptr || bytes <= 0) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_alloc: bad arguments");
    const size_t total = align256((size_t)bytes) + 256;
    void* p = nullptr;
    CUDA_OK(cudaMalloc(&p, total));
    CUDA_OK(cudaMemset(p, 0, total));
    *ptr = p;
    return SHACIRA_OK;
}

int shacira_peer_free(void* ptr) {
    if (ptr) CUDA_OK(cudaFree(ptr));
    return SHACIRA_OK;
}

int shacira_peer_export(void* ptr, void* handle64) {
    if (!ptr || !handle64) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_export: NULL");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CUDA_OK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)handle64, ptr));
    return SHACIRA_OK;
}

int shacira_peer_open(const void* handle64, void** ptr) {
    if (!handle64 || !ptr) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_open: NULL");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    CUDA_OK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SHACIRA_OK;
}

int shacira_peer_close(void* ptr) {
    if (ptr) CUDA_OK(cudaIpcCloseMemHandle(ptr));
    return SHACIRA_OK;
}

int shacira_peer_enable_access(int32_t device, int32_t peer_device) {
    int prev = 0, can = 0;
    CUDA_OK(cudaGetDevice(&prev));
    CUDA_OK(cudaDeviceCanAccessPeer(&can, device, peer_device));
    if (!can) return fail(SHACIRA_ERR_UNSUPPORTED, "device %d cannot access device %d", device, peer_device);
    CUDA_OK(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
    cudaSetDevice(prev);
    CUDA_OK(e);
    return SHACIRA_OK;
}

int shacira_peer_status(const void* buf, int64_t flags_offset, int32_t* timed_out) {
    if (!buf || !timed_out) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_status: NULL");
    unsigned w = 0;
    CUDA_OK(cudaMemcpy(&w, (const char*)buf + flags_offset + 18 * sizeof(unsigned), sizeof(w), cudaMemcpyDeviceToHost));
    *timed_out = w ? 1 : 0;
    return SHACIRA_OK;
}

int shacira_peer_allreduce(void* const* bufs, int64_t flags_offset, int32_t rank, int32_t world, int64_t numel,
                           shacira_stream_t stream) {
    PeerView v;
    if (int rc = fill_view(v, bufs, flags_offset, rank, world)) return rc;
    if (numel <= 0 || (numel & 3)) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce: numel %lld must be a positive multiple of 4", (long long)numel);
    if ((int64_t)numel * 4 > flags_offset) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce: numel exceeds the arena");
    PeerAdam ad;
    memset(&ad, 0, sizeof(ad));
    return launch_peer<false>(v, numel / 4, ad, (cudaStream_t)stream);
}

int shacira_peer_allreduce_adam(void* const* bufs, int64_t flags_offset, int32_t rank, int32_t world, int64_t numel,
                                void* const* params, int64_t table_numel, float* exp_avg, float* exp_avg_sq,
                                const float* step, float lr, float beta1, float beta2, float eps, float weight_decay,
                                shacira_stream_t stream) {
    PeerView v;
    if (int rc = fill_view(v, bufs, flags_offset, rank, world)) return rc;
    if (numel <= 0 || (numel & 3) || table_numel <= 0 || (table_numel & 3) || table_numel > numel)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_adam: numel / table_numel must be positive multiples of 4");
    if ((int64_t)numel * 4 > flags_offset) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_adam: numel exceeds the arena");
    if (!params || !exp_avg || !exp_avg_sq || !step) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_adam: NULL");
    PeerAdam ad;
    memset(&ad, 0, sizeof(ad));
    for (int p = 0; p < world; ++p) {
        if (!params[p]) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_adam: table of rank %d is NULL", p);
        ad.param[p] = (float*)params[p];
    }
    ad.exp_avg = exp_avg;
    ad.exp_avg_sq = exp_avg_sq;
    ad.step = step;
    ad.lr = lr; ad.beta1 = beta1; ad.beta2 = beta2; ad.eps = eps; ad.weight_decay = weight_decay;
    ad.numel = table_numel;
    return launch_peer<true>(v, numel / 4, ad, (cudaStream_t)stream);
}

int shacira_peer_allreduce_multimem(void* multicast_ptr, void* const* flag_bufs, int64_t flags_offset, int32_t rank,
                                    int32_t world, int64_t numel, shacira_stream_t stream) {
    PeerView v;
    if (int rc = fill_view(v, flag_bufs, flags_offset, rank, world)) return rc;
    if (!multicast_ptr) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_multimem: multicast pointer is NULL");
    if (numel <= 0 || (numel & 3) || ((uintptr_t)multicast_ptr & 15))
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "peer_allreduce_multimem: numel must be a positive multiple of 4, the pointer 16-byte aligned");
    const int64_t numel4 = numel / 4;
    const int64_t per = (numel4 + world - 1) / world;
    int64_t blocks = (per + kPeerThreads * 4 - 1) / (kPeerThreads * 4);
    const int64_t cap = (int64_t)sm_count() * kPeerBlocksPerSm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    cudaStream_t s = (cudaStream_t)stream;
    switch (world) {
        case 2: peer_allreduce_mc_kernel<2><<<(int)blocks, kPeerThreads, 0, s>>>(v, (float*)multicast_ptr, numel4); break;
        case 4: peer_allreduce_mc_kernel<4><<<(int)blocks, kPeerThreads, 0, s>>>(v, (float*)multicast_ptr, numel4); break;
        default: peer_allreduce_mc_kernel<8><<<(int)blocks, kPeerThreads, 0, s>>>(v, (float*)multicast_ptr, numel4); break;
    }
    LAUNCHED();
    return SHACIRA_OK;
}

}  // extern "C"
