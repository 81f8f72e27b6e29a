// tiled_capi.cu -- extern "C" entry points of the tiled fast path: plan create/destroy and the
// planned fused forward/backward (declared in include/shacira_b200.h).
#include <cstdlib>

#include "capi_internal.h"
#include "tiled_kernels.cuh"
#include "fit_kernels.cuh"

using namespace shacira;

struct shacira_plan {
    int32_t dim;
    int64_t n;
    int32_t g;       // tiles per axis
    int32_t ntiles;
    int device;
    void* block;     // one allocation: perm | coords_sorted | tile_off | cursor | counts | tile_id
    size_t block_bytes;
    // node table of the last level configuration used with this plan (PlanView::node_tab)
    int2* node_tab;
    size_t node_tab_bytes;
    int32_t node_stride, node_g, node_dim;
    uint64_t node_sig;
    int32_t* perm;
    float* coords_sorted;
    int32_t* tile_off;
    int32_t sorted_io;  // rows of feats / grad_output indexed by sorted position (shacira_plan_set_sorted_io)
};

namespace {

// dynamic shared memory per CTA for node storage (stays under 48 KB); SHACIRA_TILE_SMEM overrides it
// (the tests shrink it to force the per-level direct fallback)
int smem_budget() {
    const char* env = getenv("SHACIRA_TILE_SMEM");
    int b = env ? atoi(env) : 40 * 1024;
    if (b < 256) b = 256;
    if (b > 40 * 1024) b = 40 * 1024;
    return b;
}

PlanView view_of(const shacira_plan* p) {
    PlanView v;
    v.perm = p->sorted_io ? nullptr : p->perm;
    v.coords_sorted = p->coords_sorted;
    v.tile_off = p->tile_off;
    v.n = p->n;
    v.g = p->g;
    v.ntiles = p->ntiles;
    v.node_tab = p->node_tab;
    v.node_stride = p->node_stride;
    return v;
}

int node_capacity(const shacira_plan* p, const LevelParams& lp, int cap_max);
inline bool num_lods_ok(const LevelParams& lp) { return lp.num_lods % 4 == 0; }

// The node table depends on the tile grid and the level configuration only. It is (re)built when either
// changes -- once per fit -- with the largest node capacity any kernel uses, so that every kernel's staged
// prefix of levels finds its slots in it. Allocation is synchronous: like plan creation it has to happen
// before a CUDA-graph capture (any eager warm-up call does it).
int ensure_node_table(shacira_plan* p, const LevelParams& lp, cudaStream_t s) {
    uint64_t sig = 1469598103934665603ull;  // FNV-1a over everything the geometry depends on
    auto mix = [&](uint64_t v) { sig = (sig ^ v) * 1099511628211ull; };
    mix((uint64_t)lp.num_lods); mix(lp.hash_mask); mix(lp.dense_mask);
    for (int l = 0; l < lp.num_lods; ++l) { mix((uint64_t)lp.res[l]); mix((uint64_t)lp.first[l]); mix((uint64_t)lp.rows[l]); }
    const int cap = node_capacity(p, lp, smem_budget() / 4);
    mix((uint64_t)cap);
    if (p->node_tab && p->node_sig == sig && p->node_g == p->g && p->node_dim == p->dim) return SHACIRA_OK;
    const size_t bytes = sizeof(int2) * (size_t)p->ntiles * cap;
    if (!p->node_tab || p->node_tab_bytes < bytes) {
        if (p->node_tab) cudaFree(p->node_tab);
        p->node_tab = nullptr;
        p->node_tab_bytes = 0;
        cudaError_t e = cudaMalloc((void**)&p->node_tab, bytes);
        if (e != cudaSuccess) return fail(SHACIRA_ERR_CUDA, "cudaMalloc(%zu) for the node table: %s", bytes, cudaGetErrorString(e));
        p->node_tab_bytes = bytes;
    }
    if (p->dim == 2) plan_nodes_kernel<2><<<p->ntiles, kTileThreads, 0, s>>>(lp, p->g, cap, p->node_tab);
    else plan_nodes_kernel<3><<<p->ntiles, kTileThreads, 0, s>>>(lp, p->g, cap, p->node_tab);
    LAUNCHED();
    p->node_stride = cap;
    p->node_sig = sig;
    p->node_g = p->g;
    p->node_dim = p->dim;
    return SHACIRA_OK;
}

// Upper bound of the node box of any tile, all levels that fit `cap_max` (coarse first, as the kernel does).
int node_capacity(const shacira_plan* p, const LevelParams& lp, int cap_max) {
    long long run = 0;
    for (int l = 0; l < lp.num_lods; ++l) {
        long long w = lp.res[l] / p->g + 3, nodes = 1;
        for (int d = 0; d < p->dim; ++d) nodes *= w;
        if (run + nodes <= cap_max) run += nodes;
    }
    if (run < 32) run = 32;
    return (int)((run + 3) & ~3LL);  // multiple of 4 slots: the arrays behind it stay 16-byte aligned
}

template <int D, int C, int F>
int launch_fwd(shacira_plan* p, const float* lat, const LevelParams& lp, const float* A, const float* shift,
               int per_level, int round_flag, float* feats, cudaStream_t s) {
    const int nA = per_level ? lp.num_lods : 1;
    const int cap = node_capacity(p, lp, smem_budget() / (4 * C));
    const int rc_tab = ensure_node_table(p, lp, s);
    if (rc_tab) return rc_tab;
    size_t smem = sizeof(float) * ((size_t)cap * C + nA * C * F + nA * F);
    // scattered rows (original point order) of 16..64 floats: collected per batch in shared memory and written as whole rows
    const int RL = lp.num_lods * F;
    const size_t rows_bytes = ((smem + 15) & ~(size_t)15) - smem + sizeof(float) * (size_t)kTileThreads * kPts * (RL + 4 + 1);
    const int rows_via_smem = !p->sorted_io && RL % 4 == 0 && RL <= 64 && smem + rows_bytes <= 46 * 1024;
    if (rows_via_smem) smem += rows_bytes;
    // 2D: the next batch's permutation entries and coordinates in slots behind the rows (or the decoder), unless they
    // would take the launch past 46 KB (48 KB with the static part); that launch loads them directly
    const size_t smem_pts = ((smem + 15) & ~(size_t)15) + kFwdPointSlotBytes;
    if (D == 2 && smem_pts <= 46 * 1024)
        latent_fwd_tiled_kernel<D, C, F, D == 2><<<p->ntiles, kTileThreads, smem_pts, s>>>(
            view_of(p), lat, lp, A, shift, per_level, round_flag, feats, cap, rows_via_smem);
    else
        latent_fwd_tiled_kernel<D, C, F, false><<<p->ntiles, kTileThreads, smem, s>>>(view_of(p), lat, lp, A, shift, per_level,
                                                                                   round_flag, feats, cap, rows_via_smem);
    LAUNCHED();
    return SHACIRA_OK;
}

template <int D, int C, int F>
int launch_bwd(shacira_plan* p, const float* g, const float* lat, const LevelParams& lp, const float* A,
               int per_level, int round_flag, float* gl, float* gA, float* gS, const float* level_max, cudaStream_t s) {
    const int nA = per_level ? lp.num_lods : 1;
    const bool dec = gA != nullptr || gS != nullptr;
    // shared memory: fixed-point accumulators (kRepBudget ints of lane-replicated copies shared by the CA
    // accumulator channels + one slot per node) and -- only when the decoder gradients need the per-point
    // interpolation (F > C) -- the staged latents. Mirrors the kernel's SG / ZP / CA constants.
    const bool sg = dec && (F <= C), zp = dec && !sg;
    const int CA = sg ? F : C;
    const bool big = smem_budget() > 24 * 1024;
    const int rep = big ? ((kRepBudget / CA) & ~3) : 0;  // per accumulator channel
    const int cap = node_capacity(p, lp, (smem_budget() - rep * 4 * CA) / (4 * (CA + (dec ? C : 0))));
    const int cap_acc = cap + rep;
    const int rc_tab = ensure_node_table(p, lp, s);
    if (rc_tab) return rc_tab;
    constexpr int NW = kTileThreads / 32;
    size_t smem = sizeof(float) * ((size_t)cap_acc * CA + (dec ? (size_t)cap * C : 0) + nA * C * F);
    if (dec) smem += sizeof(float) * (size_t)(zp ? NW : 1) * lp.num_lods * (C * F + F);
    // 2D: the next-chunk slots, unless they would take the launch past 46 KB (48 KB with the static part) -- the
    // largest node boxes, which keep the register loop
    const size_t smem_pipe = ((smem + 15) & ~(size_t)15) + bwd_slot_bytes(D, F);
    if constexpr (bwd_pipelined(D, F)) {
        if (smem_pipe <= 46 * 1024) {
            if (dec)
                latent_bwd_tiled_kernel<D, C, F, true, true><<<p->ntiles, kTileThreads, smem_pipe, s>>>(
                    view_of(p), g, lat, lp, A, per_level, round_flag, gl, gA, gS, cap, cap_acc, level_max, SHACIRA_MAX_LEVELS, 0);
            else
                latent_bwd_tiled_kernel<D, C, F, false, true><<<p->ntiles, kTileThreads, smem_pipe, s>>>(
                    view_of(p), g, lat, lp, A, per_level, round_flag, gl, gA, gS, cap, cap_acc, level_max, SHACIRA_MAX_LEVELS, 0);
            LAUNCHED();
            return SHACIRA_OK;
        }
    }
    if (dec)
        latent_bwd_tiled_kernel<D, C, F, true, false><<<p->ntiles, kTileThreads, smem, s>>>(view_of(p), g, lat, lp, A, per_level,
                                                                                      round_flag, gl, gA, gS, cap, cap_acc, level_max, SHACIRA_MAX_LEVELS, 0);
    else
        latent_bwd_tiled_kernel<D, C, F, false, false><<<p->ntiles, kTileThreads, smem, s>>>(view_of(p), g, lat, lp, A, per_level,
                                                                                       round_flag, gl, gA, gS, cap, cap_acc, level_max, SHACIRA_MAX_LEVELS, 0);
    LAUNCHED();
    return SHACIRA_OK;
}

// ---- 3D (NeRF samples): lane-pair kernels on the sorted samples + tile-staged coarse levels ------------------------
// Number of leading levels the tiled backward stages in shared memory for this plan: while the (upper bound of the)
// node box of a tile stays below the corner touches of an average tile (otherwise staging only adds a flush) and
// the boxes fit the shared-memory budget.
int staged_prefix_3d(const shacira_plan* p, const LevelParams& lp, int cap_max, int* cap_out) {
    const double touches = 8.0 * (double)p->n / (double)p->ntiles;
    long long run = 0;
    int ns = 0;
    for (int l = 0; l < lp.num_lods; ++l) {
        const long long w = lp.res[l] / p->g + 3, nodes = w * w * w;
        if (run + nodes > cap_max) break;
        if ((double)nodes > touches) break;
        run += nodes;
        ++ns;
    }
    if (run < 32) run = 32;
    *cap_out = (int)((run + 3) & ~3LL);
    return ns;
}

template <int C, int F>
int launch_bwd_staged3d(shacira_plan* p, const float* g, const LevelParams& lp, const float* A, int per_level, float* gl,
                        int ns, int cap, cudaStream_t s) {
    const int nA = per_level ? lp.num_lods : 1;
    const int rep = (kRepBudget / C) & ~3;
    const int cap_acc = cap + rep;
    const size_t smem = sizeof(float) * ((size_t)cap_acc * C + nA * C * F);
    PlanView v = view_of(p);
    v.node_tab = nullptr;   // rows from the tile geometry at flush time (a 3D node table would be tens of MB)
    v.node_stride = 0;
    latent_bwd_tiled_kernel<3, C, F, false><<<p->ntiles, kTileThreads, smem, s>>>(
        v, g, nullptr, lp, A, per_level, 0, gl, nullptr, nullptr, cap, cap_acc, nullptr, ns, 1);
    LAUNCHED();
    return SHACIRA_OK;
}

// Two kernels side by side: the tiled kernel accumulates the staged (coarse / middle) levels per tile in shared memory,
// the lane-pair kernel sends the fine levels' reds and reduces the decoder gradients. Measured alternative, dropped:
// both regimes in ONE persistent tile-walking kernel (rows staged once, no second read) -- 306 / 384 us against
// 209 / 243 us for this form at the NeRF shape (profiles/r02e_probe3d_fused_ab.jsonl): five CTA-wide barriers per
// 128-sample tile serialise staging, scale, accumulation and flush, and with 3 resident CTAs per SM nothing hides them.
int backward_3d_two(shacira_plan* p, const float* g, const float* zsave, const LevelParams& lp, int C, int F, const float* A,
                    int per_level, float* gl, float* gA, float* gS, int ns, int cap, cudaStream_t s) {
    const uint32_t skip = ns >= 32 ? 0xffffffffu : ((1u << ns) - 1u);
    SideStream* ss = nullptr;
    if (ns > 0) {
        if (int rc = side_stream(&ss)) return rc;
        CUDA_OK(cudaEventRecord(ss->fork, s));
        CUDA_OK(cudaStreamWaitEvent(ss->stream, ss->fork, 0));
    }
    // The fine levels first: that kernel is bound by L2 reds and needs few warps (2 persistent CTAs per SM when the
    // staged kernel runs beside it), the tile-staged kernel by shared memory and issue slots; launched in this
    // order the two share every SM instead of queueing behind each other's CTAs.
    int rc = launch_bwd3d(C, F, p->coords_sorted, p->sorted_io ? nullptr : p->perm, p->n, g, zsave, lp, A, per_level, skip,
                          0xffffffffu, gl, gA, gS, s, ns > 0 ? 2 : 4);
    if (rc) return rc;
    bool forked = false;
    if (ns > 0) {
        if (C == 1) {
            switch (F) {
                case 1: rc = launch_bwd_staged3d<1, 1>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                case 2: rc = launch_bwd_staged3d<1, 2>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                case 4: rc = launch_bwd_staged3d<1, 4>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                default: rc = launch_bwd_staged3d<1, 8>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
            }
        } else {
            switch (F) {
                case 1: rc = launch_bwd_staged3d<2, 1>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                case 2: rc = launch_bwd_staged3d<2, 2>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                case 4: rc = launch_bwd_staged3d<2, 4>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
                default: rc = launch_bwd_staged3d<2, 8>(p, g, lp, A, per_level, gl, ns, cap, ss->stream); break;
            }
        }
        if (rc) return rc;
        CUDA_OK(cudaEventRecord(ss->join, ss->stream));
        forked = true;
    }
    if (forked) CUDA_OK(cudaStreamWaitEvent(s, ss->join, 0));
    return SHACIRA_OK;
}

int backward_3d(shacira_plan* p, const float* g, const float* zsave, const LevelParams& lp, int C, int F, const float* A,
                int per_level, float* gl, float* gA, float* gS, cudaStream_t s) {
    int cap = 32;
    const int budget = smem_budget();
    const int rep = (kRepBudget / C) & ~3;
    const int ns = staged_prefix_3d(p, lp, (budget - rep * 4 * C) / (4 * C), &cap);
    if (!num_lods_ok(lp)) cap = 32;
    const int ns_two = num_lods_ok(lp) ? ns : 0;   // the two-kernel form: the tiled kernel unrolls 4 levels
    return backward_3d_two(p, g, zsave, lp, C, F, A, per_level, gl, gA, gS, ns_two, cap, s);
}

#define T_DISPATCH_F(F_, CALL)                                                                     \
    switch (F_) {                                                                                  \
        case 1: { constexpr int kF = 1; return CALL; }                                             \
        case 2: { constexpr int kF = 2; return CALL; }                                             \
        case 4: { constexpr int kF = 4; return CALL; }                                             \
        case 8: { constexpr int kF = 8; return CALL; }                                             \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "feature_dim %d not in {1,2,4,8}", (int)F_); \
    }
#define T_DISPATCH_CF(C_, F_, CALL)                                                                \
    switch (C_) {                                                                                  \
        case 1: { constexpr int kC = 1; T_DISPATCH_F(F_, CALL) }                                   \
        case 2: { constexpr int kC = 2; T_DISPATCH_F(F_, CALL) }                                   \
        case 4: { constexpr int kC = 4; T_DISPATCH_F(F_, CALL) }                                   \
        default: return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d not in {1,2,4}", (int)C_);    \
    }

}  // namespace

namespace {

int choose_tiles_per_axis(int dim, int64_t n, int tile_points) {
    if (tile_points <= 0) {
        // 2D: ~384 points per tile (tuned round 1). 3D: ~128 samples, i.e. 16 tiles per axis at the NeRF batch: the
        // middle levels' node boxes stay small enough to live in L1 / shared memory (profiles/r02b_probe3d.jsonl)
        tile_points = dim == 3 ? 128 : 384;
    }
    // power of two per axis, about tile_points points per tile, at most kMaxTiles tiles
    int g = 1;
    for (;;) {
        long long tiles = 1, cur = 1;
        for (int d = 0; d < dim; ++d) { tiles *= 2LL * g; cur *= g; }
        if (tiles > kMaxTiles) break;
        // stop when doubling would drop below ~tile_points/2 points per tile
        if ((double)n / (double)cur <= (double)tile_points * (dim == 2 ? 2.0 : 2.83)) break;
        g *= 2;
    }
    return g;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// (Re)build the plan's arrays for `coords` on `stream`; the allocation is reused when it is large enough.
int plan_build(shacira_plan* p, int32_t dim, const float* coords, int64_t n, int32_t tile_points, cudaStream_t s) {
    const int g = choose_tiles_per_axis(dim, n, tile_points);
    int ntiles = 1;
    for (int d = 0; d < dim; ++d) ntiles *= g;
    const size_t b_perm = align256(4 * (size_t)n), b_coords = align256(4 * (size_t)n * dim);
    const size_t b_off = align256(4 * (size_t)(ntiles + 1)), b_cnt = align256(4 * (size_t)ntiles), b_tid = align256(4 * (size_t)n);
    const size_t total = b_perm + b_coords + b_off + 2 * b_cnt + b_tid;
    if (!p->block || p->block_bytes < total) {
        if (p->block) cudaFree(p->block);
        p->block = nullptr;
        p->block_bytes = 0;
        cudaError_t e = cudaMalloc(&p->block, total);
        if (e != cudaSuccess) return fail(SHACIRA_ERR_CUDA, "cudaMalloc(%zu) for the plan: %s", total, cudaGetErrorString(e));
        p->block_bytes = total;
    }
    p->dim = dim;
    p->n = n;
    p->g = g;
    p->ntiles = ntiles;
    char* q = (char*)p->block;
    p->perm = (int32_t*)q; q += b_perm;
    p->coords_sorted = (float*)q; q += b_coords;
    p->tile_off = (int32_t*)q; q += b_off;
    int32_t* cursor = (int32_t*)q; q += b_cnt;
    int32_t* counts = (int32_t*)q; q += b_cnt;
    int32_t* tile_id = (int32_t*)q;
    CUDA_OK(cudaMemsetAsync(counts, 0, 4 * (size_t)ntiles, s));
    const size_t hist = 4 * (size_t)ntiles;
    const int blocks = (int)((n + 1023) / 1024);
    const int count_blocks = blocks < 296 ? blocks : 296;
    if (dim == 2) plan_count_kernel<2><<<count_blocks, 1024, hist, s>>>(coords, n, g, ntiles, tile_id, counts);
    else plan_count_kernel<3><<<count_blocks, 1024, hist, s>>>(coords, n, g, ntiles, tile_id, counts);
    LAUNCHED();
    plan_scan_kernel<<<1, 1024, 0, s>>>(counts, ntiles, p->tile_off, cursor);
    LAUNCHED();
    if (dim == 2) plan_scatter_kernel<2><<<blocks, 1024, hist, s>>>(coords, n, ntiles, tile_id, cursor, p->perm, p->coords_sorted);
    else plan_scatter_kernel<3><<<blocks, 1024, hist, s>>>(coords, n, ntiles, tile_id, cursor, p->perm, p->coords_sorted);
    LAUNCHED();
    return SHACIRA_OK;
}

int check_plan_args(int32_t dim, const float* coords, int64_t n) {
    if (dim != 2 && dim != 3) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "dim must be 2 or 3, got %d", dim);
    if (n <= 0 || !coords) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan needs n > 0 points");
    if (n > 0x7fffffff) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan supports up to 2^31-1 points");
    return SHACIRA_OK;
}

}  // namespace

extern "C" {

int shacira_plan_create(int32_t dim, const float* coords, int64_t n, int32_t tile_points, shacira_stream_t stream,
                        shacira_plan_t** out) {
    if (!out) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan output pointer is NULL");
    *out = nullptr;
    int rc = check_plan_args(dim, coords, n);
    if (rc) return rc;
    shacira_plan* p = new (std::nothrow) shacira_plan();
    if (!p) return fail(SHACIRA_ERR_CUDA, "out of host memory");
    p->block = nullptr;
    p->block_bytes = 0;
    p->node_tab = nullptr;
    p->node_tab_bytes = 0;
    p->node_sig = 0;
    p->node_g = p->node_dim = p->node_stride = 0;
    cudaGetDevice(&p->device);
    rc = plan_build(p, dim, coords, n, tile_points, (cudaStream_t)stream);
    if (rc != SHACIRA_OK) {
        if (p->block) cudaFree(p->block);
        if (p->node_tab) cudaFree(p->node_tab);
        delete p;
        return rc;
    }
    *out = p;
    return SHACIRA_OK;
}

int shacira_plan_rebuild(shacira_plan_t* plan, int32_t dim, const float* coords, int64_t n, int32_t tile_points,
                         shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    int rc = check_plan_args(dim, coords, n);
    if (rc) return rc;
    return plan_build(plan, dim, coords, n, tile_points, (cudaStream_t)stream);
}

int shacira_plan_destroy(shacira_plan_t* plan) {
    if (!plan) return SHACIRA_OK;
    if (plan->block) cudaFree(plan->block);  // synchronises with outstanding work that uses the plan
    if (plan->node_tab) cudaFree(plan->node_tab);
    delete plan;
    return SHACIRA_OK;
}

int shacira_plan_info(const shacira_plan_t* plan, int64_t* n, int32_t* dim, int32_t* tiles_per_axis, int32_t* ntiles) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (n) *n = plan->n;
    if (dim) *dim = plan->dim;
    if (tiles_per_axis) *tiles_per_axis = plan->g;
    if (ntiles) *ntiles = plan->ntiles;
    return SHACIRA_OK;
}

int shacira_plan_debug(const shacira_plan_t* plan, const int32_t** perm, const float** coords_sorted,
                       const int32_t** tile_off) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (perm) *perm = plan->perm;
    if (coords_sorted) *coords_sorted = plan->coords_sorted;
    if (tile_off) *tile_off = plan->tile_off;
    return SHACIRA_OK;
}

int shacira_plan_set_sorted_io(shacira_plan_t* plan, int32_t sorted_io) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    plan->sorted_io = sorted_io ? 1 : 0;
    return SHACIRA_OK;
}

int shacira_latent_forward_planned(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                                   const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth,
                                   int32_t latent_dim, int32_t feature_dim, int32_t round_flag, const float* A,
                                   const float* shift, int32_t per_level, float* feats, shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    LevelParams lp;
    int rc = build_levels(plan->dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!latents || !feats || !A) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/feats/A is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (plan->dim == 3 && grid3d_supported(latent_dim, feature_dim, latents))
        return launch_fwd3d(latent_dim, feature_dim, plan->coords_sorted, plan->sorted_io ? nullptr : plan->perm, plan->n,
                            latents, lp, A, shift, per_level, round_flag, feats, nullptr, s);
    if (num_lods % 4) return fail(SHACIRA_ERR_UNSUPPORTED, "the tiled path needs num_lods %% 4 == 0 (got %d)", num_lods);
    if (plan->dim == 2) {
        T_DISPATCH_CF(latent_dim, feature_dim,
                      (launch_fwd<2, kC, kF>(const_cast<shacira_plan*>(plan), latents, lp, A, shift, per_level, round_flag, feats, s)))
    }
    T_DISPATCH_CF(latent_dim, feature_dim,
                  (launch_fwd<3, kC, kF>(const_cast<shacira_plan*>(plan), latents, lp, A, shift, per_level, round_flag, feats, s)))
}

int shacira_latent_backward_planned_bounded(const shacira_plan_t* plan, const float* grad_output, const float* latents,
                                    const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                                    int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                                    int32_t round_flag, const float* A, int32_t per_level, int64_t table_rows,
                                    int32_t zero_first, float* grad_latents, float* grad_A, float* grad_shift,
                                    const float* level_max, shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    LevelParams lp;
    int rc = build_levels(plan->dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!grad_latents || !A || !grad_output) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_latents/A/grad_output is NULL");
    if ((rc = check_table(lp, table_rows))) return rc;
    if ((grad_A || grad_shift) && !latents)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "decoder gradients need the latents (the interpolation is recomputed)");
    if (latent_dim != 1 && latent_dim != 2 && latent_dim != 4)
        return fail(SHACIRA_ERR_UNSUPPORTED, "latent_dim %d not in {1,2,4}", latent_dim);
    cudaStream_t s = (cudaStream_t)stream;
    if (plan->dim == 3 && !grad_A && !grad_shift && grid3d_supported(latent_dim, feature_dim, grad_latents)) {
        if (zero_first) CUDA_OK(cudaMemsetAsync(grad_latents, 0, sizeof(float) * (size_t)table_rows * latent_dim, s));
        return backward_3d(const_cast<shacira_plan*>(plan), grad_output, nullptr, lp, latent_dim, feature_dim, A, per_level,
                           grad_latents, nullptr, nullptr, s);
    }
    if (num_lods % 4) return fail(SHACIRA_ERR_UNSUPPORTED, "the tiled path needs num_lods %% 4 == 0 (got %d)", num_lods);
    if (zero_first) CUDA_OK(cudaMemsetAsync(grad_latents, 0, sizeof(float) * (size_t)table_rows * latent_dim, s));
    if (plan->dim == 2) {
        T_DISPATCH_CF(latent_dim, feature_dim,
                      (launch_bwd<2, kC, kF>(const_cast<shacira_plan*>(plan), grad_output, latents, lp, A, per_level, round_flag, grad_latents,
                                             grad_A, grad_shift, level_max, s)))
    }
    T_DISPATCH_CF(latent_dim, feature_dim,
                  (launch_bwd<3, kC, kF>(const_cast<shacira_plan*>(plan), grad_output, latents, lp, A, per_level, round_flag, grad_latents, grad_A,
                                         grad_shift, level_max, s)))
}


int shacira_latent_forward_planned_z(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                                     const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth,
                                     int32_t latent_dim, int32_t feature_dim, int32_t round_flag, const float* A,
                                     const float* shift, int32_t per_level, float* feats, float* zsave,
                                     shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (plan->dim != 3) return fail(SHACIRA_ERR_UNSUPPORTED, "forward_planned_z: 3D plans only (2D recomputes z on chip)");
    LevelParams lp;
    int rc = build_levels(plan->dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!latents || !feats || !A) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "latents/feats/A is NULL");
    if (!grid3d_supported(latent_dim, feature_dim, latents))
        return fail(SHACIRA_ERR_UNSUPPORTED, "forward_planned_z: latent_dim %d / feature_dim %d / table alignment", latent_dim, feature_dim);
    return launch_fwd3d(latent_dim, feature_dim, plan->coords_sorted, plan->sorted_io ? nullptr : plan->perm, plan->n,
                        latents, lp, A, shift, per_level, round_flag, feats, zsave, (cudaStream_t)stream);
}

int shacira_latent_backward_planned_z(const shacira_plan_t* plan, const float* grad_output, const float* zsave,
                                      const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                                      int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim, const float* A,
                                      int32_t per_level, int64_t table_rows, int32_t zero_first, float* grad_latents,
                                      float* grad_A, float* grad_shift, shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (plan->dim != 3) return fail(SHACIRA_ERR_UNSUPPORTED, "backward_planned_z: 3D plans only");
    LevelParams lp;
    int rc = build_levels(plan->dim, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!grad_latents || !A || !grad_output) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_latents/A/grad_output is NULL");
    if (grad_A && !zsave) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "grad_A requested without zsave");
    if (!grid3d_supported(latent_dim, feature_dim, grad_latents))
        return fail(SHACIRA_ERR_UNSUPPORTED, "backward_planned_z: latent_dim %d / feature_dim %d / table alignment", latent_dim, feature_dim);
    if ((rc = check_table(lp, table_rows))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (zero_first) CUDA_OK(cudaMemsetAsync(grad_latents, 0, sizeof(float) * (size_t)table_rows * latent_dim, s));
    return backward_3d(const_cast<shacira_plan*>(plan), grad_output, zsave, lp, latent_dim, feature_dim, A, per_level,
                       grad_latents, grad_A, grad_shift, s);
}

int shacira_latent_backward_planned(const shacira_plan_t* plan, const float* grad_output, const float* latents,
                                    const int32_t* first_idx, const int32_t* resolutions, int32_t num_lods,
                                    int32_t codebook_bitwidth, int32_t latent_dim, int32_t feature_dim,
                                    int32_t round_flag, const float* A, int32_t per_level, int64_t table_rows,
                                    int32_t zero_first, float* grad_latents, float* grad_A, float* grad_shift,
                                    shacira_stream_t stream) {
    return shacira_latent_backward_planned_bounded(plan, grad_output, latents, first_idx, resolutions, num_lods,
                                                   codebook_bitwidth, latent_dim, feature_dim, round_flag, A, per_level,
                                                   table_rows, zero_first, grad_latents, grad_A, grad_shift, nullptr,
                                                   stream);
}

int shacira_fit_tile_step(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                          const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth, int32_t round_flag,
                          const float* A, const float* shift, const float* target_sorted, const float* W1,
                          const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                          int64_t table_rows, float* grad_latents, float* grad_A, float* grad_shift, void* mlp_out,
                          shacira_stream_t stream) {
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (plan->dim != 2 || !plan->sorted_io)
        return fail(SHACIRA_ERR_UNSUPPORTED, "fit_tile_step: needs a 2D plan in sorted-I/O mode");
    if (num_lods != 16) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_tile_step: 16 levels (got %d)", num_lods);
    LevelParams lp;
    int rc = build_levels(2, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!latents || !A || !target_sorted || !W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !grad_latents || !mlp_out)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_tile_step: NULL argument");
    if ((rc = check_table(lp, table_rows))) return rc;
    shacira_plan* p = const_cast<shacira_plan*>(plan);
    // every level must live in the tile's node box: the upper bound of the box over all levels against the budget
    long long all = 0;
    for (int l = 0; l < lp.num_lods; ++l) { const long long w = lp.res[l] / p->g + 3; all += w * w; }
    const int rep = kRepBudget & ~3;
    const int cap_max = (smem_budget() - rep * 4) / 8;   // float slot + int accumulator per node
    if (all > cap_max) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_tile_step: %lld nodes per tile exceed the shared-memory box", all);
    const int cap = node_capacity(p, lp, cap_max);
    const int cap_acc = cap + rep;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = ensure_node_table(p, lp, s))) return rc;
    const size_t smem = sizeof(FitSmem) + sizeof(float) * ((size_t)cap + cap_acc);
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(fit_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    if (smem > 100 * 1024) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_tile_step: %zu bytes of shared memory", smem);
    CUDA_OK(cudaMemsetAsync(mlp_out, 0, 8 + sizeof(float) * kFitParams, s));
    int blocks = sm_count() * SHACIRA_FIT_MIN_CTAS;
    if (blocks > p->ntiles) blocks = p->ntiles;
    const int headroom = 1;   // bits of slack of the fixed-point gradient scale (fit_kernels.cuh)
    const float scale = (float)(2.0 / ((double)p->n * 3.0));
    fit_tile_kernel<<<blocks, kTileThreads, smem, s>>>(view_of(p), latents, lp, A, shift, round_flag, target_sorted, W1, b1,
                                                       W2, b2, W3, b3, scale, grad_latents, grad_A, grad_shift,
                                                       (double*)mlp_out, (float*)((char*)mlp_out + 8), cap, cap_acc, headroom);
    LAUNCHED();
    return SHACIRA_OK;
}

int shacira_fit_render(const shacira_plan_t* plan, const float* latents, const int32_t* first_idx,
                       const int32_t* resolutions, int32_t num_lods, int32_t codebook_bitwidth, const float* A,
                       const float* shift, const float* W1, const float* b1, const float* W2, const float* b2,
                       const float* W3, const float* b3, float* rgb, const float* target, uint64_t* sse_u8,
                       shacira_stream_t stream) {
    if (num_lods != 16) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_render: 16 levels (got %d)", num_lods);
    LevelParams lp;
    int rc = build_levels(2, first_idx, resolutions, num_lods, codebook_bitwidth, lp);
    if (rc) return rc;
    if (!latents || !A || !W1 || !b1 || !W2 || !b2 || !W3 || !b3)
        return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_render: NULL argument");
    if (!rgb && !target) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_render: neither rgb nor target: nothing to compute");
    if (target && !sse_u8) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "fit_render: target needs sse_u8");
    if (!plan) return fail(SHACIRA_ERR_INVALID_ARGUMENT, "plan is NULL");
    if (plan->dim != 2) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_render: needs a 2D plan");
    shacira_plan* p = const_cast<shacira_plan*>(plan);
    // every level must live in the tile's node box (one float slot per node, no accumulators)
    long long all = 0;
    for (int l = 0; l < lp.num_lods; ++l) { const long long w = lp.res[l] / p->g + 3; all += w * w; }
    const int cap_max = smem_budget() / 4;
    if (all > cap_max) return fail(SHACIRA_ERR_UNSUPPORTED, "fit_render: %lld nodes per tile exceed the shared-memory box", all);
    const int cap = node_capacity(p, lp, cap_max);
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = ensure_node_table(p, lp, s))) return rc;
    const size_t smem = sizeof(RenderSmem) + sizeof(float) * (size_t)cap;
    static unsigned long long configured = 0ull;
    if (needs_config(configured))
        CUDA_OK(cudaFuncSetAttribute(fit_render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    if (target) CUDA_OK(cudaMemsetAsync(sse_u8, 0, sizeof(uint64_t), s));
    int blocks = sm_count() * SHACIRA_FIT_MIN_CTAS;
    if (blocks > p->ntiles) blocks = p->ntiles;
    fit_render_kernel<<<blocks, kTileThreads, smem, s>>>(view_of(p), latents, lp, A, shift, W1, b1, W2, b2, W3, b3, rgb,
                                                         target, (unsigned long long*)sse_u8, cap);
    LAUNCHED();
    return SHACIRA_OK;
}

}  // extern "C"
