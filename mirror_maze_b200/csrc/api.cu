// api.cu — implementation of the device half of include/mirror_maze_cuda.h: context, scene upload, dispatch.
// Stands where the reference's Metal glue stood (reference src/utils.rs:14-102, src/main.rs:616-730, 861-894).
// No CPU fallback exists: every entry point fails with MM_ERR_CUDA when no sm_100-class device is usable.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include "scene_prep.h"

using namespace mmk;

#include <algorithm>
#include <mutex>
#include <vector>
#include "ctx.h"

static thread_local std::string g_create_err;

#define CK(call) MM_CK(call)

namespace mmapi {
int fail(mm_ctx *ctx, int code, const std::string &msg) {
    ctx->err = msg;
    return code;
}

// Mapped pinned host memory the library knows about (mm_host_alloc / mm_host_register): process-wide, any context.
struct HostRange { uintptr_t base; size_t bytes; bool owned; uintptr_t dev; };
static std::mutex g_host_mu;
static std::vector<HostRange> g_host;

void *host_device_alias(const void *p, size_t bytes) {
    if (!p || bytes == 0) return nullptr;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        for (const HostRange &r : g_host)
            if (a >= r.base && a + bytes <= r.base + r.bytes) return reinterpret_cast<void *>(r.dev + (a - r.base));
    }
    // pinned by someone else (cudaHostAlloc / cudaHostRegister in the caller, e.g. a torch pinned tensor): under unified
    // addressing such memory is mapped too; accept it when both ends of the range resolve to one contiguous device alias
    cudaPointerAttributes a0, a1;
    if (cudaPointerGetAttributes(&a0, p) != cudaSuccess || cudaPointerGetAttributes(&a1, reinterpret_cast<const char *>(p) + bytes - 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (a0.type != cudaMemoryTypeHost || a1.type != cudaMemoryTypeHost || !a0.devicePointer || !a1.devicePointer) return nullptr;
    if (reinterpret_cast<uintptr_t>(a1.devicePointer) - reinterpret_cast<uintptr_t>(a0.devicePointer) != bytes - 1) return nullptr;
    return a0.devicePointer;
}
}  // namespace mmapi
using mmapi::fail;

extern "C" {

int mm_create(int cuda_device, mm_ctx **out) {
    if (!out) return MM_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_err = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return MM_ERR_CUDA;
    }
    if (cuda_device < 0 || cuda_device >= n) { g_create_err = "cuda_device out of range"; return MM_ERR_INVALID; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cuda_device)) != cudaSuccess) { g_create_err = cudaGetErrorString(e); return MM_ERR_CUDA; }
    if (prop.major != 10) {
        g_create_err = "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + "; this library is built for sm_100a only";
        return MM_ERR_CUDA;
    }
    mm_ctx *ctx = new (std::nothrow) mm_ctx();
    if (!ctx) return MM_ERR_NOMEM;
    ctx->device = cuda_device;
    ctx->n_sms = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    bool ok = cudaSetDevice(cuda_device) == cudaSuccess && cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreate(&ctx->ev0) == cudaSuccess && cudaEventCreate(&ctx->ev1) == cudaSuccess &&
              cudaEventCreateWithFlags(&ctx->ev2, cudaEventDisableTiming) == cudaSuccess &&
              cudaMalloc(&ctx->d_counters, sizeof(Counters)) == cudaSuccess &&
              cudaMallocHost(&ctx->h_counters, sizeof(Counters)) == cudaSuccess;
    if (!ok) {
        g_create_err = std::string("context setup failed: ") + cudaGetErrorString(cudaGetLastError());
        mm_destroy(ctx);
        return MM_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    memset(ctx->h_counters, 0, sizeof(Counters));
    g_create_err.clear();
    *out = ctx;
    return MM_OK;
}

int mm_destroy(mm_ctx *ctx) {
    if (!ctx) return MM_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_pairs); cudaFree(ctx->d_pairs_y); cudaFree(ctx->d_rects); cudaFree(ctx->d_rects_axis); cudaFree(ctx->d_shade); cudaFree(ctx->d_noise);
    cudaFree(ctx->d_chunks);
    cudaFree(ctx->d_counters); cudaFree(ctx->d_screen); cudaFree(ctx->d_screen2); cudaFree(ctx->d_dbg_rad);
    for (auto p : ctx->d_dbg_u32) cudaFree(p);
    cudaFree(ctx->d_tail_q); cudaFree(ctx->d_tail_pix);
    if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    cudaFree(ctx->d_screen8);
    cudaFree(ctx->d_snap);
    cudaFree(ctx->d_view_chunks); cudaFree(ctx->d_views);
    cudaFree(ctx->d_vscreen); cudaFree(ctx->d_vscreen2); cudaFree(ctx->d_vsnap); cudaFree(ctx->d_vscreen8);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->ev_snap) cudaEventDestroy(ctx->ev_snap);
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return MM_OK;
}

const char *mm_last_error(const mm_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int mm_upload_scene(mm_ctx *ctx, const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes,
                    const uint32_t *indices, const uint8_t *materials, const mm_float4 *emissions, const uint8_t *noise_rgba8,
                    uint32_t noise_w, uint32_t noise_h) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!planes || !nodes || !indices || !materials || !emissions || !noise_rgba8 || n_planes == 0 || n_nodes == 0 || noise_w == 0 ||
        noise_h == 0)
        return fail(ctx, MM_ERR_INVALID, "mm_upload_scene: null pointer or zero size");
    Prepared prep;
    std::string perr;
    int rc;
    try {
        rc = prepare_scene(planes, n_planes, nodes, n_nodes, indices, materials, emissions, prep, perr);
    } catch (...) {
        return fail(ctx, MM_ERR_NOMEM, "mm_upload_scene: out of host memory");
    }
    if (rc != MM_OK) return fail(ctx, rc, perr);
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_scene = false;
    cudaFree(ctx->d_pairs); cudaFree(ctx->d_pairs_y); cudaFree(ctx->d_rects); cudaFree(ctx->d_rects_axis); cudaFree(ctx->d_shade); cudaFree(ctx->d_noise);
    ctx->d_pairs = nullptr; ctx->d_pairs_y = nullptr; ctx->d_rects = nullptr; ctx->d_rects_axis = nullptr; ctx->d_shade = nullptr; ctx->d_noise = nullptr;
    ctx->n_yiv = 0;
    const size_t noise_bytes = (size_t)noise_w * noise_h * 4;
    // The kernel forms record addresses as {high word, low word + offset} (one 32-bit add, render_kernel.cu), so a pair
    // table must not straddle a 4-GB boundary.  An allocation that does is kept until a second one — which then cannot
    // cover the same boundary — has been made.
    auto alloc_window = [&](size_t bytes, void **out) -> int {
        void *first = nullptr, *second = nullptr;
        CK(cudaMalloc(&first, bytes));
        auto straddles = [&](void *p) {
            const uintptr_t a = reinterpret_cast<uintptr_t>(p);
            return (a >> 32) != ((a + bytes - 1) >> 32);
        };
        if (straddles(first)) {
            cudaError_t e = cudaMalloc(&second, bytes);
            cudaFree(first);
            if (e != cudaSuccess) return fail(ctx, MM_ERR_NOMEM, std::string("mm_upload_scene: ") + cudaGetErrorString(e));
            if (straddles(second)) { cudaFree(second); return fail(ctx, MM_ERR_CUDA, "mm_upload_scene: pair table straddles a 4-GB boundary"); }
            first = second;
        }
        *out = first;
        return MM_OK;
    };
    {
        void *p = nullptr;
        if ((rc = alloc_window(prep.pairs.size() * sizeof(PairRec), &p)) != MM_OK) return rc;
        ctx->d_pairs = static_cast<PairRec *>(p);
    }
    if (!prep.pairs_y.empty()) {
        const size_t rec_bytes = prep.pairs_y.size() * sizeof(PairRecY), iv_bytes = prep.y_ivals.size() * sizeof(float4);
        void *p = nullptr;
        if ((rc = alloc_window(rec_bytes + iv_bytes, &p)) != MM_OK) return rc;
        ctx->d_pairs_y = static_cast<PairRecY *>(p);
        CK(cudaMemcpyAsync(ctx->d_pairs_y, prep.pairs_y.data(), rec_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(static_cast<char *>(p) + rec_bytes, prep.y_ivals.data(), iv_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMalloc(&ctx->d_rects, prep.rects.size() * sizeof(RectI)));
    CK(cudaMalloc(&ctx->d_shade, prep.shade.size() * sizeof(RectS)));
    if (prep.axis_ok) {
        CK(cudaMalloc(&ctx->d_rects_axis, prep.rects_axis.size() * sizeof(RectA)));
        CK(cudaMemcpyAsync(ctx->d_rects_axis, prep.rects_axis.data(), prep.rects_axis.size() * sizeof(RectA), cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMalloc(&ctx->d_noise, noise_bytes));
    CK(cudaMemcpyAsync(ctx->d_pairs, prep.pairs.data(), prep.pairs.size() * sizeof(PairRec), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_rects, prep.rects.data(), prep.rects.size() * sizeof(RectI), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_shade, prep.shade.data(), prep.shade.size() * sizeof(RectS), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_noise, noise_rgba8, noise_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_pairs = prep.n_pairs; ctx->n_slots = n_planes; ctx->n_nodes = n_nodes;
    ctx->root_link = prep.root_link; ctx->root_count = prep.root_count;
    ctx->depth = prep.depth; ctx->max_leaf = prep.max_leaf; ctx->fast_ok = prep.fast_ok; ctx->rect_fast_ok = prep.rect_fast_ok;
    ctx->noise_w = noise_w; ctx->noise_h = noise_h;
    ctx->n_pairs_y = (uint32_t)prep.pairs_y.size();
    ctx->n_yiv = ctx->d_pairs_y ? (uint32_t)prep.y_ivals.size() : 0u;
    ctx->have_scene = true;
    return MM_OK;
}

int mm_set_chunks(mm_ctx *ctx, const mm_chunk *chunks, uint32_t n_chunks) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!chunks || n_chunks == 0) return fail(ctx, MM_ERR_INVALID, "mm_set_chunks: null or empty chunk list");
    CK(cudaSetDevice(ctx->device));
    if (n_chunks > ctx->chunks_cap) {
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_chunks);
        ctx->d_chunks = nullptr; ctx->chunks_cap = 0;
        CK(cudaMalloc(&ctx->d_chunks, (size_t)n_chunks * sizeof(mm_chunk)));
        ctx->chunks_cap = n_chunks;
    }
    CK(cudaMemcpyAsync(ctx->d_chunks, chunks, (size_t)n_chunks * sizeof(mm_chunk), cudaMemcpyHostToDevice, ctx->stream));
    ctx->n_chunks = n_chunks;
    return MM_OK;
}

}  // extern "C"

namespace mmapi {

static uint32_t env_u32(const char *name, uint32_t dflt, uint32_t lo, uint32_t hi) {
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    const long x = strtol(v, nullptr, 10);
    return x < (long)lo ? lo : (x > (long)hi ? hi : (uint32_t)x);
}

// The persistent ray-pool kernel (pool_kernel.cu; opt-in: MM_FLAG_POOL_KERNEL, or MM_KERNEL=pool in the environment for
// tuning runs) covers the common arithmetic mode: exact shared-reciprocal slab quotients, divide-free rect edge tests,
// spp <= 64.  Everything else (MM_FLAG_FORCE_LITERAL, MM_FLAG_RCP_SLAB, scenes outside the guarded coordinate / edge-length
// ranges, spp > 64) runs the default one-thread-per-path kernel whatever the flag says.  Geometry of a warp's
// pool: M path records of (24 + stack) words, five 128-byte ring queues, R pixel records of (4 + 3 spp) words.
// MM_POOL_M / MM_POOL_WARPS / MM_POOL_BLOCKS / MM_POOL_TH are developer overrides for tuning runs.
static bool configure_pool(mm_ctx *ctx, const mm_params *par, Launch &L) {
    KParams &p = L.p;
    const char *env_kernel = getenv("MM_KERNEL");
    const bool want = (par->flags & MM_FLAG_POOL_KERNEL) || (env_kernel && !strcmp(env_kernel, "pool"));
    if (!want || p.force_literal || p.rcp_mode || !p.scene_fast_ok || !p.rect_fast_ok ||
        p.spp > 64 || p.total_paths >= 0xFFFF0000ull || ctx->depth > 200)
        return false;
    const uint32_t stack_words = ((ctx->depth > 4 ? ctx->depth : 4) + 3u) & ~3u;     // occupancy <= depth - 1, plus the sentinel
    const uint32_t warps = env_u32("MM_POOL_WARPS", 1, 1, 4);
    uint32_t M = env_u32("MM_POOL_M", 96, 32, 128);
    const uint32_t SW = 24 + stack_words;
    uint32_t R = 0, region = 0;
    for (;; M -= 8) {                                                             // shrink the pool until the block fits the SM's shared memory
        R = (M + p.spp - 1) / p.spp + (32 + p.spp - 1) / p.spp + 3;
        region = (M * SW + 5 * 128 / 4 + R * (4 + 3 * p.spp) + 3u) & ~3u;
        if ((size_t)region * 4 * warps <= ctx->smem_optin || M <= 32) break;
    }
    if ((size_t)region * 4 * warps > ctx->smem_optin || R > 255) return false;
    p.pool_M = M; p.pool_slot_words = SW; p.pool_R = R; p.pool_region_words = region;
    p.pool_th_leaf = env_u32("MM_POOL_TH_LEAF", env_u32("MM_POOL_TH", 24, 1, 32), 1, 32);
    p.pool_th_shade = env_u32("MM_POOL_TH_SHADE", env_u32("MM_POOL_TH", 24, 1, 32), 1, 32);
    L.choice.pool = true;
    L.choice.block_threads = (int)(32 * warps);
    L.smem = (size_t)region * 4 * warps;
    L.blocks = 0;                                                                  // persistent grid: sized in do_launch from the occupancy query
    return true;
}

// The scene and flag part of a launch's parameters, shared by every render and by mm_trace_rays: the BVH root, the tables,
// and the arithmetic and rect form the traversal uses under flags (MM_FLAG_FORCE_LITERAL, MM_FLAG_RCP_SLAB,
// MM_FLAG_GENERAL_RECTS, MM_FLAG_NO_Y_TABLE).  Returns whether the y-table traversal applies (trace_ytab_kernel, DESIGN.md
// §3-4): it covers the exact slab arithmetic of scenes that have the table; MM_FLAG_NO_Y_TABLE keeps trace_kernel for
// comparisons.  The y-table fields are set only then.
bool traversal_params(const mm_ctx *ctx, uint32_t flags, KParams &p) {
    p.n_pairs = ctx->n_pairs; p.n_slots = ctx->n_slots;
    p.root_link = ctx->root_link; p.root_count = ctx->root_count;
    p.force_literal = (flags & MM_FLAG_FORCE_LITERAL) ? 1u : 0u;
    p.rcp_mode = (flags & MM_FLAG_RCP_SLAB) ? 1u : 0u;
    p.scene_fast_ok = ctx->fast_ok ? 1u : 0u;
    p.rect_fast_ok = (ctx->rect_fast_ok && !(flags & MM_FLAG_FORCE_LITERAL)) ? 1u : 0u;
    p.pairs = ctx->d_pairs; p.rects = ctx->d_rects; p.shade = ctx->d_shade;
    p.rects_axis = (p.rect_fast_ok && !(flags & MM_FLAG_GENERAL_RECTS)) ? ctx->d_rects_axis : nullptr;
    const bool ytab = ctx->n_yiv && !p.force_literal && !p.rcp_mode && p.scene_fast_ok && !(flags & MM_FLAG_NO_Y_TABLE);
    if (ytab) {
        p.pairs_y = ctx->d_pairs_y;
        p.y_ivals = reinterpret_cast<const float4 *>(ctx->d_pairs_y + ctx->n_pairs_y);
        p.n_yiv = ctx->n_yiv;
    }
    return ytab;
}

int build_launch(mm_ctx *ctx, const mm_uniform *uni, const mm_params *par, bool debug, Launch &L, uint32_t n_views) {
    if (!uni || !par) return fail(ctx, MM_ERR_INVALID, "null uniform or params");
    if (!ctx->have_scene) return fail(ctx, MM_ERR_NO_SCENE, "no scene uploaded");
    const uint32_t spp = par->spp, chunk = uni->chunk_width;
    if (spp == 0 || (spp & (spp - 1)) || spp > kMaxSpp) return fail(ctx, MM_ERR_UNSUPPORTED, "spp must be a power of two in 1..1024");
    if (chunk == 0 || chunk > 64) return fail(ctx, MM_ERR_UNSUPPORTED, "chunk_width must be in 1..64");
    const uint64_t T = (uint64_t)chunk * chunk * spp;
    if (T > (1u << 20)) return fail(ctx, MM_ERR_UNSUPPORTED, "chunk_width^2 * spp too large");
    if (T > 32 && (T % 32) != 0) return fail(ctx, MM_ERR_UNSUPPORTED, "chunk_width^2 * spp must be <= 32 or a multiple of 32 (virtual threadgroup = 32 x T/32)");
    if (par->grid_x == 0 || par->grid_y == 0) return fail(ctx, MM_ERR_INVALID, "empty grid");
    const uint64_t n_groups = (uint64_t)par->grid_x * par->grid_y;
    if (!n_views && n_groups != ctx->n_chunks) return fail(ctx, MM_ERR_INVALID, "grid_x*grid_y must equal the chunk count");
    if (par->bounce_limit > 4096 || par->mirror_limit > 4096) return fail(ctx, MM_ERR_INVALID, "bounce/mirror limit too large");
    if (!(uni->view_width >= 1.0f) || !(uni->view_height >= 1.0f) || uni->view_width > 65536.0f || uni->view_height > 65536.0f)
        return fail(ctx, MM_ERR_INVALID, "bad view size");
    uint32_t first = par->group_first, step = par->group_step ? par->group_step : 1, count = par->group_count;
    if (count == 0) { first = 0; step = 1; count = (uint32_t)n_groups; }
    if ((uint64_t)first + (uint64_t)(count - 1) * step >= n_groups) return fail(ctx, MM_ERR_INVALID, "group range outside the grid");

    KParams &p = L.p;
    memset(&p, 0, sizeof(p));
    p.uni = *uni;
    p.spp = spp;
    p.log2_spp = (uint32_t)__builtin_ctz(spp);
    p.bounce_limit = (int32_t)par->bounce_limit;
    p.mirror_limit = (int32_t)par->mirror_limit;
    p.grid_x = par->grid_x; p.grid_y = par->grid_y;
    p.group_first = first; p.group_step = step; p.group_count = count;
    p.T = (uint32_t)T;
    p.dim_x = p.T < 32 ? p.T : 32;
    p.dim_y = p.T / p.dim_x;
    p.ppc = chunk * chunk;
    p.W = (uint32_t)uni->view_width; p.H = (uint32_t)uni->view_height;
    p.noise_w = ctx->noise_w; p.noise_h = ctx->noise_h;
    const bool ytab = traversal_params(ctx, par->flags, p);
    p.quant8 = (par->flags & MM_FLAG_SCREEN_RGBA8) ? 1u : 0u;
    p.total_paths = (uint64_t)count * T * (n_views ? n_views : 1);
    p.chunks = n_views ? ctx->d_view_chunks : ctx->d_chunks; p.noise = ctx->d_noise;
    p.counters = ctx->d_counters;

    L.choice.debug = debug;
    L.choice.counters = debug || (par->flags & MM_FLAG_COUNTERS);
    L.choice.pool = false;
    L.choice.regroup = false;
    L.choice.ytab = false;
    L.choice.views = n_views != 0;
    L.views = n_views ? ctx->d_views : nullptr;
    // the multi-view kernels exist for the default kernel only (mm_render_views refuses the flags of the other two)
    if (!n_views && configure_pool(ctx, par, L)) return MM_OK;
    // opt-in (MM_FLAG_REGROUP, or MM_KERNEL=regroup for tuning runs): the kernel that re-forms the block's warps at segment
    // boundaries.  Its largest block is kLargeBlock, so above spp 256 the default kernel runs whatever the flag says.
    const char *env_kernel = getenv("MM_KERNEL");
    L.choice.regroup = !n_views && p.spp <= (uint32_t)kLargeBlock && ((par->flags & MM_FLAG_REGROUP) || (env_kernel && !strcmp(env_kernel, "regroup")));
    int bt = block_threads_for(p.spp);
    if (L.choice.regroup) {
        const int want = (int)env_u32("MM_RG_BLOCK", kLargeBlock, 64, kLargeBlock);       // developer override: 64 / 128 / 256
        bt = want >= 256 ? 256 : (want >= 128 ? 128 : 64);
        if ((uint32_t)bt < p.spp) bt = kLargeBlock;                                       // a block holds whole pixels
        const char *m = getenv("MM_RG_MASK");
        p.rg_mask = m && *m ? (uint32_t)strtoul(m, nullptr, 0) : 0xFFFFFFFFu;
    }
    L.choice.block_threads = bt;
    // Straggler tail (render_kernel.cu): the default kernel queues the paths of warps past bounce_limit segments with at most
    // kTailK live lanes, and trace_tail_kernel runs them densely.  The queue holds an eighth of the frame's paths (a replay
    // of the 1080p 16-spp frame queues 6 %, profiles/r3_tail_replay.txt) within kTailBudget; paths past it stay in their
    // warp.  MM_TAIL_K / MM_TAIL_CAP are developer overrides for tuning runs and tests.
    if (!L.choice.regroup && !(par->flags & MM_FLAG_NO_TAIL) && (p.total_paths >> p.log2_spp) < (1ull << 32)) {
        constexpr uint32_t kTailK = 8;
        constexpr size_t kTailBudget = size_t(1) << 30;
        const size_t pix_bytes = (4 + 3 * (size_t)spp) * sizeof(float);
        uint64_t cap = p.total_paths / 8 + 1024;
        if (cap > kTailBudget / (sizeof(TailPath) + pix_bytes)) cap = kTailBudget / (sizeof(TailPath) + pix_bytes);
        cap = std::min<uint64_t>(cap, env_u32("MM_TAIL_CAP", 0xFFFFFFFFu, 0, 0xFFFFFFFFu));
        const uint64_t pixels = std::min<uint64_t>(cap, p.total_paths >> p.log2_spp);   // a deferred pixel has a queued path
        if (cap && (ctx->tail_q_cap < cap || ctx->tail_pix_bytes < pixels * pix_bytes)) {
            CK(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_tail_q); cudaFree(ctx->d_tail_pix);
            ctx->d_tail_q = nullptr; ctx->d_tail_pix = nullptr; ctx->tail_q_cap = 0; ctx->tail_pix_bytes = 0;
            CK(cudaMalloc(&ctx->d_tail_q, cap * sizeof(TailPath)));
            CK(cudaMalloc(&ctx->d_tail_pix, pixels * pix_bytes));
            ctx->tail_q_cap = cap; ctx->tail_pix_bytes = pixels * pix_bytes;
        }
        p.tail_k = cap ? env_u32("MM_TAIL_K", kTailK, 0, 32) : 0u;
        p.tail_cap = (uint32_t)cap;
        p.tail_q = ctx->d_tail_q;
        p.tail_pix = ctx->d_tail_pix;
    }
    L.choice.ytab = !L.choice.regroup && ytab;
    L.smem = 3 * (size_t)bt * sizeof(float);                             // reduction scratch
    if (L.choice.ytab) L.smem += (size_t)(bt / 32) * p.n_yiv * kYEntryStride;                 // y-table: [warp][interval][lane]
    if (L.choice.regroup) L.smem += 4 * (size_t)bt * sizeof(float4) + 64 * sizeof(uint32_t);   // path state in flight + bin counters
    const uint64_t blocks = (p.total_paths + (uint64_t)bt - 1) / (uint64_t)bt;
    if (blocks > 0x7FFFFFFFull) return fail(ctx, MM_ERR_UNSUPPORTED, "too many paths for one launch");
    L.blocks = (unsigned)blocks;
    return MM_OK;
}

int do_launch(mm_ctx *ctx, Launch &L) {
    const void *fn = L.choice.pool ? pool_kernel_ptr(L.choice) : kernel_ptr(L.choice);
    if (fn != ctx->cfg_fn || L.smem != ctx->cfg_smem) {   // once per kernel variant, not per frame
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, L.choice.block_threads, L.smem));
        ctx->last_blocks_per_sm = (uint32_t)per_sm;
        ctx->cfg_fn = fn; ctx->cfg_smem = L.smem;
    }
    ctx->last_smem = (uint32_t)L.smem; ctx->last_block_threads = (uint32_t)L.choice.block_threads;
    ctx->last_tail_cap = L.p.tail_k ? L.p.tail_cap : 0u;
    ctx->last_y_table = L.choice.ytab ? L.p.n_yiv : 0u;
    CK(cudaMemsetAsync(ctx->d_counters, 0, sizeof(Counters), ctx->stream));
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (L.choice.pool) {
        uint32_t per_sm = ctx->last_blocks_per_sm ? ctx->last_blocks_per_sm : 1u;
        const uint32_t cap = env_u32("MM_POOL_BLOCKS", 0, 0, 64);
        if (cap && cap < per_sm) per_sm = cap;
        const uint64_t unit = L.p.spp > 32 ? L.p.spp : 32, units = (L.p.total_paths + unit - 1) / unit;
        uint64_t blocks = (uint64_t)ctx->n_sms * per_sm;
        const uint64_t want = (units + (uint64_t)(L.choice.block_threads / 32) - 1) / (uint64_t)(L.choice.block_threads / 32);
        if (blocks > want) blocks = want ? want : 1;                                 // tiny dispatches: no more warps than units
        CK(launch_pool(L.p, L.choice, (unsigned)blocks, (unsigned)L.choice.block_threads, L.smem, ctx->stream));
    } else {
        CK(launch_trace(L.p, L.choice, L.blocks, L.smem, ctx->stream, L.views));
        if (L.p.tail_k) {                 // one thread per queued path; the grid strides over whatever the queue holds
            const uint64_t want = ((uint64_t)L.p.tail_cap + kTailBlock - 1) / kTailBlock, full = (uint64_t)ctx->n_sms * (1024 / kTailBlock);
            const size_t tail_smem = L.choice.ytab ? (size_t)(kTailBlock / 32) * L.p.n_yiv * kYEntryStride : 0;
            CK(launch_tail(L.p, L.choice, (unsigned)(want < full ? want : full), tail_smem, ctx->stream, L.views));
        }
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev2, ctx->stream));      // mm_last_counters waits on this, not on the whole stream
    ctx->timed = true;
    return MM_OK;
}

int ensure_screen(mm_ctx *ctx, uint32_t W, uint32_t H) {
    if (ctx->d_screen && ctx->screen_w == W && ctx->screen_h == H) return MM_OK;
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->d_screen);
    cudaFree(ctx->d_screen2);
    cudaFree(ctx->d_screen8);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    cudaFree(ctx->d_snap);
    ctx->d_screen = nullptr; ctx->d_screen2 = nullptr; ctx->d_screen8 = nullptr; ctx->d_snap = nullptr;
    CK(cudaMalloc(&ctx->d_screen, (size_t)W * H * 4 * sizeof(float)));
    CK(cudaMemsetAsync(ctx->d_screen, 0, (size_t)W * H * 4 * sizeof(float), ctx->stream));
    ctx->screen_w = W; ctx->screen_h = H;
    return MM_OK;
}

// Device per-path debug arrays for n_paths paths, and the kernel's pointers to those the caller asked for.
static int setup_debug(mm_ctx *ctx, const mm_debug *debug, size_t n_paths, KParams &p) {
    if (n_paths > ctx->dbg_cap) {
        CK(cudaStreamSynchronize(ctx->stream));
        for (auto &q : ctx->d_dbg_u32) { cudaFree(q); q = nullptr; }
        cudaFree(ctx->d_dbg_rad); ctx->d_dbg_rad = nullptr; ctx->dbg_cap = 0;
        for (auto &q : ctx->d_dbg_u32) CK(cudaMalloc(&q, n_paths * sizeof(uint32_t)));
        CK(cudaMalloc(&ctx->d_dbg_rad, n_paths * 3 * sizeof(float)));
        ctx->dbg_cap = n_paths;
    }
    p.dbg_first_hit = debug->first_hit ? ctx->d_dbg_u32[0] : nullptr;
    p.dbg_segments = debug->segments ? ctx->d_dbg_u32[1] : nullptr;
    p.dbg_mirror_hits = debug->mirror_hits ? ctx->d_dbg_u32[2] : nullptr;
    p.dbg_radiance = debug->radiance ? ctx->d_dbg_rad : nullptr;
    return MM_OK;
}

// The read-back of the debug arrays into the caller's host arrays, on the context's stream.
static int copy_debug(mm_ctx *ctx, const mm_debug *debug, size_t n_paths) {
    if (debug->first_hit) CK(cudaMemcpyAsync(debug->first_hit, ctx->d_dbg_u32[0], n_paths * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (debug->segments) CK(cudaMemcpyAsync(debug->segments, ctx->d_dbg_u32[1], n_paths * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (debug->mirror_hits) CK(cudaMemcpyAsync(debug->mirror_hits, ctx->d_dbg_u32[2], n_paths * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (debug->radiance) CK(cudaMemcpyAsync(debug->radiance, ctx->d_dbg_rad, n_paths * 12, cudaMemcpyDeviceToHost, ctx->stream));
    return MM_OK;
}

// The pinned staging buffer for callers whose frame memory is not known to be pinned, at least `bytes` long.
static int ensure_stage(mm_ctx *ctx, size_t bytes) {
    if (ctx->stage_bytes >= bytes) return MM_OK;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    ctx->h_stage = nullptr; ctx->stage_bytes = 0;
    CK(cudaMallocHost(&ctx->h_stage, bytes));
    ctx->stage_bytes = bytes;
    return MM_OK;
}

// The second stream and its events of the asynchronous present, created at first use.
static int ensure_copy_stream(mm_ctx *ctx) {
    if (ctx->copy_stream) return MM_OK;
    CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->ev_snap, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming));
    return MM_OK;
}

void counters_out(const Counters *h, mm_counters *o) {
    o->paths = h->paths; o->rays = h->rays; o->inner_visits = h->inner_visits; o->leaf_visits = h->leaf_visits;
    o->rect_tests = h->rect_tests; o->hits = h->hits; o->literal_rays = h->literal_rays; o->max_stack = h->max_stack;
}

}  // namespace mmapi
using namespace mmapi;

extern "C" {

int mm_render_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, float *d_image, float *d_tiles) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!d_image && !d_tiles) return fail(ctx, MM_ERR_INVALID, "mm_render_device: both outputs are null");
    CK(cudaSetDevice(ctx->device));
    Launch L;
    int rc = build_launch(ctx, uni, params, false, L);
    if (rc != MM_OK) return rc;
    L.p.image = d_image;
    L.p.tiles = d_tiles;
    return do_launch(ctx, L);
}

int mm_render_multicast_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, float *mc_frame) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!mc_frame) return fail(ctx, MM_ERR_INVALID, "mm_render_multicast_device: null multicast address");
    CK(cudaSetDevice(ctx->device));
    Launch L;
    int rc = build_launch(ctx, uni, params, false, L);
    if (rc != MM_OK) return rc;
    L.p.n_peers = 1;
    L.p.peers[0] = mc_frame;
    L.p.peers_multicast = 1;
    return do_launch(ctx, L);
}

int mm_render_peers_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, float *const *frames, uint32_t n_frames) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!frames || n_frames == 0 || n_frames > MM_MAX_PEERS) return fail(ctx, MM_ERR_INVALID, "mm_render_peers_device: 1..MM_MAX_PEERS frames");
    for (uint32_t i = 0; i < n_frames; i++)
        if (!frames[i]) return fail(ctx, MM_ERR_INVALID, "mm_render_peers_device: null frame pointer");
    CK(cudaSetDevice(ctx->device));
    Launch L;
    int rc = build_launch(ctx, uni, params, false, L);
    if (rc != MM_OK) return rc;
    L.p.image = nullptr;
    L.p.tiles = nullptr;
    L.p.n_peers = n_frames;
    for (uint32_t i = 0; i < n_frames; i++) L.p.peers[i] = frames[i];
    return do_launch(ctx, L);
}

/* ---- pinned host memory the kernel can write into directly ------------------------------------------------------------ */

int mm_host_alloc(size_t bytes, void **out) {
    if (!out || bytes == 0) return MM_ERR_INVALID;
    *out = nullptr;
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return MM_ERR_NOMEM; }
    void *d = nullptr;
    if (cudaHostGetDevicePointer(&d, p, 0) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(p); return MM_ERR_CUDA; }
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        g_host.push_back({reinterpret_cast<uintptr_t>(p), bytes, true, reinterpret_cast<uintptr_t>(d)});
    }
    *out = p;
    return MM_OK;
}

int mm_host_register(void *ptr, size_t bytes) {
    if (!ptr || bytes == 0) return MM_ERR_INVALID;
    if (cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped) != cudaSuccess) { cudaGetLastError(); return MM_ERR_CUDA; }
    void *d = nullptr;
    if (cudaHostGetDevicePointer(&d, ptr, 0) != cudaSuccess) { cudaGetLastError(); cudaHostUnregister(ptr); return MM_ERR_CUDA; }
    std::lock_guard<std::mutex> lock(g_host_mu);
    g_host.push_back({reinterpret_cast<uintptr_t>(ptr), bytes, false, reinterpret_cast<uintptr_t>(d)});
    return MM_OK;
}

static int host_release(void *ptr, bool owned) {
    if (!ptr) return MM_OK;
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        size_t i = 0;
        for (; i < g_host.size(); i++)
            if (g_host[i].base == reinterpret_cast<uintptr_t>(ptr) && g_host[i].owned == owned) break;
        if (i == g_host.size()) return MM_ERR_INVALID;
        g_host.erase(g_host.begin() + (long)i);
    }
    cudaError_t e = owned ? cudaFreeHost(ptr) : cudaHostUnregister(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return MM_ERR_CUDA; }
    return MM_OK;
}
int mm_host_free(void *ptr) { return host_release(ptr, true); }
int mm_host_unregister(void *ptr) { return host_release(ptr, false); }

/* ---- host-buffer frames ------------------------------------------------------------------------------------------------ */

int mm_wait(mm_ctx *ctx, mm_counters *counters) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->pending_out) {                              // staged frame: pinned staging -> the caller's (pageable) buffer
        memcpy(ctx->pending_out, ctx->h_stage, ctx->pending_bytes);
        ctx->pending_out = nullptr;
    }
    for (uint32_t v = 0; v < MM_MAX_VIEWS; v++) {          // staged views of mm_render_views_async
        if (!ctx->pending_views[v]) continue;
        memcpy(ctx->pending_views[v], reinterpret_cast<const char *>(ctx->h_stage) + v * ctx->pending_bytes, ctx->pending_bytes);
        ctx->pending_views[v] = nullptr;
    }
    ctx->in_flight = false;
    if (counters) {
        if (!ctx->timed) return fail(ctx, MM_ERR_INVALID, "mm_wait: nothing rendered yet");
        counters_out(ctx->h_counters, counters);
    }
    return MM_OK;
}

int mm_render_async(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, const mm_chunk *chunks, uint32_t n_chunks,
                    float *out_rgba, const mm_debug *debug) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    int rc;
    CK(cudaSetDevice(ctx->device));
    if (ctx->in_flight && (rc = mm_wait(ctx, nullptr)) != MM_OK) return rc;     // one host-buffer frame in flight per context
    if (chunks) {
        if ((rc = mm_set_chunks(ctx, chunks, n_chunks)) != MM_OK) return rc;
    } else if (ctx->n_chunks == 0) {
        return fail(ctx, MM_ERR_INVALID, "mm_render: null chunk list and none set earlier");
    }
    const bool dbg = debug && (debug->first_hit || debug->segments || debug->mirror_hits || debug->radiance);
    Launch L;
    rc = build_launch(ctx, uni, params, dbg, L);
    if (rc != MM_OK) return rc;
    rc = ensure_screen(ctx, L.p.W, L.p.H);
    if (rc != MM_OK) return rc;
    L.p.image = ctx->d_screen;
    const size_t frame_bytes = (size_t)L.p.W * L.p.H * 4 * sizeof(float);
    // Zero-copy output: a caller buffer inside mapped pinned memory (mm_host_alloc / mm_host_register) is written by the
    // kernel itself, pixel by pixel over PCIe while it traces; no screen copy follows.
    void *pinned = out_rgba ? host_device_alias(out_rgba, frame_bytes) : nullptr;
    void *alias = (params->flags & MM_FLAG_NO_ZERO_COPY) ? nullptr : pinned;
    L.p.host_out = static_cast<float *>(alias);
    ctx->last_zero_copy = alias ? 1u : 0u;
    const size_t n_paths = (size_t)L.p.total_paths;
    if (dbg && (rc = setup_debug(ctx, debug, n_paths, L.p)) != MM_OK) return rc;
    const bool staged = out_rgba && !pinned;
    if (staged && (rc = ensure_stage(ctx, frame_bytes)) != MM_OK) return rc;
    rc = do_launch(ctx, L);
    if (rc != MM_OK) return rc;
    ctx->in_flight = true;
    if (out_rgba && !alias) {
        // the whole persistent screen: DMA into the caller's pinned buffer, or into the library's pinned staging buffer
        // when the caller's memory is not known to be pinned (copied on to it by mm_wait)
        float *dst = staged ? ctx->h_stage : out_rgba;
        CK(cudaMemcpyAsync(dst, ctx->d_screen, frame_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        if (staged) { ctx->pending_out = out_rgba; ctx->pending_bytes = frame_bytes; }
    }
    if (dbg) return copy_debug(ctx, debug, n_paths);
    return MM_OK;
}

int mm_render(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, const mm_chunk *chunks, uint32_t n_chunks,
              float *out_rgba, mm_counters *counters, const mm_debug *debug) {
    int rc = mm_render_async(ctx, uni, params, chunks, n_chunks, out_rgba, debug);
    if (rc != MM_OK) return rc;
    return mm_wait(ctx, counters);
}

/* ---- several views in one launch -------------------------------------------------------------------------------------- */

namespace mmapi {
// The persistent view screens: n screens of W x H, zero-filled whenever n or the size changes.
static int ensure_view_screens(mm_ctx *ctx, uint32_t n, uint32_t W, uint32_t H) {
    if (ctx->d_vscreen && ctx->vscreen_n == n && ctx->vscreen_w == W && ctx->vscreen_h == H) return MM_OK;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->copy_stream) CK(cudaStreamSynchronize(ctx->copy_stream));
    cudaFree(ctx->d_vscreen); cudaFree(ctx->d_vscreen2); cudaFree(ctx->d_vsnap); cudaFree(ctx->d_vscreen8);
    ctx->d_vscreen = nullptr; ctx->d_vscreen2 = nullptr; ctx->d_vsnap = nullptr; ctx->d_vscreen8 = nullptr;
    ctx->vscreen_n = 0;
    const size_t bytes = (size_t)n * W * H * 4 * sizeof(float);
    CK(cudaMalloc(&ctx->d_vscreen, bytes));
    CK(cudaMemsetAsync(ctx->d_vscreen, 0, bytes, ctx->stream));
    ctx->vscreen_n = n; ctx->vscreen_w = W; ctx->vscreen_h = H;
    return MM_OK;
}
}  // namespace mmapi

int mm_render_views_async(mm_ctx *ctx, const mm_uniform *unis, uint32_t n_views, const mm_params *params, const mm_chunk *chunks,
                          uint32_t n_chunks, float *const *out_rgba, const mm_debug *debug) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!unis || !params || !chunks) return fail(ctx, MM_ERR_INVALID, "mm_render_views: null uniforms, params or chunk list");
    if (n_views == 0 || n_views > MM_MAX_VIEWS) return fail(ctx, MM_ERR_INVALID, "mm_render_views: n_views must be in 1..MM_MAX_VIEWS");
    if (params->flags & (MM_FLAG_POOL_KERNEL | MM_FLAG_REGROUP))
        return fail(ctx, MM_ERR_UNSUPPORTED, "mm_render_views: MM_FLAG_POOL_KERNEL and MM_FLAG_REGROUP have no multi-view kernel");
    for (uint32_t v = 1; v < n_views; v++)
        if (unis[v].view_width != unis[0].view_width || unis[v].view_height != unis[0].view_height || unis[v].chunk_width != unis[0].chunk_width)
            return fail(ctx, MM_ERR_INVALID, "mm_render_views: every view must have the same view size and chunk width");
    const uint64_t n_groups = (uint64_t)params->grid_x * params->grid_y;
    if (n_groups == 0 || (uint64_t)n_chunks != n_groups * n_views)
        return fail(ctx, MM_ERR_INVALID, "mm_render_views: n_chunks must equal n_views*grid_x*grid_y");
    int rc;
    CK(cudaSetDevice(ctx->device));
    if (ctx->in_flight && (rc = mm_wait(ctx, nullptr)) != MM_OK) return rc;     // one host-buffer frame in flight per context
    if (!ctx->d_views) CK(cudaMalloc(&ctx->d_views, MM_MAX_VIEWS * sizeof(ViewRec)));
    if (n_chunks > ctx->view_chunks_cap) {
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_view_chunks);
        ctx->d_view_chunks = nullptr; ctx->view_chunks_cap = 0;
        CK(cudaMalloc(&ctx->d_view_chunks, (size_t)n_chunks * sizeof(mm_chunk)));
        ctx->view_chunks_cap = n_chunks;
    }
    const bool dbg = debug && (debug->first_hit || debug->segments || debug->mirror_hits || debug->radiance);
    Launch L;
    rc = build_launch(ctx, unis, params, dbg, L, n_views);
    if (rc != MM_OK) return rc;
    const uint32_t W = L.p.W, H = L.p.H;
    rc = ensure_view_screens(ctx, n_views, W, H);
    if (rc != MM_OK) return rc;
    const size_t frame_floats = (size_t)W * H * 4, frame_bytes = frame_floats * sizeof(float);
    // Per view: zero-copy into a mapped pinned host frame (the kernel stores the view's pixels), a DMA copy of the view's
    // screen into other pinned memory, or one through the pinned staging buffer for pageable memory (as mm_render_async).
    ViewRec rec[MM_MAX_VIEWS];
    bool copy[MM_MAX_VIEWS] = {}, staged[MM_MAX_VIEWS] = {}, any_staged = false;
    uint32_t zero_copy = 0;
    for (uint32_t v = 0; v < n_views; v++) {
        float *out = out_rgba ? out_rgba[v] : nullptr;
        void *pinned = out ? host_device_alias(out, frame_bytes) : nullptr;
        void *alias = (params->flags & MM_FLAG_NO_ZERO_COPY) ? nullptr : pinned;
        memset(&rec[v], 0, sizeof(ViewRec));
        rec[v].uni = unis[v];
        rec[v].chunk_off = (uint32_t)(v * n_groups);
        rec[v].screen = ctx->d_vscreen + v * frame_floats;
        rec[v].host_out = static_cast<float *>(alias);
        copy[v] = out && !alias;
        staged[v] = out && !pinned;
        any_staged = any_staged || staged[v];
        zero_copy |= alias ? 1u : 0u;
    }
    const size_t n_paths = (size_t)L.p.total_paths;
    if (dbg && (rc = setup_debug(ctx, debug, n_paths, L.p)) != MM_OK) return rc;
    if (any_staged && (rc = ensure_stage(ctx, n_views * frame_bytes)) != MM_OK) return rc;
    CK(cudaMemcpyAsync(ctx->d_view_chunks, chunks, (size_t)n_chunks * sizeof(mm_chunk), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_views, rec, n_views * sizeof(ViewRec), cudaMemcpyHostToDevice, ctx->stream));
    ctx->last_zero_copy = zero_copy;
    rc = do_launch(ctx, L);
    if (rc != MM_OK) return rc;
    ctx->in_flight = true;
    for (uint32_t v = 0; v < n_views; v++) {
        if (!copy[v]) continue;
        float *dst = staged[v] ? ctx->h_stage + v * frame_floats : out_rgba[v];
        CK(cudaMemcpyAsync(dst, rec[v].screen, frame_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        if (staged[v]) { ctx->pending_views[v] = out_rgba[v]; ctx->pending_bytes = frame_bytes; }
    }
    if (dbg) return copy_debug(ctx, debug, n_paths);
    return MM_OK;
}

int mm_render_views(mm_ctx *ctx, const mm_uniform *unis, uint32_t n_views, const mm_params *params, const mm_chunk *chunks,
                    uint32_t n_chunks, float *const *out_rgba, mm_counters *counters, const mm_debug *debug) {
    int rc = mm_render_views_async(ctx, unis, n_views, params, chunks, n_chunks, out_rgba, debug);
    if (rc != MM_OK) return rc;
    return mm_wait(ctx, counters);
}

int mm_present_views(mm_ctx *ctx, uint32_t rgba8, void *const *out) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->d_vscreen) return fail(ctx, MM_ERR_INVALID, "mm_present_views: no views rendered yet");
    if (rgba8 > 1) return fail(ctx, MM_ERR_INVALID, "mm_present_views: rgba8 must be 0 or 1");
    const uint32_t n = ctx->vscreen_n;
    const size_t n_px = (size_t)ctx->vscreen_w * ctx->vscreen_h, screen_bytes = n_px * 4 * sizeof(float);
    const size_t out_bytes = rgba8 ? n_px * 4 : screen_bytes;
    bool any_out = false;
    for (uint32_t v = 0; out && v < n; v++) {
        if (!out[v]) continue;
        if (!host_device_alias(out[v], out_bytes))
            return fail(ctx, MM_ERR_INVALID, "mm_present_views: out[v] must be pinned host memory (mm_host_alloc / mm_host_register)");
        any_out = true;
    }
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_copy_stream(ctx);
    if (rc != MM_OK) return rc;
    if (!ctx->d_vscreen2) CK(cudaMalloc(&ctx->d_vscreen2, n * screen_bytes));
    if (rgba8 && !ctx->d_vscreen8) CK(cudaMalloc(&ctx->d_vscreen8, n * n_px * 4));
    if (!rgba8 && any_out && !ctx->d_vsnap) CK(cudaMalloc(&ctx->d_vsnap, n * screen_bytes));
    if (rgba8 && ctx->present_in_flight) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));   // the previous texels have left the device
    CK(launch_blur_views(ctx->d_vscreen, ctx->d_vscreen2, ctx->vscreen_w, ctx->vscreen_h, n, ctx->stream, rgba8 != 0,
                         rgba8 ? ctx->d_vscreen8 : nullptr));
    float *t = ctx->d_vscreen; ctx->d_vscreen = ctx->d_vscreen2; ctx->d_vscreen2 = t;   // the blurred images are the screens now
    if (!any_out) return MM_OK;
    if (!rgba8) {
        // snapshot for the read-back: the next dispatch may write into the screens while the copies are still on the wire
        if (ctx->present_in_flight) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));   // the previous snapshot has left the device
        for (uint32_t v = 0; v < n; v++)
            if (out[v]) CK(cudaMemcpyAsync(ctx->d_vsnap + v * n_px * 4, ctx->d_vscreen + v * n_px * 4, screen_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CK(cudaEventRecord(ctx->ev_snap, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_snap, 0));
    for (uint32_t v = 0; v < n; v++) {
        if (!out[v]) continue;
        const void *src = rgba8 ? static_cast<const void *>(ctx->d_vscreen8 + v * n_px * 4) : static_cast<const void *>(ctx->d_vsnap + v * n_px * 4);
        CK(cudaMemcpyAsync(out[v], src, out_bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
    }
    CK(cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    ctx->present_in_flight = true;
    return MM_OK;
}

int mm_scatter_tiles_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, const float *d_tiles, float *d_image) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!uni || !params || !d_tiles || !d_image) return fail(ctx, MM_ERR_INVALID, "mm_scatter_tiles_device: null argument");
    if (!ctx->d_chunks) return fail(ctx, MM_ERR_INVALID, "mm_scatter_tiles_device: no chunk list set");
    const uint64_t n_groups = (uint64_t)params->grid_x * params->grid_y;
    if (n_groups != ctx->n_chunks) return fail(ctx, MM_ERR_INVALID, "grid_x*grid_y must equal the chunk count");
    uint32_t first = params->group_first, step = params->group_step ? params->group_step : 1, count = params->group_count;
    if (count == 0) { first = 0; step = 1; count = (uint32_t)n_groups; }
    if ((uint64_t)first + (uint64_t)(count - 1) * step >= n_groups) return fail(ctx, MM_ERR_INVALID, "group range outside the grid");
    CK(cudaSetDevice(ctx->device));
    CK(launch_scatter(d_tiles, d_image, ctx->d_chunks, (uint32_t)n_groups, first, step, count, uni->chunk_width, (uint32_t)uni->view_width,
                      (uint32_t)uni->view_height, ctx->stream));
    return MM_OK;
}

int mm_scatter_gathered_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, uint32_t world, uint32_t max_count,
                               const float *d_gathered, float *d_image) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!uni || !params || !d_gathered || !d_image || world == 0 || max_count == 0)
        return fail(ctx, MM_ERR_INVALID, "mm_scatter_gathered_device: bad argument");
    if (!ctx->d_chunks) return fail(ctx, MM_ERR_INVALID, "mm_scatter_gathered_device: no chunk list set");
    const uint64_t n_groups = (uint64_t)params->grid_x * params->grid_y;
    if (n_groups != ctx->n_chunks) return fail(ctx, MM_ERR_INVALID, "grid_x*grid_y must equal the chunk count");
    if ((uint64_t)world * max_count < n_groups) return fail(ctx, MM_ERR_INVALID, "gathered buffer smaller than the grid");
    CK(cudaSetDevice(ctx->device));
    CK(launch_scatter_all(d_gathered, d_image, ctx->d_chunks, world, max_count, (uint32_t)n_groups, uni->chunk_width,
                          (uint32_t)uni->view_width, (uint32_t)uni->view_height, ctx->stream));
    return MM_OK;
}

int mm_sync(mm_ctx *ctx) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return MM_OK;
}

int mm_set_stream(mm_ctx *ctx, void *stream) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stream = stream ? (cudaStream_t)stream : ctx->own_stream;
    return MM_OK;
}

int mm_present_blur_device(mm_ctx *ctx, const float *d_src, float *d_dst, uint32_t width, uint32_t height) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!d_src || !d_dst || d_src == d_dst || width == 0 || height == 0) return fail(ctx, MM_ERR_INVALID, "mm_present_blur_device: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(launch_blur(d_src, d_dst, width, height, ctx->stream));
    return MM_OK;
}

static int present_impl(mm_ctx *ctx, float *out_rgba, bool q8, uint8_t *out_rgba8) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->d_screen) return fail(ctx, MM_ERR_INVALID, "mm_present: nothing rendered yet");
    CK(cudaSetDevice(ctx->device));
    const size_t n_px = (size_t)ctx->screen_w * ctx->screen_h, bytes = n_px * 4 * sizeof(float);
    if (!ctx->d_screen2) CK(cudaMalloc(&ctx->d_screen2, bytes));
    if (out_rgba8 && !ctx->d_screen8) CK(cudaMalloc(&ctx->d_screen8, n_px * 4));
    if (out_rgba8 && ctx->present_in_flight) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));   // mm_present_async_rgba8's texels have left the device
    CK(launch_blur(ctx->d_screen, ctx->d_screen2, ctx->screen_w, ctx->screen_h, ctx->stream, q8, out_rgba8 ? ctx->d_screen8 : nullptr));
    float *t = ctx->d_screen; ctx->d_screen = ctx->d_screen2; ctx->d_screen2 = t;   // the blurred image is the screen now
    if (out_rgba) CK(cudaMemcpyAsync(out_rgba, ctx->d_screen, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_rgba8) CK(cudaMemcpyAsync(out_rgba8, ctx->d_screen8, n_px * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return MM_OK;
}
int mm_present(mm_ctx *ctx, float *out_rgba) { return present_impl(ctx, out_rgba, false, nullptr); }

int mm_wait_present(mm_ctx *ctx) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->present_in_flight) return MM_OK;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventSynchronize(ctx->ev_copy));
    ctx->present_in_flight = false;
    return MM_OK;
}

int mm_present_async_rgba8(mm_ctx *ctx, uint8_t *out_rgba8) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->d_screen) return fail(ctx, MM_ERR_INVALID, "mm_present_async_rgba8: nothing rendered yet");
    const size_t n_px = (size_t)ctx->screen_w * ctx->screen_h, bytes = n_px * 4 * sizeof(float);
    if (!out_rgba8 || !host_device_alias(out_rgba8, n_px * 4))
        return fail(ctx, MM_ERR_INVALID, "mm_present_async_rgba8: out_rgba8 must be pinned host memory (mm_host_alloc / mm_host_register)");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_copy_stream(ctx);
    if (rc != MM_OK) return rc;
    if (!ctx->d_screen2) CK(cudaMalloc(&ctx->d_screen2, bytes));
    if (!ctx->d_screen8) CK(cudaMalloc(&ctx->d_screen8, n_px * 4));
    if (ctx->present_in_flight) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));       // the previous texels have left the device
    CK(launch_blur(ctx->d_screen, ctx->d_screen2, ctx->screen_w, ctx->screen_h, ctx->stream, true, ctx->d_screen8));
    float *t = ctx->d_screen; ctx->d_screen = ctx->d_screen2; ctx->d_screen2 = t;   // the blurred, quantised image is the screen now
    CK(cudaEventRecord(ctx->ev_snap, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_snap, 0));
    CK(cudaMemcpyAsync(out_rgba8, ctx->d_screen8, n_px * 4, cudaMemcpyDeviceToHost, ctx->copy_stream));   // the texel buffer is not the screen: no snapshot
    CK(cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    ctx->present_in_flight = true;
    return MM_OK;
}

int mm_present_async(mm_ctx *ctx, float *out_rgba) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->d_screen) return fail(ctx, MM_ERR_INVALID, "mm_present_async: nothing rendered yet");
    const size_t bytes = (size_t)ctx->screen_w * ctx->screen_h * 4 * sizeof(float);
    if (!out_rgba || !host_device_alias(out_rgba, bytes))
        return fail(ctx, MM_ERR_INVALID, "mm_present_async: out_rgba must be pinned host memory (mm_host_alloc / mm_host_register); use mm_present otherwise");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_copy_stream(ctx);
    if (rc != MM_OK) return rc;
    if (!ctx->d_screen2) CK(cudaMalloc(&ctx->d_screen2, bytes));
    if (!ctx->d_snap) CK(cudaMalloc(&ctx->d_snap, bytes));
    CK(launch_blur(ctx->d_screen, ctx->d_screen2, ctx->screen_w, ctx->screen_h, ctx->stream));
    float *t = ctx->d_screen; ctx->d_screen = ctx->d_screen2; ctx->d_screen2 = t;   // the blurred image is the screen now
    // snapshot for the read-back: the next dispatch may write into the screen while the copy is still on the wire
    if (ctx->present_in_flight) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));       // the previous snapshot has left the device
    CK(cudaMemcpyAsync(ctx->d_snap, ctx->d_screen, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaEventRecord(ctx->ev_snap, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_snap, 0));
    CK(cudaMemcpyAsync(out_rgba, ctx->d_snap, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
    CK(cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    ctx->present_in_flight = true;
    return MM_OK;
}
int mm_present_rgba8(mm_ctx *ctx, float *out_rgba, uint8_t *out_rgba8) { return present_impl(ctx, out_rgba, true, out_rgba8); }

int mm_microbench(mm_ctx *ctx, int kind, uint64_t table_bytes, double *result) {
    if (!ctx || !result) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    const unsigned blocks = (unsigned)ctx->n_sms * 8u;
    float *sink = reinterpret_cast<float *>(ctx->d_counters);
    float ms = 0.0f;
    if (kind == MM_MICROBENCH_GATHER) {
        if (table_bytes < sizeof(PairRec)) return fail(ctx, MM_ERR_INVALID, "mm_microbench: table smaller than one record");
        const uint32_t n_records = (uint32_t)(table_bytes / sizeof(PairRec) > 0x7FFFFFFFull ? 0x7FFFFFFFull : table_bytes / sizeof(PairRec));
        void *table = nullptr;
        CK(cudaMalloc(&table, (size_t)n_records * sizeof(PairRec)));
        cudaError_t e = cudaMemsetAsync(table, 0, (size_t)n_records * sizeof(PairRec), ctx->stream);
        const uint32_t iters = 4096;
        if (e == cudaSuccess) e = launch_mb_gather(table, n_records, 256, blocks, sink, ctx->stream);      // warm-up
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev0, ctx->stream);
        if (e == cudaSuccess) e = launch_mb_gather(table, n_records, iters, blocks, sink, ctx->stream);
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev1, ctx->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(ctx->ev1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        cudaFree(table);
        if (e != cudaSuccess) return fail(ctx, MM_ERR_CUDA, std::string("mm_microbench: ") + cudaGetErrorString(e));
        *result = (double)blocks * 256.0 * iters * 56.0 / (ms * 1e-3) / 1e9;            // GB/s of useful bytes
    } else if (kind == MM_MICROBENCH_FFMA) {
        const uint32_t iters = 1u << 16;
        CK(launch_mb_ffma(1024, blocks, sink, ctx->stream));
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        CK(launch_mb_ffma(iters, blocks, sink, ctx->stream));
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *result = (double)blocks * 256.0 * iters * 8.0 / (ms * 1e-3) / 1e12;             // T lane-instructions/s
    } else {
        return fail(ctx, MM_ERR_INVALID, "mm_microbench: unknown kind");
    }
    ctx->timed = false;
    return MM_OK;
}

int mm_rect_edge_thresholds(float length, float *lo, float *up) {
    if (!lo || !up) return MM_ERR_INVALID;
    return edge_thresholds(length, lo, up) ? MM_OK : MM_ERR_UNSUPPORTED;
}

int mm_axis_rect(const mm_plane *plane, float out[5], uint32_t *k) {
    if (!plane || !out || !k) return MM_ERR_INVALID;
    RectA r;
    if (!axis_rect(*plane, &r)) return MM_ERR_UNSUPPORTED;
    out[0] = r.c; out[1] = r.lo_a; out[2] = r.hi_a; out[3] = r.lo_b; out[4] = r.hi_b;
    *k = r.k;
    return MM_OK;
}

int mm_selftest_quotient(mm_ctx *ctx, uint64_t n_pairs, uint64_t seed, uint64_t *mismatches) {
    if (!ctx || !mismatches) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->d_counters, 0, sizeof(Counters), ctx->stream));
    CK(launch_quot_selftest(n_pairs, seed, &ctx->d_counters->paths, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *mismatches = ctx->h_counters->paths;
    return MM_OK;
}

int mm_trace_rays(mm_ctx *ctx, uint32_t flags, const float *rays, const uint32_t *slots, uint32_t n, float *t_out, uint32_t *index_out,
                  uint32_t *tally_out) {
    if (!ctx) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!rays || !t_out || !index_out || !tally_out || n == 0) return fail(ctx, MM_ERR_INVALID, "mm_trace_rays: null pointer or zero size");
    if (n > (1u << 30)) return fail(ctx, MM_ERR_UNSUPPORTED, "mm_trace_rays: more than 2^30 rays in one call");
    if (flags & ~(MM_FLAG_FORCE_LITERAL | MM_FLAG_RCP_SLAB | MM_FLAG_GENERAL_RECTS | MM_FLAG_NO_Y_TABLE))
        return fail(ctx, MM_ERR_INVALID, "mm_trace_rays: flags other than FORCE_LITERAL, RCP_SLAB, GENERAL_RECTS and NO_Y_TABLE");
    if (!ctx->have_scene) return fail(ctx, MM_ERR_NO_SCENE, "no scene uploaded");
    if (slots)
        for (uint32_t i = 0; i < n; i++)
            if (slots[i] != 0xFFFFFFFFu && slots[i] >= ctx->n_slots) return fail(ctx, MM_ERR_INVALID, "mm_trace_rays: slot out of range");
    KParams p;
    memset(&p, 0, sizeof(p));
    const bool ytab = traversal_params(ctx, flags, p);
    CK(cudaSetDevice(ctx->device));
    // one allocation: rays (8 floats), slot, t, index, tallies (6 words) per ray
    const size_t rays_b = (size_t)n * 8 * sizeof(float), word_b = (size_t)n * sizeof(uint32_t);
    char *buf = nullptr;
    CK(cudaMalloc(&buf, rays_b + 9 * word_b));
    float *d_rays = reinterpret_cast<float *>(buf), *d_t = reinterpret_cast<float *>(buf + rays_b + word_b);
    uint32_t *d_slots = reinterpret_cast<uint32_t *>(buf + rays_b), *d_index = reinterpret_cast<uint32_t *>(buf + rays_b + 2 * word_b);
    uint32_t *d_tally = reinterpret_cast<uint32_t *>(buf + rays_b + 3 * word_b);
    cudaError_t e = cudaMemcpyAsync(d_rays, rays, rays_b, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && slots) e = cudaMemcpyAsync(d_slots, slots, word_b, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_probe(p, ytab, d_rays, slots ? d_slots : nullptr, n, d_t, d_index, d_tally, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(t_out, d_t, word_b, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(index_out, d_index, word_b, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tally_out, d_tally, 6 * word_b, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(buf);
    if (e != cudaSuccess) return fail(ctx, MM_ERR_CUDA, std::string("mm_trace_rays: ") + cudaGetErrorString(e));
    return MM_OK;
}

int mm_selftest_div3(mm_ctx *ctx, uint64_t *mismatches) {
    if (!ctx || !mismatches) return MM_ERR_INVALID;
    ctx->err.clear();
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->d_counters, 0, sizeof(Counters), ctx->stream));
    CK(launch_div3_selftest(&ctx->d_counters->paths, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *mismatches = ctx->h_counters->paths;
    ctx->timed = false;
    return MM_OK;
}

int mm_last_counters(mm_ctx *ctx, mm_counters *out) {
    if (!ctx || !out) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->timed) return fail(ctx, MM_ERR_INVALID, "mm_last_counters: nothing rendered yet");
    CK(cudaEventSynchronize(ctx->ev2));              // the asynchronous counter copy of the last launch has landed
    counters_out(ctx->h_counters, out);
    return MM_OK;
}

int mm_last_ms(mm_ctx *ctx, float *ms) {
    if (!ctx || !ms) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->timed) return fail(ctx, MM_ERR_INVALID, "mm_last_ms: nothing rendered yet");
    CK(cudaEventSynchronize(ctx->ev1));
    CK(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return MM_OK;
}

int mm_last_tail(mm_ctx *ctx, uint64_t *queued_paths, uint64_t *deferred_pixels) {
    if (!ctx || !queued_paths || !deferred_pixels) return MM_ERR_INVALID;
    ctx->err.clear();
    if (!ctx->timed) return fail(ctx, MM_ERR_INVALID, "mm_last_tail: nothing rendered yet");
    CK(cudaEventSynchronize(ctx->ev2));
    const uint64_t cap = ctx->last_tail_cap, head = ctx->h_counters->tail_paths;
    *queued_paths = head < cap ? head : cap;
    *deferred_pixels = ctx->h_counters->tail_pixels;
    return MM_OK;
}

int mm_stream(mm_ctx *ctx, void **stream) {
    if (!ctx || !stream) return MM_ERR_INVALID;
    *stream = (void *)ctx->stream;
    return MM_OK;
}

int mm_get_scene_info(mm_ctx *ctx, mm_scene_info *out) {
    if (!ctx || !out) return MM_ERR_INVALID;
    if (!ctx->have_scene) return fail(ctx, MM_ERR_NO_SCENE, "no scene uploaded");
    out->n_planes = ctx->n_slots; out->n_nodes = ctx->n_nodes; out->bvh_depth = ctx->depth; out->max_leaf = ctx->max_leaf;
    out->fast_rect_ok = ctx->rect_fast_ok ? 1u : 0u;
    out->axis_rects = ctx->d_rects_axis ? 1u : 0u;
    out->fast_slab_ok = ctx->fast_ok ? 1u : 0u;
    out->smem_bytes = ctx->last_smem; out->block_threads = ctx->last_block_threads; out->blocks_per_sm = ctx->last_blocks_per_sm;
    out->n_sms = (uint32_t)ctx->n_sms;
    out->y_table = ctx->last_y_table;
    return MM_OK;
}

}  // extern "C"
