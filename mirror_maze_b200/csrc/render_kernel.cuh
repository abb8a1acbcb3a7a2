// render_kernel.cuh — device data layout and kernel parameters shared by render_kernel.cu and api.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/mirror_maze_cuda.h"

namespace mmk {

// One interior node's two children, 192 B.
// The reference node array (32 B each, children adjacent; shaders.metal:30-35,134-135) is re-laid per interior node for the
// packed-FP32 slab test: x and y of a plane sit in adjacent words (one register pair after the load) and every axis is
// stored in both travel orders, so that whatever the ray's direction signs the near plane is the first value:
//   ab[sx + 2*sy] = (c0.near.x, c0.near.y, c0.far.x, c0.far.y,  c1.near.x, c1.near.y, c1.far.x, c1.far.y)
//                   with near = min, far = max on an axis the ray travels up (s = 0), swapped when it travels down (s = 1)
//   z[sz]         = (c0.near.z, c1.near.z, c0.far.z, c1.far.z),  link[sz] = (c0.desc, c1.desc, 0, 0)   (same link in both)
//   desc: interior child = byte offset of its record (pair index * 192, < 2^31);
//         leaf child     = 0x80000000 | count << 24 | first slot in the leaf-ordered rect array (count <= 126).
// ab[0] / z[0] are the reference's (min, max) order, which the general (literal) slab form reads.
// One traversal step reads 56 B: ab[s] as one 32-B load (LDG.256), then z[sz] (16 B) and link (8 B).
struct __align__(32) PairRec {
    float4 ab[4][2];
    struct { float4 z; uint4 link; } zl[2];
};
static_assert(sizeof(PairRec) == 192, "pair record is 192 B");

// The same pair for the y-table traversal (traverse<..., YT = true>), 160 B.  Every maze has only a handful of distinct
// (min.y, max.y) child intervals (floor, roof, walls, light panels, outer walls: 5), so the ray's y quotients of all of them
// are computed once per traversal call into a per-lane table in shared memory, and a visit reads its two children's
// (near.y, far.y) from there instead of recomputing four quotients.  x and z are laid out like PairRec::zl's z:
//   xz[sx + 2*sz] = (c0.near.x, c1.near.x, c0.far.x, c1.far.x,  c0.near.z, c1.near.z, c0.far.z, c1.far.z)
//   link          = (c0.desc, c1.desc, c0.yoff, c1.yoff)     yoff = y-interval index * kYEntryStride (shared-memory byte offset)
//   desc: as in PairRec, with interior children at pair index * 160.
// A visit reads xz[s] as one 32-B load and link as one 16-B load; the record is padded to 160 B so that every xz stays
// 32-B aligned.  The intervals themselves follow the last record as float4 (min.y, max.y, max.y, min.y): the ray's travel
// order picks .xy (dir.y >= 0) or .zw.
struct __align__(32) PairRecY {
    float4 xz[4][2];
    uint4 link;
    uint4 pad;
};
static_assert(sizeof(PairRecY) == 160, "y-table pair record is 160 B");
constexpr uint32_t kMaxYIntervals = 8;         // scenes with more distinct child y-intervals use PairRec only
constexpr uint32_t kYEntryStride = 32 * 8;     // table layout [warp][interval][lane], 8 B per entry (near, far)
constexpr uint32_t kLeafBit = 0x80000000u;
constexpr uint32_t kMaxLeafCount = 126;

// One rectangle in leaf order (slot s = position in the reference `indices` array), 64 B.
// The normal is a per-rect constant of ray_rect_intersect (shaders.metal:52); it is evaluated once at upload with the
// same IEEE operations the literal code performs per call, hence bit-identical.  The edge tests of :60-63,
//     d = RN(x / L),  0 <= d && d <= L        (x = dot(isect - origin, edge), L = length(edge), a per-rect constant)
// are stored as an interval on x itself: lo <= x && x <= up decides exactly what the divide-then-compare decides, for
// every x including zeros, denormals, infinities and NaN (edge_thresholds in scene_prep.cpp derives both bounds from the
// round-to-nearest-even rule; tests/test_host_surface.py checks them against real divisions around every boundary).
struct __align__(16) RectI {
    float4 o_upv;   // origin.xyz, upper bound for dot(rv, v)
    float4 n_upu;   // normalize(cross(v,u)).xyz, upper bound for dot(rv, u)
    float4 v_lov;   // v.xyz, lower bound for dot(rv, v)
    float4 u_lou;   // u.xyz, lower bound for dot(rv, u)
};
static_assert(sizeof(RectI) == 64, "rect is 64 B");

// The same rectangle for scenes whose rects are all axis-aligned (every maze is: walls, floor, roof, light panels), 32 B.
// With n = +-e_k the literal test collapses exactly: dot(dir, n) = +-dir_k and dot(origin - o, n) = +-RN(c - o_k) (the other
// products are +-0), so a = RN(RN(c - o_k) / dir_k) bit for bit; and with v, u along the other two axes the edge tests
// lo <= RN(RN(p_j - origin_j) * edge_j) <= up are monotone in the intersection point's coordinate p_j = RN(o_j + RN(dir_j * a)),
// i.e. an interval [lo_j, hi_j] on p_j itself, found at upload by bisection over the floats with the literal operations
// (scene_prep.cpp::axis_rect).  Whenever the literal test can accept (0.1 < a < t <= 1e30, all terms finite) both forms decide
// alike; whenever it cannot, neither accepts.  a, b = the two in-plane axes in increasing order.
struct __align__(32) RectA {
    float c;                 // plane coordinate origin[k]
    float lo_a, hi_a, lo_b;
    float hi_b;
    uint32_t k;              // normal axis 0 / 1 / 2; 3 = never hit (degenerate rect: zero-length edge, NaN normal)
    uint32_t pad[2];
};
static_assert(sizeof(RectA) == 32, "axis-aligned rect is 32 B");

// Shading constants per slot, 32 B: albedo and emissions.rgb * emissions.a (shaders.metal:312,314,327).
struct __align__(16) RectS {
    float4 color;    // rgb, bits = material (0 matte, 1 mirror)
    float4 emitted;  // rgb * a, bits = original plane index
};

struct Counters {   // device-side mirror of mm_counters
    unsigned long long paths, rays, inner_visits, leaf_visits, rect_tests, hits, literal_rays, max_stack;
    unsigned long long next_unit;   // pool kernel: work-distribution ticket (zeroed with the counters before every launch)
    unsigned long long tail_paths;  // straggler queue head: paths trace_kernel handed to trace_tail_kernel (may pass tail_cap)
    unsigned long long tail_pixels; // deferred-pixel slots handed out
};

// One straggler path in the queue trace_kernel fills and trace_tail_kernel drains, 80 B:
//   a = (ori.xyz, dir.x)  b = (dir.yz, color.xy)  c = (color.z, light.xyz)
//   d = (RNG state, n | mirror_hits << 16, path index low, high word)   e = (first_hit, deferred-pixel slot, -, -)
// A path is only queued while alive, so every segment it ran was a hit: its segment count so far is n.
struct __align__(16) TailPath { float4 a, b, c, d, e; };
static_assert(sizeof(TailPath) == 80, "straggler record is 80 B");
// A deferred-pixel slot is 4 + 3 spp words: (samples still missing, pixel x, pixel y, tile index), then the pixel's tone-mapped
// samples as three planes of spp floats.

// One view of a multi-view launch (mm_render_views), 80 B, uploaded with every call.  The multi-view kernels take the array
// as a second parameter after KParams, which keeps KParams, and with it every single-view kernel, as it is.  The views share
// everything of KParams but its camera and time (uni carries their common view size and chunk width); of its outputs,
// image, tiles, peers and host_out are unused.
struct __align__(16) ViewRec {
    mm_uniform uni;            // the view's camera and time
    uint32_t chunk_off;        // the view's chunk list starts at KParams::chunks + chunk_off
    uint32_t pad;
    float *screen;             // the view's persistent screen, H*W*4 floats
    float *host_out;           // zero-copy output: the device alias of the view's mapped pinned host frame, or null
};
static_assert(sizeof(ViewRec) == 80, "view record is 80 B");

struct KParams {
    mm_uniform uni;           // the reference's 56-byte uniform, by value like set_bytes (main.rs:875-879)
    uint32_t spp, log2_spp;
    int32_t bounce_limit, mirror_limit;
    uint32_t grid_x, grid_y;
    uint32_t group_first, group_step, group_count;
    uint32_t T;                // threads per virtual group = chunk^2 * spp
    uint32_t dim_x, dim_y;     // virtual threads_per_threadgroup
    uint32_t ppc;
    uint32_t W, H;
    uint32_t n_pairs, n_slots;
    uint32_t rect_fast_ok;            // every edge length inside the guarded range of edge_thresholds
    uint32_t root_link, root_count;   // descriptor of node 0 (pair 0 unless the root is a leaf)
    uint32_t noise_w, noise_h;
    uint32_t force_literal;
    uint32_t rcp_mode;         // MM_FLAG_RCP_SLAB: slab quotients as (b - o) * RN(1/d)
    uint32_t scene_fast_ok;
    uint32_t rg_mask;          // trace_kernel_rg: bit r set = re-form the block's warps after segment r
    uint32_t quant8;           // MM_FLAG_SCREEN_RGBA8: stored pixels are quantised to k/255 (round to nearest even)
    uint64_t total_paths;
    const PairRec *pairs;
    const PairRecY *pairs_y;          // y-table pair records (trace_ytab_kernel; null otherwise)
    const float4 *y_ivals;            // their n_yiv y-intervals, right after the last PairRecY
    uint32_t n_yiv;
    const RectI *rects;
    const RectA *rects_axis;          // non-null when every rect of the scene is axis-aligned (and MM_FLAG_FORCE_LITERAL is off)
    const RectS *shade;
    const mm_chunk *chunks;
    const uint8_t *noise;
    float *image;              // may be null
    float *tiles;              // may be null
    float *peers[MM_MAX_PEERS];  // extra frames every finished pixel is stored into (peer-mapped or multicast), n_peers used
    uint32_t n_peers;
    uint32_t peers_multicast;  // peers[0] is an NVSwitch multicast address: stored with multimem.st, the only defined access to one
    float *host_out;           // mapped pinned host frame every finished pixel is also stored into (zero-copy output); may be null
    // pool kernel (pool_kernel.cu): per-warp pool geometry in shared memory
    uint32_t pool_M;            // path records per warp (<= 128)
    uint32_t pool_slot_words;   // record stride in words: 24 + traversal stack (BVH depth rounded up to 4)
    uint32_t pool_R;            // pixel records per warp
    uint32_t pool_region_words; // words of shared memory per warp
    uint32_t pool_th_leaf, pool_th_shade;   // a body below 32 ready paths runs once this many wait for it
    // straggler tail (trace_kernel -> trace_tail_kernel)
    uint32_t tail_k;            // a warp past bounce_limit segments with 1..tail_k live lanes queues them and stops; 0 = off
    uint32_t tail_cap;          // queue entries; deferred-pixel slots are never more than queued paths
    TailPath *tail_q;
    float *tail_pix;            // deferred-pixel slots of 4 + 3 spp words
    Counters *counters;
    uint32_t *dbg_first_hit, *dbg_segments, *dbg_mirror_hits;
    float *dbg_radiance;
};

// Block shapes: 32 warps/SM at <= 64 registers either way.  A block must hold whole pixels (spp | block threads, for the
// in-block reduction); small blocks retire sooner after their slowest warp (profiles/r1_block_shape.txt), so frames with
// spp <= kSmallBlock use kSmallBlock threads and only larger sample counts use kLargeBlock.  spp 512 and 1024 take the
// largest block there is, kHugeBlock (two pixels or one a block, one block an SM; DESIGN.md §4).
#ifndef MM_SMALL_BLOCK
#define MM_SMALL_BLOCK 64
#endif
constexpr int kSmallBlock = MM_SMALL_BLOCK;
constexpr int kLargeBlock = 256;
constexpr int kHugeBlock = 1024;
constexpr uint32_t kMaxSpp = kHugeBlock;       // a pixel never spans blocks
inline int block_threads_for(uint32_t spp) {
    return spp <= (uint32_t)kSmallBlock ? kSmallBlock : (spp <= (uint32_t)kLargeBlock ? kLargeBlock : kHugeBlock);
}

// Returns the kernel's static properties for the occupancy query and launch.
// ytab: trace_ytab_kernel / trace_tail_kernel<..., true> (the y-table traversal) instead of trace_kernel.
// views: the multi-view kernels (views_kernel / views_ytab_kernel, views_tail_kernel) of mm_render_views.
struct KernelChoice { bool counters, debug; int block_threads; bool pool; bool regroup; bool ytab; bool views; };
const void *kernel_ptr(KernelChoice c);
const void *pool_kernel_ptr(KernelChoice c);
cudaError_t launch_pool(const KParams &p, KernelChoice c, unsigned blocks, unsigned threads, size_t smem_bytes, cudaStream_t stream);
// views: the view records of a multi-view launch (c.views), device memory.
cudaError_t launch_trace(const KParams &p, KernelChoice c, unsigned blocks, size_t smem_bytes, cudaStream_t stream, const ViewRec *views = nullptr);
cudaError_t launch_tail(const KParams &p, KernelChoice c, unsigned blocks, size_t smem_bytes, cudaStream_t stream, const ViewRec *views = nullptr);
constexpr int kTailBlock = 256;
// mm_trace_rays: probe_rays_kernel over n rays (ytab: the y-table traversal; device buffers as in the header's prototype)
constexpr uint32_t kProbeBlock = 64;
cudaError_t launch_probe(const KParams &p, bool ytab, const float *rays, const uint32_t *slots, uint32_t n, float *t_out, uint32_t *index_out,
                         uint32_t *tally_out, cudaStream_t stream);
cudaError_t launch_mb_gather(const void *table, uint32_t n_records, uint32_t iters, unsigned blocks, float *sink, cudaStream_t stream);
cudaError_t launch_mb_ffma(uint32_t iters, unsigned blocks, float *sink, cudaStream_t stream);
cudaError_t launch_scatter_all(const float *gathered, float *image, const mm_chunk *chunks, uint32_t world, uint32_t max_count,
                               uint32_t n_groups, uint32_t chunk, uint32_t W, uint32_t H, cudaStream_t stream);
cudaError_t launch_blur(const float *src, float *dst, uint32_t W, uint32_t H, cudaStream_t stream, bool quant8 = false, uint8_t *bytes = nullptr);
// The same over n screens stored back to back ([n][H][W]) in one launch; no tap crosses a screen's border.
cudaError_t launch_blur_views(const float *src, float *dst, uint32_t W, uint32_t H, uint32_t n, cudaStream_t stream, bool quant8, uint8_t *bytes);
cudaError_t launch_div3_selftest(unsigned long long *d_mismatches, cudaStream_t stream);
cudaError_t launch_quot_selftest(uint64_t n, uint64_t seed, unsigned long long *d_mismatches, cudaStream_t stream);
cudaError_t launch_scatter(const float *tiles, float *image, const mm_chunk *chunks, uint32_t grid_groups, uint32_t group_first,
                           uint32_t group_step, uint32_t group_count, uint32_t chunk, uint32_t W, uint32_t H, cudaStream_t stream);

}  // namespace mmk
