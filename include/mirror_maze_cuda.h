/*
 * mirror_maze_cuda.h — C-ABI drop-in boundary for mirror-maze's per-pixel render kernel on B200 (sm_100a).
 *
 * What this replaces.  The reference has no plugin/operator API: the boundary of its hot path is the Metal
 * argument table of `compute_shader` (reference src/shaders.metal:245-259) as bound by the frame loop
 * (reference src/main.rs:867-886): texture(0) = screen, texture(1) = noise, buffer(0) = chunk list,
 * buffer(1) = rects, buffer(2) = BVH nodes, buffer(3) = prim indices, buffer(4) = one `uni` by value,
 * buffer(5) = materials, buffer(6) = emissions, plus the grid shape (src/main.rs:641-650).
 * Every entry point below names the reference call it stands in for.  Plain pointers and sizes only.
 *
 * A Rust driver binds this header with an `extern "C"` block (see INTEGRATION.md); all POD structs are
 * byte-identical to the reference's #[repr(C)] types (src/main.rs:32-90, src/maths.rs:3-16,50-52).
 *
 * Threading: a context is not thread-safe; it owns one CUDA device, one stream and all device memory.
 * mm_multi (below) is the same over a list of devices in one process: it owns one context per device, the peer
 * mappings between them and, optionally, the NCCL communicators of the tile gather.
 * Errors: every function returns 0 on success or a negative MM_ERR_* code and never aborts or throws
 * across the ABI (the reference panics through .expect()/.unwrap(), e.g. src/utils.rs:19,43).
 */
#ifndef MIRROR_MAZE_CUDA_H
#define MIRROR_MAZE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- POD layouts (SURVEY Appendix A) ------------------------------------------------------------- */

typedef struct mm_float2 { float x, y; } mm_float2;             /* maths.rs:50-52  (8 B)  */
typedef struct mm_float3 { float x, y, z; } mm_float3;          /* maths.rs:14-16  (12 B) */
typedef struct mm_float4 { float x, y, z, w; } mm_float4;       /* maths.rs:3-5    (16 B) */

/* main.rs:51-58 `Plane`  ==  shaders.metal:19-24 `rect`  (48 B, align 4) */
typedef struct mm_plane { mm_float3 origin, v, u, color; } mm_plane;

/* main.rs:74-81 `BVHNode`  ==  shaders.metal:30-35 `bvh_node`  (32 B).
 * tri_count > 0: leaf over indices[left_first .. left_first+tri_count); else children at left_first, +1. */
typedef struct mm_bvh_node { mm_float3 aabb_min, aabb_max; uint32_t left_first, tri_count; } mm_bvh_node;

/* main.rs:32-39 `Camera`  ==  shaders.metal:37-42 `camera`  (40 B) */
typedef struct mm_camera { mm_float3 camera_center; float focal_length; mm_float4 rotation; mm_float2 viewport; } mm_camera;

/* main.rs:41-49 `Uniform`  ==  shaders.metal:237-243 `uni`  (56 B) */
typedef struct mm_uniform { mm_camera cam; float view_width, view_height; uint32_t chunk_width, time; } mm_uniform;

/* One entry of `pixel_update_buffer` (shaders.metal:248; main.rs:293-326): top-left pixel of a chunk. */
typedef struct mm_chunk { uint32_t x, y; } mm_chunk;

/* ---- Dispatch parameters ------------------------------------------------------------------------- */

/*
 * The reference hard-codes these in the shader or the dispatch (shaders.metal:294-295 bounce_limit = 5,
 * mirror_limit = 15; main.rs:641-650 grid 32x24 groups of 32x32 threads => spp = 1024/16 = 64).
 * They are passed beside the 56-byte `uni` so that its layout stays the reference's.
 *
 * Virtual dispatch (SURVEY §8 D5).  The kernel's RNG seed is a function of the Metal thread coordinates
 * (shaders.metal:298), so the Metal grid is part of the contract and is kept as a *virtual* grid:
 *   threads per group T = chunk_width^2 * spp (<= 32, or a multiple of 32),   dims = (min(32,T), T/min(32,T))   (execution width 32),
 *   grid = grid_x x grid_y groups,   group (tgid.x, tgid.y) renders chunk  chunks[tgid.x + tgid.y*grid_x]
 *   (shaders.metal:266 uses (width/2)/ppc as the row stride, which equals grid_x = 32 in the reference's
 *   only configuration; the stride is grid_x here),  flat = gid.x + dims.x*gid.y,  pixel = flat / spp,
 *   sample = flat % spp,  texid = tgid*dims + gid.
 * With spp = 64, chunk 4, grid 32x24 this is the reference dispatch exactly.
 *
 * Tiles.  One call renders the groups  g = group_first + k*group_step,  k in [0, group_count)  of the
 * linear group index g = tgid.x + tgid.y*grid_x.  Seeds depend on g, not on k, so any partition of the
 * groups over calls or GPUs gives the bits of a single full-grid call.  group_count = 0 means "all".
 */
typedef struct mm_params {
    uint32_t spp;            /* samples per pixel: power of two, 1..256                              */
    uint32_t bounce_limit;   /* shaders.metal:294                                                    */
    uint32_t mirror_limit;   /* shaders.metal:295                                                    */
    uint32_t grid_x, grid_y; /* virtual threadgroups per grid (main.rs:646-650)                      */
    uint32_t group_first, group_step, group_count;
    uint32_t flags;          /* MM_FLAG_*                                                            */
} mm_params;

#define MM_FLAG_COUNTERS      1u   /* fill mm_counters beyond `rays` (slower kernel variant)          */
#define MM_FLAG_FORCE_LITERAL 2u   /* use the literal-divide traversal for every ray (validation)     */
#define MM_FLAG_RCP_SLAB     64u   /* opt-in arithmetic variant: slab quotients (b - o) * RN(1/d) instead of the literal
                                      (b - o) / d of shaders.metal:88-93 — what a fast-math compile of the shader amounts to.
                                      NOT the default; the oracle implements the same rule under the same flag and the
                                      kernel matches it bit for bit, but results differ from the literal mode's.       */
#define MM_FLAG_NO_ZERO_COPY 128u  /* mm_render / mm_render_async: copy the screen with a DMA transfer even when out_rgba is mapped pinned
                                      memory the kernel could store into directly (for comparisons)                        */
#define MM_FLAG_POOL_KERNEL  256u   /* trace with the persistent ray-pool kernel (pool_kernel.cu: warps own a pool of paths in shared
                                      memory and run interior / leaf / shade bodies on work queues) instead of the default
                                      one-thread-per-path kernel (render_kernel.cu).  Same bits; measured slower on B200
                                      (profiles/r2_pool_kernel.md), kept as the evidence for that design                    */
#define MM_FLAG_SCREEN_RGBA8 512u   /* the screen is an RGBA8Unorm texture, as the reference's is (main.rs:702-709): every pixel the dispatch
                                      stores is quantised per channel to rte(clamp(v, 0, 1) * 255) / 255 — what a read of the RGBA8Unorm
                                      texel returns (Metal's float -> unorm8 conversion rounds to nearest even) — so the persistent
                                      screen, the blur that feeds on it (mm_present_rgba8) and the frame hold 8-bit values.  Default is
                                      the unquantised fp32 screen the 1e-3 radiance tolerance is stated on.                       */
#define MM_FLAG_GENERAL_RECTS 2048u /* use the general rect test even when every rect of the scene is axis-aligned and the collapsed
                                      axis-aligned test applies (validation; same bits)                                         */
#define MM_FLAG_REGROUP     1024u   /* trace with trace_kernel_rg: the default kernel plus warp-level ray compaction — at segment boundaries
                                      the block's live paths are re-formed into warps through shared memory, sorted by ray steepness
                                      |dir.y|, ended paths dropped.  Same bits; fewer instructions (-14 % interior-body executions) but
                                      measured slower on B200 (profiles/r2_experiments.md), kept as the evidence for that design    */
#define MM_FLAG_NO_TAIL     4096u   /* trace every path to its end in the one-thread-per-path kernel (for comparisons; same bits).  By
                                      default a warp that is past bounce_limit segments with at most 8 live lanes hands those paths to
                                      a second kernel that runs them densely, one thread per path (render_kernel.cu, DESIGN.md §4)  */
#define MM_FLAG_NO_Y_TABLE  8192u   /* trace with trace_kernel even when the scene has the y-table (for comparisons; same bits).  By default
                                      a scene with at most 8 distinct child y-intervals (every maze has 5) is traced by
                                      trace_ytab_kernel, which computes a ray's y slab quotients once per traversal instead of in
                                      every interior visit (DESIGN.md §3-4)                                                       */

/* Exact event counts of one render call; identical on CPU oracle and GPU (SURVEY §8 d). */
typedef struct mm_counters {
    uint64_t paths;          /* (pixel, sample) pairs traced                                         */
    uint64_t rays;           /* calls of the traversal routine = bounce-loop iterations (the metric) */
    uint64_t inner_visits;   /* interior nodes whose two children were slab-tested                   */
    uint64_t leaf_visits;    /* leaves whose rects were tested                                       */
    uint64_t rect_tests;     /* ray_rect_intersect calls                                             */
    uint64_t hits;           /* traversal calls that returned a hit                                  */
    uint64_t literal_rays;   /* rays traced by the literal-divide traversal (GPU only; 0 on CPU)     */
    uint64_t max_stack;      /* deepest traversal-stack occupancy seen                               */
} mm_counters;

/*
 * Optional per-path observables (definitions: SURVEY Appendix C tail).  Each non-null pointer receives
 * group_count*T entries, entry [k*T + flat].  Host pointers for mm_render, ignored by the device variants.
 */
typedef struct mm_debug {
    uint32_t *first_hit;     /* beam.index after the n = 0 traversal, 0xFFFFFFFF on miss             */
    uint32_t *segments;      /* traversal calls made by this path                                    */
    uint32_t *mirror_hits;   /* final mirror_hits (shaders.metal:305,325)                            */
    float    *radiance;      /* 3 floats per path: incoming_light before the sqrt tone-map           */
} mm_debug;

/* ---- Error codes ---------------------------------------------------------------------------------- */

#define MM_OK                 0
#define MM_ERR_INVALID       -1   /* null pointer, zero size, bad parameter combination              */
#define MM_ERR_CUDA          -2   /* a CUDA runtime call failed; see mm_last_error                   */
#define MM_ERR_NO_SCENE      -3   /* render before mm_upload_scene                                   */
#define MM_ERR_BVH           -4   /* malformed BVH: child out of range, cycle, depth above MM_MAX_STACK */
#define MM_ERR_UNSUPPORTED   -5   /* spp not a power of two <= 256, chunk_width^2*spp > limits, ...  */
#define MM_ERR_NOMEM         -6

#define MM_MAX_STACK 52           /* device traversal stack: the reference's 50 entries (unchecked, shaders.metal:123) plus
                                     a bottom sentinel, rounded up.  Occupancy <= BVH depth - 1, so every tree the
                                     reference's stack can hold (depth <= 51) uploads; deeper ones return MM_ERR_BVH */
#define MM_MAX_BVH_DEPTH 51

typedef struct mm_ctx mm_ctx;

/* ---- Context --------------------------------------------------------------------------------------- */

/* Replaces Device::system_default + new_command_queue + pipeline creation (main.rs:616-644). */
int mm_create(int cuda_device, mm_ctx **out);
int mm_destroy(mm_ctx *ctx);
/* Never null; empty string when the last call on ctx succeeded.  mm_last_error(NULL) = last create error. */
const char *mm_last_error(const mm_ctx *ctx);

/*
 * Replaces the six make_buf calls and the noise-texture upload (main.rs:667-695, 723-730; utils.rs:86-94).
 * Copies everything; the caller keeps ownership.  materials: 1 byte per plane (Rust bool).
 * noise_rgba8: nw*nh*4 bytes, row pitch 4*nw (main.rs:695).  Validates the BVH (MM_ERR_BVH).
 */
int mm_upload_scene(mm_ctx *ctx,
                    const mm_plane *planes, uint32_t n_planes,
                    const mm_bvh_node *nodes, uint32_t n_nodes,
                    const uint32_t *indices,
                    const uint8_t *materials,
                    const mm_float4 *emissions,
                    const uint8_t *noise_rgba8, uint32_t noise_w, uint32_t noise_h);

/*
 * Replaces copy_to_buf(pixel_data) + set_bytes(uni) + dispatch_thread_groups (main.rs:784, 867-886) and the
 * read-back of the screen texture.  Synchronous.  `chunks` has grid_x*grid_y entries; chunks == NULL keeps the list of the
 * previous call / mm_set_chunks (the reference rewrites the buffer every frame, utils.rs:96-102; a full-frame caller
 * need not).  The context owns a persistent device screen image, the counterpart of the reference's GPU-private screen
 * texture (main.rs:702-709): created zero-filled at first use (and again when the view size changes), written only
 * at the pixels of the chunks a call renders, kept across calls.  out_rgba is a HOST buffer of
 * view_height*view_width*4 floats, row-major [y][x][rgba]; it may be null when the caller reads the screen later
 * (mm_present).  counters/debug may be null.  How out_rgba is filled depends on the memory it lies in:
 *   - mapped pinned memory (from mm_host_alloc / mm_host_register, or pinned by the caller's own CUDA allocator): ZERO-COPY —
 *     the kernel stores every pixel it finishes straight into out_rgba over PCIe while it traces, no copy follows.  Only
 *     the pixels of the chunks this call renders are written: out_rgba is then the caller's persistent copy of the
 *     screen, exactly like the reference's texture, and equals the device screen as long as every dispatch since the
 *     screen was created went into the same buffer.  MM_FLAG_NO_ZERO_COPY selects a DMA copy of the whole screen instead.
 *   - any other (pageable) memory, e.g. a Rust Vec<f32>: the whole screen is DMA-copied into a pinned staging buffer of
 *     the context and memcpy'd to out_rgba (what a pageable caller really pays; register the Vec once with
 *     mm_host_register to avoid it).
 */
int mm_render(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params,
              const mm_chunk *chunks, uint32_t n_chunks,
              float *out_rgba, mm_counters *counters, const mm_debug *debug);
/*
 * The same without the wait: the reference's frame loop commits and goes on (commit() without wait_until_completed,
 * main.rs:894).  mm_render_async returns once the frame is enqueued; out_rgba (and the debug arrays) are valid after
 * mm_wait, which also returns the frame's counters.  One host-buffer frame is in flight per context: a second
 * mm_render_async waits for the first.  mm_render == mm_render_async + mm_wait.
 */
int mm_render_async(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params,
                    const mm_chunk *chunks, uint32_t n_chunks, float *out_rgba, const mm_debug *debug);
int mm_wait(mm_ctx *ctx, mm_counters *counters);
/*
 * Pinned, device-mapped host memory for frames (the counterpart of the reference's StorageModeManaged buffers,
 * utils.rs:86-94): mm_host_alloc allocates it, mm_host_register pins and maps memory the caller already owns (a
 * Vec<f32>'s buffer; it must stay allocated until mm_host_unregister).  Process-wide, usable with every context and
 * device.  A frame buffer from here makes mm_render's output zero-copy (above).
 */
int mm_host_alloc(size_t bytes, void **out);
int mm_host_free(void *ptr);
int mm_host_register(void *ptr, size_t bytes);
int mm_host_unregister(void *ptr);

/*
 * Device-resident variants for callers that keep frames on the GPU (multi-GPU tile gather, frame batching).
 * mm_set_chunks replaces copy_to_buf (utils.rs:96-102) and is only needed when the chunk list changes.
 * mm_render_device is asynchronous on the context's stream (the reference's commit() does not wait either,
 * main.rs:894); mm_sync waits.  d_image: device pointer, H*W*4 floats.  d_tiles: device pointer,
 * group_count * chunk_width^2 * 4 floats, tile k = group group_first + k*group_step, pixel order = the
 * kernel's pixel_number (x offset = pn / chunk, y offset = pn % chunk; shaders.metal:272-275).
 * Exactly one of d_image / d_tiles may be null.
 */
int mm_set_chunks(mm_ctx *ctx, const mm_chunk *chunks, uint32_t n_chunks);
int mm_render_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params,
                     float *d_image, float *d_tiles);
/* Scatter gathered tiles (any rank's d_tiles layout) into an image: tile k -> chunk of group
 * group_first + k*group_step.  Asynchronous on the context's stream. */
int mm_scatter_tiles_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params,
                            const float *d_tiles, float *d_image);
/* The same for a whole all-gather result in one launch: d_gathered = world x max_count tiles, rank r's tile k at
 * row r*max_count + k, holding group r + k*world (the interleaved partition of tile_partition / TiledFrameRenderer). */
int mm_scatter_gathered_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, uint32_t world, uint32_t max_count,
                               const float *d_gathered, float *d_image);
/*
 * Render + exchange in one kernel (multi-GPU, no gather and no scatter): renders this rank's groups
 * (params->group_first / group_step / group_count) and stores every finished pixel straight into each of the n_frames
 * device frames given — the peer-mapped frame buffers of all ranks (NVLink peer stores), or ONE NVSwitch multicast
 * address that replicates the store into every rank's buffer.  frames[i]: H*W*4 floats each; 1 <= n_frames <= MM_MAX_PEERS.
 * Asynchronous on the context's stream; the caller orders a cross-rank barrier after it (the stores are complete when the
 * kernel is).  The reference is single-GPU (main.rs:867-886 writes its one screen texture); this is the tile exchange
 * of SURVEY section 8 (e) fused into the producing kernel.
 */
#define MM_MAX_PEERS 8
int mm_render_peers_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params,
                           float *const *frames, uint32_t n_frames);
/* The same through ONE NVSwitch multicast address mapped over every rank's frame (e.g. torch symmetric memory's
 * multicast_ptr): each pixel is one `multimem.st` that the switch replicates into all frames — the only instruction
 * family PTX defines for multicast addresses; plain stores to one are undefined. */
int mm_render_multicast_device(mm_ctx *ctx, const mm_uniform *uni, const mm_params *params, float *mc_frame);
int mm_sync(mm_ctx *ctx);
/* Run the context's work on a caller-owned cudaStream_t (e.g. torch's current stream) from now on; NULL
 * restores the context's own stream.  The caller keeps the stream alive while the context uses it. */
int mm_set_stream(mm_ctx *ctx, void *stream);
/* Counters of the most recent render launch; waits for that launch's (asynchronous) counter copy, not for the stream. */
int mm_last_counters(mm_ctx *ctx, mm_counters *out);
/* Device time of the most recent render launch in milliseconds (CUDA events on the context's stream, around the trace kernel
 * and, unless MM_FLAG_NO_TAIL, the straggler kernel after it). */
int mm_last_ms(mm_ctx *ctx, float *ms);
/* Straggler tail of the most recent render launch: paths the trace kernel queued for the second kernel, and pixels whose delivery
 * was deferred to it.  Both 0 under MM_FLAG_NO_TAIL.  Waits like mm_last_counters. */
int mm_last_tail(mm_ctx *ctx, uint64_t *queued_paths, uint64_t *deferred_pixels);
/* The context's cudaStream_t, for callers that order their own work (NCCL, torch) after the kernel. */
int mm_stream(mm_ctx *ctx, void **stream);
/* Static facts of the loaded scene / selected kernel (for reports). */
typedef struct mm_scene_info {
    uint32_t n_planes, n_nodes, bvh_depth, max_leaf;
    uint32_t fast_rect_ok;      /* 1 when every edge length allows the divide-free rect edge test      */
    uint32_t fast_slab_ok;      /* 1 when scene bounds allow the shared-reciprocal exact slab test    */
    uint32_t smem_bytes, block_threads, blocks_per_sm, n_sms;
    uint32_t axis_rects;        /* 1 when every rect is axis-aligned: the collapsed 32-byte rect test is in use */
    uint32_t y_table;           /* y-table entries the last render launch used (trace_ytab_kernel), 0 when it ran without one */
} mm_scene_info;
int mm_get_scene_info(mm_ctx *ctx, mm_scene_info *out);

/*
 * f-1 (SURVEY §8 f): the present pass' 5-tap blur, fragment_shader (shaders.metal:214-225, drawn at main.rs:888-892):
 *   c = img[p];  c += (img[p+(1,0)] + img[p-(1,0)]) / 2;  c += (img[p+(0,1)] + img[p-(0,1)]) / 2;  c /= 3;  img[p] = (c.rgb, 1)
 * The reference runs it in place on the persistent screen texture every frame (order-dependent read-modify-write
 * of neighbours); here it is the race-free ping-pong version: every read sees the previous frame's texture, reads
 * outside the texture return 0.  mm_present blurs the context's persistent screen image (the compute pass'
 * target) and, when out_rgba is non-null, copies the result to the host buffer (H*W*4 floats).  Synchronous.
 * mm_present_blur_device is the same kernel on caller device buffers (src != dst), asynchronous.
 */
int mm_present(mm_ctx *ctx, float *out_rgba);
/* The present pass on an RGBA8Unorm screen (use with MM_FLAG_SCREEN_RGBA8 dispatches): the blur's result is written back
 * quantised, like fragment_shader's store into the 8-bit drawable / screen texture.  out_rgba (H*W*4 floats, values k/255) and
 * out_rgba8 (H*W*4 bytes, the texels themselves) may each be null.  Synchronous. */
int mm_present_rgba8(mm_ctx *ctx, float *out_rgba, uint8_t *out_rgba8);
/* The present pass without the wait, as the reference's loop runs it (present_drawable + commit and on to the next frame,
 * main.rs:888-894): blur on the context's stream, then the blurred screen is snapshot on the device and read back into
 * out_rgba on a second stream, so the next dispatch overlaps the 16 bytes per pixel going over PCIe.  out_rgba must be pinned
 * host memory (mm_host_alloc / mm_host_register) and stay untouched until mm_wait_present returns; a later mm_present_async
 * into another buffer queues behind it. */
int mm_present_async(mm_ctx *ctx, float *out_rgba);
/* The same on an RGBA8Unorm screen (MM_FLAG_SCREEN_RGBA8 dispatches): the blur's quantised result is the new screen and its
 * texels — 4 bytes per pixel, what the reference's drawable holds (main.rs:702-709, 888-893) — are read back into pinned
 * out_rgba8 (H*W*4 bytes) on the second stream. */
int mm_present_async_rgba8(mm_ctx *ctx, uint8_t *out_rgba8);
int mm_wait_present(mm_ctx *ctx);
int mm_present_blur_device(mm_ctx *ctx, const float *d_src, float *d_dst, uint32_t width, uint32_t height);

/*
 * Micro-benchmarks behind the rooflines of this path (SURVEY §8 d; neither is in MEASURED_PEAKS.json):
 *   MM_MICROBENCH_GATHER  GB/s of useful bytes when every lane fetches the traversal's per-visit pattern (a 32-B, a 16-B
 *                         and an 8-B load = 56 B) from random 192-B records of a table of `table_bytes`
 *                         (pass the scene's pair-table size: L1-resident at 32x32, L2-resident at 256x256);
 *   MM_MICROBENCH_FFMA    T lane-instructions/s of dependent-chain-free FP32 FMAs (table_bytes ignored).
 */
#define MM_MICROBENCH_GATHER 0
#define MM_MICROBENCH_FFMA   1
int mm_microbench(mm_ctx *ctx, int kind, uint64_t table_bytes, double *result);

/*
 * Self-test of the kernel's shared-reciprocal slab quotient (see render_kernel.cu header): evaluates n_pairs
 * pseudo-random (x, d) pairs inside the guarded ranges, half of them adjacent to rounding midpoints, with both
 * the fast sequence (scalar, and packed with non-zero origins as the traversal runs it) and __fdiv_rn, then a fixed
 * set of edge operands (docs/exact_quotient.md, Evidence), and returns how many differ (must be 0).
 */
int mm_selftest_quotient(mm_ctx *ctx, uint64_t n_pairs, uint64_t seed, uint64_t *mismatches);
/* The present blur divides by 3 (shaders.metal:222) with a three-operation exact sequence instead of the IEEE divide; this
 * compares the two over ALL 2^32 float bit patterns and returns how many differ (must be 0). */
int mm_selftest_div3(mm_ctx *ctx, uint64_t *mismatches);

/*
 * Verification hook for the rect edge tests (reference src/shaders.metal:60-63: d = dot(rv, edge) / length(edge),
 * 0 <= d && d <= length).  The kernel stores, per edge, the interval [lo, up] on x = dot(rv, edge) that decides exactly
 * what the divide-then-compare decides under IEEE round-to-nearest-even; this returns that interval for a length.
 * MM_ERR_UNSUPPORTED when the length is outside the guarded range (such a scene renders with the literal divides).
 * Host-only, no GPU needed.
 */
int mm_rect_edge_thresholds(float length, float *lo, float *up);
/*
 * Verification hook for the axis-aligned rect test.  For a rect whose normal is +-e_k and whose edges lie along the other two
 * axes (every wall, floor, roof and light panel of a maze) ray_rect_intersect (shaders.metal:51-67) collapses exactly to
 * a = RN(RN(origin_k - o_k) / dir_k) and interval tests lo_j <= p_j <= hi_j on the intersection point's in-plane coordinates
 * p_j = RN(o_j + RN(dir_j * a)); the intervals are found by bisection over the floats with the literal operations.  out[0..5] =
 * c, lo_a, hi_a, lo_b, hi_b (a < b the in-plane axes), *k = normal axis (3: degenerate rect, never hit).  MM_ERR_UNSUPPORTED
 * when the rect is not axis-aligned (a scene with such a rect uses the general test throughout).  Host-only.
 */
int mm_axis_rect(const mm_plane *plane, float out[5], uint32_t *k);
/*
 * Verification hook for the traversal (intersect_bvh_iterative, shaders.metal:115-156) ray by ray, on the uploaded scene.
 * rays: n x 8 floats (ori.xyz, dir.xyz, starting t, alive: non-zero = traced); slots: n starting slots in leaf order (the
 * beam's index before the call), or NULL for none (0xFFFFFFFF).  Rays go 32 to a warp in the order given (a partial last warp
 * has dead lanes), and each warp selects its traversal form exactly as the bounce loop of mm_render does under the same
 * flags: MM_FLAG_FORCE_LITERAL, MM_FLAG_RCP_SLAB, MM_FLAG_GENERAL_RECTS and MM_FLAG_NO_Y_TABLE (any other flag is
 * MM_ERR_INVALID).  Per ray: t_out = the returned t; index_out = the hit's plane index, as mm_debug.first_hit reports it
 * (0xFFFFFFFF for none); tally_out = 6 words (interior visits, leaf visits, rect tests, deepest stack occupancy, lit = 1 when
 * the ray needs the literal-divide slab form, form = the traversal its warp ran: bit 0 mixed literal, bit 1 reciprocal-
 * multiply, bit 2 axis-aligned rect test, bit 3 y-table).  A dead ray returns its t and slot and counts nothing.  Synchronous.
 */
int mm_trace_rays(mm_ctx *ctx, uint32_t flags, const float *rays, const uint32_t *slots, uint32_t n,
                  float *t_out, uint32_t *index_out, uint32_t *tally_out);

/* ---- One process, several GPUs (SURVEY §8 b/e) ---------------------------------------------------------------------- */

/*
 * The reference drives one device from one thread (main.rs:616-623, 867-894).  mm_multi splits the same dispatch over a
 * list of CUDA devices inside ONE process, behind the same kind of calls: the scene is replicated on every device, the
 * frame's virtual groups are interleaved over the devices (device i renders groups i, i+n, ...; seeds depend on the group
 * index, so the assembled frame is bit-identical to a one-device frame), and the finished pixels are exchanged by
 *   MM_EXCHANGE_PEER  (default) the render kernel itself: every device's kernel stores each pixel it finishes into the
 *                     frame buffers of ALL devices through NVLink peer mappings (cudaDeviceEnablePeerAccess);
 *   MM_EXCHANGE_NCCL  tiles gathered with ncclAllGather over communicators from ncclCommInitAll (libnccl is loaded
 *                     at run time, only for this mode), then one scatter launch per device;
 *   MM_EXCHANGE_NONE  no device-side exchange: every device keeps only its own pixels; the frame is assembled in the
 *                     caller's mapped pinned host buffer by the kernels' zero-copy stores (n PCIe links in parallel).
 * out_rgba as for mm_render: a mapped pinned buffer is written by all kernels directly (zero-copy, every mode); any
 * other buffer gets device 0's assembled frame through a staged copy (not available with MM_EXCHANGE_NONE).
 */
typedef struct mm_multi mm_multi;
#define MM_EXCHANGE_PEER 0
#define MM_EXCHANGE_NCCL 1
#define MM_EXCHANGE_NONE 2
int mm_multi_create(const int *cuda_devices, int n_devices, int exchange, mm_multi **out);
int mm_multi_destroy(mm_multi *m);
const char *mm_multi_last_error(const mm_multi *m);     /* m == NULL: last mm_multi_create error */
int mm_multi_n_devices(const mm_multi *m);
int mm_multi_upload_scene(mm_multi *m,
                          const mm_plane *planes, uint32_t n_planes,
                          const mm_bvh_node *nodes, uint32_t n_nodes,
                          const uint32_t *indices, const uint8_t *materials, const mm_float4 *emissions,
                          const uint8_t *noise_rgba8, uint32_t noise_w, uint32_t noise_h);
/* One frame over all devices.  params->group_first/step/count are ignored (the library partitions the whole grid).
 * counters: sums over the devices (max for max_stack).  mm_multi_render == mm_multi_render_async + mm_multi_wait. */
int mm_multi_render(mm_multi *m, const mm_uniform *uni, const mm_params *params,
                    const mm_chunk *chunks, uint32_t n_chunks, float *out_rgba, mm_counters *counters);
int mm_multi_render_async(mm_multi *m, const mm_uniform *uni, const mm_params *params,
                          const mm_chunk *chunks, uint32_t n_chunks, float *out_rgba);
int mm_multi_wait(mm_multi *m, mm_counters *counters);
/* After mm_multi_wait: device `index`'s frame buffer (H*W*4 floats on that device; the whole frame with
 * MM_EXCHANGE_PEER / MM_EXCHANGE_NCCL, only that device's pixels with MM_EXCHANGE_NONE). */
int mm_multi_frame_device(mm_multi *m, int index, float **d_frame);
/* Slowest device's render-kernel time of the last frame, ms (CUDA events on each device's stream). */
int mm_multi_last_ms(mm_multi *m, float *ms);
/* The per-device context (scene info, microbenchmarks); owned by m. */
mm_ctx *mm_multi_ctx(mm_multi *m, int index);

/* ---- Host surface kept from the reference (restated in C++; no device work) ------------------------- */

/*
 * Maze -> walls -> planes/materials/emissions -> BVH, as main() does once at start (main.rs:357-588),
 * generalised from the hard-wired 10x10 to n x n (SURVEY §8 H3).  Arrays are owned by the scene object.
 */
typedef struct mm_scene mm_scene;
int mm_scene_build(uint32_t maze_n, uint64_t seed, int fast_bvh, mm_scene **out);
int mm_scene_free(mm_scene *s);
uint32_t mm_scene_n_planes(const mm_scene *s);
uint32_t mm_scene_n_nodes(const mm_scene *s);
const mm_plane    *mm_scene_planes(const mm_scene *s);
const mm_bvh_node *mm_scene_nodes(const mm_scene *s);
const uint32_t    *mm_scene_indices(const mm_scene *s);
const uint8_t     *mm_scene_materials(const mm_scene *s);
const mm_float4   *mm_scene_emissions(const mm_scene *s);
const uint8_t     *mm_scene_grid(const mm_scene *s);       /* n*n passage bits, row-major [y][x] (main.rs:388-394) */
uint32_t mm_scene_n_vert_walls(const mm_scene *s);
uint32_t mm_scene_n_hori_walls(const mm_scene *s);
const float *mm_scene_vert_walls(const mm_scene *s);       /* 3 floats each (x, start, len)   main.rs:409,416 */
const float *mm_scene_hori_walls(const mm_scene *s);       /* 3 floats each (y, start, len)   main.rs:431,437 */

/* build_bvh alone (main.rs:247-263) on caller planes; nodes must hold 2n-1 entries, indices n. */
int mm_build_bvh(const mm_plane *planes, uint32_t n, int fast, mm_bvh_node *nodes, uint32_t *n_nodes_out,
                 uint32_t *indices);

/* rand 0.8.5 StdRng (ChaCha12) restatement used by the maze (main.rs:381-382,460,467,494,501). */
typedef struct mm_stdrng mm_stdrng;
int mm_stdrng_new(uint64_t seed, mm_stdrng **out);
int mm_stdrng_free(mm_stdrng *r);
uint32_t mm_stdrng_next_u32(mm_stdrng *r);
float mm_stdrng_gen_f32(mm_stdrng *r);
uint32_t mm_stdrng_gen_range_u32(mm_stdrng *r, uint32_t low, uint32_t high);
/* Raw ChaCha block function with `rounds` rounds (8/12/20), 64-bit counter, 64-bit stream id. */
int mm_chacha_block(const uint8_t key[32], uint64_t counter, uint64_t stream, int rounds, uint32_t out[16]);

/* maths.rs:139-162, 175-178 */
mm_float4 mm_calculate_quaternion(mm_float3 dir);
mm_float4 mm_update_quat_angle(mm_float4 q, float theta);
mm_float3 mm_quat_mult(mm_float3 v, mm_float4 q);

/* gen_pixels without the shuffle (main.rs:293-302): x-major outer, y inner.  Returns the count written. */
uint32_t mm_gen_chunks(float view_width, float view_height, uint32_t chunk_width, mm_chunk *out, uint32_t cap);
/* Start-of-run camera and uniform as main.rs:732-755, generalised to an n x n maze (SURVEY §8 H3). */
int mm_default_uniform(uint32_t maze_n, float view_width, float view_height, uint32_t chunk_width,
                       uint32_t time, mm_uniform *out);

/* f-3 (SURVEY §8 f): player-box collision walk, main.rs:265-291. Returns node index or -1. */
int mm_check_collision(const mm_bvh_node *nodes, uint32_t n_nodes, mm_float3 bmin, mm_float3 bmax);
/* f-3: one frame of WASD movement with collision (main.rs:786-826).  keys = macOS key codes in press order
 * (0 = A, 1 = S, 2 = D, 13 = W; others ignored); each moves by 5/fps along the rotated axis; the move is undone
 * when the player box center +-(0.5, 0.2, 0.5) overlaps a leaf box.  Returns 1 if the move was blocked, 0 if not. */
int mm_move_camera(const mm_bvh_node *nodes, uint32_t n_nodes, mm_float3 center, mm_float4 quat, const uint16_t *keys,
                   uint32_t n_keys, float fps, mm_float3 *out_center);

/* f-1: the progressive-refresh chunk bag, gen_pixels + random_pixels (main.rs:293-326, 713-720, 778-784).  The
 * reference shuffles with the non-deterministic thread_rng; here the shuffle is rand 0.8.5's Fisher-Yates driven by
 * StdRng::seed_from_u64(seed).  mm_bag_next pops n chunk origins from the end of the bag and refills it with a clone
 * of the shuffled original when it runs dry; mm_bag_reshuffle is the regeneration on a rotation change (main.rs:838-839). */
typedef struct mm_bag mm_bag;
int mm_bag_new(float view_width, float view_height, uint32_t chunk_width, uint64_t seed, mm_bag **out);
int mm_bag_free(mm_bag *bag);
int mm_bag_next(mm_bag *bag, uint32_t n, mm_chunk *out);
int mm_bag_reshuffle(mm_bag *bag);
uint32_t mm_bag_size(const mm_bag *bag);

const char *mm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MIRROR_MAZE_CUDA_H */
