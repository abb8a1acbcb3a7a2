// render_kernel.cu — the hot path: mirror-maze's per-pixel path-tracing kernel, hand-written for sm_100a.
//
// One CUDA thread = one Metal thread of the reference's `compute_shader` (reference src/shaders.metal:245-368):
// one (pixel, sample) path through ray generation (:281-284), seed + jitter (:291,298,303), the bounce loop
// (:306-340) around intersect_bvh_iterative (:115-156) with intersect_aabb (:87-95) and ray_rect_intersect
// (:51-67), per-sample tone-map (:344) and the per-pixel reduction in the reference's summation order (:347-366).
//
// Arithmetic contract (SURVEY §8 a-0): every fp32 + - * / sqrt is one IEEE round-to-nearest operation, written
// with explicit __f*_rn intrinsics so that no compiler flag can contract or approximate them.  Results are
// bit-identical to oracle/mm_oracle.cpp.
//
// Slab test without twelve divides.  The literal test divides (bound - origin) by the ray direction twelve times
// per interior node.  In the common case the same correctly rounded quotients are produced from one IEEE
// reciprocal per axis per ray: with r = RN(1/d), rho = 1 - d*r (exact by FMA), rl = RN(rho*r),
//     q1 = RN(x*r + RN(x*rl))      error < 1/2 ulp + 2^-23 ulp  (faithful)
//     e  = x - d*q1                exact by FMA
//     q  = RN(q1 + e*r)            == RN(x/d)   (Markstein's theorem: r = RN(1/d), q1 faithful, no over/underflow)
// The no-over/underflow side conditions are guaranteed by range checks: the scene's box coordinates are 0 or in
// [2^-10, 2^30] (checked at upload) and a ray uses this path only when every |d| is in [2^-60, 2^60] and every
// |origin| is 0 or in [2^-40, 2^30]; any other ray (zero / denormal / huge / NaN components) takes the literal
// __fdiv_rn traversal, so the union is exact for all inputs.  MM_FLAG_FORCE_LITERAL disables the fast path.
#include "trace_device.cuh"

namespace mmk {
namespace {

// Stores one finished pixel, from the sums of its spp tone-mapped samples in the reference's order (shaders.metal:343-366),
// into every output of the dispatch: the frame, the tiles, the zero-copy host frame and the frames of the fused exchange.
__device__ __forceinline__ void deliver_pixel(const KParams &P, float sx, float sy, float sz, uint32_t pxx, uint32_t pxy, size_t tile) {
    const float d = (float)(int)P.spp;
    float4 px = make_float4(fdiv(sx, d), fdiv(sy, d), fdiv(sz, d), 1.0f);
    if (P.quant8) px = quant8(px);
    if (P.image && pxx < P.W && pxy < P.H) reinterpret_cast<float4 *>(P.image)[(size_t)pxy * P.W + pxx] = px;
    if (P.tiles) reinterpret_cast<float4 *>(P.tiles)[tile] = px;
    if ((P.n_peers || P.host_out) && pxx < P.W && pxy < P.H) {
        const size_t at = (size_t)pxy * P.W + pxx;
        if (P.host_out) reinterpret_cast<float4 *>(P.host_out)[at] = px;        // zero-copy output: mapped pinned host frame, over PCIe
        if (P.peers_multicast) {                                    // fused exchange, NVSwitch multicast: one store, replicated by the switch
            float4 *mc = reinterpret_cast<float4 *>(P.peers[0]) + at;
            asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(px.x), "f"(px.y), "f"(px.z), "f"(px.w) : "memory");
        } else {                                                    // fused exchange, NVLink peer mappings: one store per rank's frame
            for (uint32_t i = 0; i < P.n_peers; i++) reinterpret_cast<float4 *>(P.peers[i])[at] = px;
        }
    }
}

// Event counts: warp-reduce, one atomic per warp and counter.
template <bool CNT>
__device__ __forceinline__ void add_counters(const KParams &P, uint32_t seg, uint32_t nhits, uint32_t nliteral, uint32_t paths, Tally tl) {
    unsigned long long v_rays = seg, v_hits = nhits, v_lit = nliteral, v_paths = paths;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v_rays += __shfl_xor_sync(0xFFFFFFFFu, v_rays, o);
        v_hits += __shfl_xor_sync(0xFFFFFFFFu, v_hits, o);
        v_lit += __shfl_xor_sync(0xFFFFFFFFu, v_lit, o);
        v_paths += __shfl_xor_sync(0xFFFFFFFFu, v_paths, o);
    }
    unsigned long long v_inner = tl.inner, v_leaf = tl.leaf, v_rect = tl.rect;
    uint32_t v_ms = tl.max_stack;
    if (CNT) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            v_inner += __shfl_xor_sync(0xFFFFFFFFu, v_inner, o);
            v_leaf += __shfl_xor_sync(0xFFFFFFFFu, v_leaf, o);
            v_rect += __shfl_xor_sync(0xFFFFFFFFu, v_rect, o);
            v_ms = max(v_ms, __shfl_xor_sync(0xFFFFFFFFu, v_ms, o));
        }
    }
    if ((threadIdx.x & 31u) == 0u) {
        if (v_rays) atomicAdd(&P.counters->rays, v_rays);
        if (v_hits) atomicAdd(&P.counters->hits, v_hits);
        if (v_paths) atomicAdd(&P.counters->paths, v_paths);
        if (v_lit) atomicAdd(&P.counters->literal_rays, v_lit);
        if (CNT) {
            atomicAdd(&P.counters->inner_visits, v_inner);
            atomicAdd(&P.counters->leaf_visits, v_leaf);
            atomicAdd(&P.counters->rect_tests, v_rect);
            atomicMax(&P.counters->max_stack, (unsigned long long)v_ms);
        }
    }
}

// Block epilogue shared by the trace kernels.  On entry red[] holds every thread's tone-mapped sample (3 planes of
// kBlockThreads floats, indexed by the thread the path started on) and the block has synchronised.
// TAIL: qi is the straggler-queue entry of the thread's path when trace_kernel queued it (0xFFFFFFFF otherwise).  A pixel with
// a queued sample is not stored here: its other samples go to a deferred-pixel slot, and trace_tail_kernel delivers the pixel
// when its last sample arrives.
template <bool CNT, bool TAIL, int kBlockThreads>
__device__ __forceinline__ void block_epilogue(const KParams &P, float *red, bool active, uint32_t flat, uint32_t pxx, uint32_t pxy, uint32_t k,
                                               uint32_t seg, uint32_t nhits, uint32_t nliteral, Tally tl, uint32_t qi) {
    const uint32_t tid = threadIdx.x;
    float *rx = red, *ry = red + kBlockThreads, *rz = red + 2 * kBlockThreads;
    bool deferred = false;
    if (TAIL && __syncthreads_or(qi != 0xFFFFFFFFu)) {
        __shared__ uint32_t pslot[kBlockThreads];                          // per pixel of the block: queued samples, then its slot
        const uint32_t pix = tid >> P.log2_spp, si = tid & (P.spp - 1);    // blocks hold whole pixels (block_threads_for)
        if (tid < (kBlockThreads >> P.log2_spp)) pslot[tid] = 0u;
        __syncthreads();
        if (qi != 0xFFFFFFFFu) atomicAdd(&pslot[pix], 1u);
        __syncthreads();
        if (si == 0u) {
            const uint32_t missing = pslot[pix];
            uint32_t s = 0xFFFFFFFFu;
            if (missing) {
                s = (uint32_t)atomicAdd(&P.counters->tail_pixels, 1ull);
                uint32_t *h = reinterpret_cast<uint32_t *>(P.tail_pix) + (size_t)s * (4u + 3u * P.spp);
                h[0] = missing; h[1] = pxx; h[2] = pxy; h[3] = k * P.ppc + (flat >> P.log2_spp);
            }
            pslot[pix] = s;
        }
        __syncthreads();
        const uint32_t s = pslot[pix];
        if (s != 0xFFFFFFFFu) {
            deferred = true;
            if (qi != 0xFFFFFFFFu) {
                P.tail_q[qi].e.y = __uint_as_float(s);
            } else {
                float *v = P.tail_pix + (size_t)s * (4u + 3u * P.spp) + 4u;
                v[si] = rx[tid]; v[P.spp + si] = ry[tid]; v[2u * P.spp + si] = rz[tid];
            }
        }
    }
    // Per-pixel reduction in the reference's order (shaders.metal:343-366): pairs, quads, octets (the phases whose
    // stride is < spp), then the pixel's first thread adds the octets serially and divides by spp.
#pragma unroll
    for (uint32_t stride = 1; stride <= 4; stride *= 2) {
        if (stride < P.spp && (tid & (2 * stride - 1)) == 0) {
            rx[tid] = fadd(rx[tid], rx[tid + stride]);
            ry[tid] = fadd(ry[tid], ry[tid + stride]);
            rz[tid] = fadd(rz[tid], rz[tid + stride]);
        }
        __syncthreads();
    }
    if (active && !deferred && (flat & (P.spp - 1)) == 0) {
        float sx = rx[tid], sy = ry[tid], sz = rz[tid];
        for (uint32_t i = 1; i < P.spp / 8; i++) {
            sx = fadd(sx, rx[tid + 8 * i]); sy = fadd(sy, ry[tid + 8 * i]); sz = fadd(sz, rz[tid + 8 * i]);
        }
        deliver_pixel(P, sx, sy, sz, pxx, pxy, (size_t)k * P.ppc + (flat >> P.log2_spp));
    }
    add_counters<CNT>(P, seg, nhits, nliteral, active ? 1u : 0u, tl);
}

// Which traverse<MIXED, CNT, RCP, AX, YT> instantiation a warp ran, as bits (reported by probe_rays_kernel).
constexpr uint32_t kFormMixed = 1u, kFormRcp = 2u, kFormAxis = 4u, kFormYTable = 8u;

// One traversal for the lanes of a warp together, in the form the warp selects: a warp with a live literal lane (or a scene
// without the divide-free rect test) runs the mixed form, any other the y-table (YT), reciprocal-multiply or plain packed
// form, with the axis-aligned rect test where the scene has it.  lit: this lane's ray is literal; form: the kForm* bits of
// the instantiation that ran, written only when FORM (so that the bounce loop compiles exactly as without it).  YT: the host
// selects it only without MM_FLAG_RCP_SLAB; ytab is the lane's column of the y-table in dynamic shared memory.
template <bool CNT, bool YT, bool FORM = false>
__device__ __forceinline__ Hit warp_traverse(const KParams &P, uint32_t root, const bool &alive, const V3 &ori, const V3 &dir, const float &t,
                                             const uint32_t &slot, Tally &tl, uint32_t ytab, bool &lit, uint32_t &form) {
    lit = ray_is_literal(P, ori, dir);
    const bool any_lit = __any_sync(0xFFFFFFFFu, alive && lit) || !P.rect_fast_ok;   // MIXED also means literal rect tests
    Hit h;
    if (YT) {
        if (!any_lit && P.rects_axis) {
            h = traverse<false, CNT, false, true, true>(P.pairs_y, P.rects_axis, root, alive, false, ori, dir, t, slot, &tl, ytab, P.y_ivals, P.n_yiv);
            if (FORM) form = kFormYTable | kFormAxis;
        } else if (!any_lit) {
            h = traverse<false, CNT, false, false, true>(P.pairs_y, P.rects, root, alive, false, ori, dir, t, slot, &tl, ytab, P.y_ivals, P.n_yiv);
            if (FORM) form = kFormYTable;
        } else {
            h = traverse<true, CNT, false>(P.pairs, P.rects, root, alive, lit, ori, dir, t, slot, &tl);
            if (FORM) form = kFormMixed;
        }
    } else if (P.rcp_mode) {
        if (!any_lit) { h = traverse<false, CNT, true>(P.pairs, P.rects, root, alive, false, ori, dir, t, slot, &tl); if (FORM) form = kFormRcp; }
        else { h = traverse<true, CNT, true>(P.pairs, P.rects, root, alive, lit, ori, dir, t, slot, &tl); if (FORM) form = kFormMixed | kFormRcp; }
    } else {
        if (!any_lit && P.rects_axis) { h = traverse<false, CNT, false, true>(P.pairs, P.rects_axis, root, alive, false, ori, dir, t, slot, &tl); if (FORM) form = kFormAxis; }
        else if (!any_lit) { h = traverse<false, CNT, false>(P.pairs, P.rects, root, alive, false, ori, dir, t, slot, &tl); if (FORM) form = 0u; }
        else { h = traverse<true, CNT, false>(P.pairs, P.rects, root, alive, lit, ori, dir, t, slot, &tl); if (FORM) form = kFormMixed; }
    }
    return h;
}

// One segment of the bounce loop (shaders.metal:306-340) for the lanes of a warp together: traverse, then shade the hit of
// every live lane.  A lane whose path has ended (or that has no path) idles with alive = false.
template <bool CNT, bool DBG, bool YT>
__device__ __forceinline__ void bounce_segment(const KParams &P, uint32_t root, bool &alive, V3 &ori, V3 &dir, V3 &color, V3 &light, float &t,
                                               uint32_t &slot, uint32_t &state, int &n, int &mirror_hits, uint32_t &first_hit,
                                               uint32_t &seg, uint32_t &nhits, uint32_t &nliteral, Tally &tl, uint32_t ytab) {
    bool lit;
    uint32_t form;
    const Hit h = warp_traverse<CNT, YT>(P, root, alive, ori, dir, t, slot, tl, ytab, lit, form);
    t = h.t; slot = h.slot;
    if (alive) {
        if (lit) nliteral++;
        seg++;
        if (!(t < 1e30f)) {                                        // :308, :336-339 (sky term is * 0.0)
            alive = false;
        } else {
            nhits++;
            uint32_t orig = 0xFFFFFFFFu;
            if (!shade_hit(P, slot, t, ori, dir, color, light, state, mirror_hits, (DBG && n == 0) ? &orig : nullptr)) alive = false;
            if (DBG && n == 0) first_hit = orig;
            t = 1e30f;                                             // :323, :330
            n++;
            alive = alive && (n < P.bounce_limit + mirror_hits);   // :306
        }
    }
}

__device__ __forceinline__ void write_dbg(const KParams &P, uint64_t path, uint32_t first_hit, uint32_t seg, int mirror_hits, V3 light) {
    if (P.dbg_first_hit) P.dbg_first_hit[path] = first_hit;
    if (P.dbg_segments) P.dbg_segments[path] = seg;
    if (P.dbg_mirror_hits) P.dbg_mirror_hits[path] = (uint32_t)mirror_hits;
    if (P.dbg_radiance) { P.dbg_radiance[3 * path] = light.x; P.dbg_radiance[3 * path + 1] = light.y; P.dbg_radiance[3 * path + 2] = light.z; }
}

// The straggler tail.  Almost every path ends after exactly bounce_limit segments; a mirror hit adds one (:306), so past
// bounce_limit a warp typically runs a whole traversal and shading for 1-3 live lanes at the price of 32.  At a segment
// boundary past bounce_limit, a warp with 1..tail_k live lanes instead writes those paths' complete state to a global queue
// (one atomic per warp; entries past tail_cap stay with the warp, which is the one-kernel behaviour) and leaves the bounce loop.
// trace_tail_kernel then runs the queued paths densely, one thread per path, with the same traversal and shading code.
// The body of trace_kernel (YT = false) and trace_ytab_kernel (YT = true: the y-table traversal, whose table follows red[] in
// dynamic shared memory, n_yiv entries of kYEntryStride bytes per warp).
template <bool CNT, bool DBG, bool YT, int kBlockThreads>
__device__ __forceinline__ void trace_body(const KParams &P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *red = reinterpret_cast<float *>(smem_raw);                      // 3 * kBlockThreads floats
    const uint32_t ytab = YT ? 3u * kBlockThreads * sizeof(float) + (threadIdx.x >> 5) * P.n_yiv * kYEntryStride + (threadIdx.x & 31u) * 8u : 0u;

    const uint64_t path = (uint64_t)blockIdx.x * kBlockThreads + threadIdx.x;
    const bool active = path < P.total_paths;
    Tally tl = {0u, 0u, 0u, 0u};
    uint32_t seg = 0, nhits = 0, nliteral = 0;
    V3 sample = mk(0.0f, 0.0f, 0.0f);
    uint32_t pxx = 0, pxy = 0, k = 0, flat = 0;
    const uint32_t root = P.root_count ? (kLeafBit | P.root_link | (P.root_count << 24)) : P.root_link;   // pair 0 is at byte offset 0
    V3 st_ori = mk(0.0f, 0.0f, 0.0f), st_dir = mk(1.0f, 1.0f, 1.0f), st_color = mk(1.0f, 1.0f, 1.0f), st_light = mk(0.0f, 0.0f, 0.0f);
    float st_t = 1e30f;
    uint32_t st_slot = 0xFFFFFFFFu, st_state = 0u, first_hit = 0xFFFFFFFFu, qi = 0xFFFFFFFFu;
    int mirror_hits = 0;
    bool n_alive = false;

    if (active) {
        const PathStart ps = start_path(P, path);
        k = ps.k; flat = ps.flat; pxx = ps.pxx; pxy = ps.pxy;
        n_alive = 0 < P.bounce_limit;                                      // :306, n = 0
        st_ori = ps.ori; st_dir = ps.dir; st_state = ps.state;
    }

    // Bounce loop (shaders.metal:306-340).  The lanes of a warp go through it together, segment by segment, so that the
    // traversal's votes can use the full warp; a lane whose path has ended (or that has no path) idles with alive = false.
    {
        V3 ori = st_ori, dir = st_dir, color = st_color, light = st_light;
        float t = st_t;
        uint32_t slot = st_slot, state = st_state;
        int n = 0;
        bool alive = active && n_alive, may_queue = P.tail_k != 0u;
        while (true) {
            unsigned live;
            while ((live = __ballot_sync(0xFFFFFFFFu, alive)) != 0u) {
                // Every live lane has hit on every segment so far, so all of them have the same n (= their segment count).
                if (may_queue && (uint32_t)__popc(live) <= P.tail_k && __ballot_sync(0xFFFFFFFFu, alive && n >= P.bounce_limit)) break;
                bounce_segment<CNT, DBG, YT>(P, root, alive, ori, dir, color, light, t, slot, state, n, mirror_hits, first_hit, seg, nhits, nliteral, tl, ytab);
            }
            if (live == 0u) break;
            // Queue the live paths: one reservation per warp.  Lanes that find the queue full keep their paths and trace on.
            may_queue = false;
            const uint32_t lead = (uint32_t)__ffs(live) - 1u, lane = threadIdx.x & 31u;
            unsigned long long base = 0;
            if (lane == lead) base = atomicAdd(&P.counters->tail_paths, (unsigned long long)__popc(live));
            base = __shfl_sync(0xFFFFFFFFu, base, lead) + (unsigned long long)__popc(live & ((1u << lane) - 1u));
            if (alive && base < P.tail_cap) {
                qi = (uint32_t)base;
                TailPath *q = P.tail_q + qi;
                q->a = make_float4(ori.x, ori.y, ori.z, dir.x);
                q->b = make_float4(dir.y, dir.z, color.x, color.y);
                q->c = make_float4(color.z, light.x, light.y, light.z);
                q->d = make_float4(__uint_as_float(state), __uint_as_float((uint32_t)n | ((uint32_t)mirror_hits << 16)),
                                   __uint_as_float((uint32_t)path), __uint_as_float((uint32_t)(path >> 32)));
                q->e = make_float4(__uint_as_float(DBG ? first_hit : 0xFFFFFFFFu), 0.0f, 0.0f, 0.0f);   // .y: deferred-pixel slot, set in the epilogue
                alive = false;
            }
        }
        sample = mk(fsqrt(fmaxf(light.x, 0.0f)), fsqrt(fmaxf(light.y, 0.0f)), fsqrt(fmaxf(light.z, 0.0f)));   // :344
        if (DBG && active && qi == 0xFFFFFFFFu) write_dbg(P, path, first_hit, seg, mirror_hits, light);
    }

    red[threadIdx.x] = sample.x; red[kBlockThreads + threadIdx.x] = sample.y; red[2 * kBlockThreads + threadIdx.x] = sample.z;
    __syncthreads();
    block_epilogue<CNT, true, kBlockThreads>(P, red, active, flat, pxx, pxy, k, seg, nhits, nliteral, tl, qi);
}

template <bool CNT, bool DBG, int kBlockThreads>
__global__ void __launch_bounds__(kBlockThreads, 1024 / kBlockThreads)
trace_kernel(const __grid_constant__ KParams P) { trace_body<CNT, DBG, false, kBlockThreads>(P); }

template <bool CNT, bool DBG, int kBlockThreads>
__global__ void __launch_bounds__(kBlockThreads, 1024 / kBlockThreads)
trace_ytab_kernel(const __grid_constant__ KParams P) { trace_body<CNT, DBG, true, kBlockThreads>(P); }

// The paths trace_kernel queued, one thread per path in queue order (dense warps), from where they stopped to their end.  The
// thread that stores a pixel's last missing sample reduces the pixel's samples in the reference's order and delivers it.
// YT: the y-table traversal, as in trace_ytab_kernel; the table is the whole dynamic shared memory.
template <bool CNT, bool DBG, bool YT>
__global__ void __launch_bounds__(kTailBlock, 1024 / kTailBlock)
trace_tail_kernel(const __grid_constant__ KParams P) {
    const unsigned long long head = P.counters->tail_paths;                // written by trace_kernel, the launch before
    const uint32_t nq = head < P.tail_cap ? (uint32_t)head : P.tail_cap;
    const uint32_t root = P.root_count ? (kLeafBit | P.root_link | (P.root_count << 24)) : P.root_link;
    const uint32_t ytab = YT ? (threadIdx.x >> 5) * P.n_yiv * kYEntryStride + (threadIdx.x & 31u) * 8u : 0u;
    const uint32_t words = 4u + 3u * P.spp;
    Tally tl = {0u, 0u, 0u, 0u};
    uint32_t seg = 0, nhits = 0, nliteral = 0;
    for (uint32_t i0 = blockIdx.x * kTailBlock; i0 < nq; i0 += gridDim.x * kTailBlock) {
        const uint32_t i = i0 + threadIdx.x;
        const bool has = i < nq;
        V3 ori = mk(0.0f, 0.0f, 0.0f), dir = mk(1.0f, 1.0f, 1.0f), color = mk(1.0f, 1.0f, 1.0f), light = mk(0.0f, 0.0f, 0.0f);
        uint32_t state = 0u, first_hit = 0xFFFFFFFFu, pix = 0u, slot = 0xFFFFFFFFu;
        uint64_t path = 0;
        int n = 0, mirror_hits = 0;
        if (has) {
            const TailPath *q = P.tail_q + i;
            const float4 a = q->a, b = q->b, c = q->c, d = q->d, e = q->e;
            ori = mk(a.x, a.y, a.z); dir = mk(a.w, b.x, b.y); color = mk(b.z, b.w, c.x); light = mk(c.y, c.z, c.w);
            state = __float_as_uint(d.x);
            const uint32_t nm = __float_as_uint(d.y);
            n = (int)(nm & 0xFFFFu); mirror_hits = (int)(nm >> 16);
            path = (uint64_t)__float_as_uint(d.z) | ((uint64_t)__float_as_uint(d.w) << 32);
            first_hit = __float_as_uint(e.x); pix = __float_as_uint(e.y);
        }
        const uint32_t pseg = (uint32_t)n - seg;                          // segments this path ran in trace_kernel, less ours so far
        float t = 1e30f;
        bool alive = has;
        while (__any_sync(0xFFFFFFFFu, alive))
            bounce_segment<CNT, DBG, YT>(P, root, alive, ori, dir, color, light, t, slot, state, n, mirror_hits, first_hit, seg, nhits, nliteral, tl, ytab);
        if (has) {
            if (DBG) write_dbg(P, path, first_hit, pseg + seg, mirror_hits, light);
            const uint32_t si = (uint32_t)path & (P.spp - 1u);           // sample within the pixel (T and group starts are multiples of spp)
            float *v = P.tail_pix + (size_t)pix * words;
            v[4u + si] = fsqrt(fmaxf(light.x, 0.0f)); v[4u + P.spp + si] = fsqrt(fmaxf(light.y, 0.0f));   // :344
            v[4u + 2u * P.spp + si] = fsqrt(fmaxf(light.z, 0.0f));
            __threadfence();                                               // the sample is visible before the count drops
            if (atomicSub(reinterpret_cast<uint32_t *>(v), 1u) == 1u) {    // the pixel's last missing sample
                __threadfence();
                const uint32_t *h = reinterpret_cast<const uint32_t *>(v);
                deliver_pixel(P, reduce_samples(v + 4, P.spp, 1), reduce_samples(v + 4 + P.spp, P.spp, 1),
                              reduce_samples(v + 4 + 2 * P.spp, P.spp, 1), h[1], h[2], h[3]);
            }
        }
    }
    add_counters<CNT>(P, seg, nhits, nliteral, 0u, tl);
}

// Verification hook (mm_trace_rays): one traversal per ray through the bounce loop's form selection, 32 consecutive rays to a
// warp, so that the caller decides each warp's composition.  rays: n x 8 floats (ori.xyz, dir.xyz, t, alive != 0); slots: the
// starting slots, or null for none.  Per ray: the returned t, the hit's plane index (the shading record's original index, as
// shade_hit reports first_hit; 0xFFFFFFFF for no slot) and (inner, leaf, rect, max_stack, lit, form).  A dead ray keeps its
// t and slot and counts nothing.  YT: the y-table traversal; the table is the whole dynamic shared memory, [warp][interval][lane].
template <bool YT>
__global__ void __launch_bounds__(kProbeBlock)
probe_rays_kernel(const __grid_constant__ KParams P, const float *__restrict__ rays, const uint32_t *__restrict__ slots, uint32_t n,
                  float *__restrict__ t_out, uint32_t *__restrict__ index_out, uint32_t *__restrict__ tally_out) {
    const uint32_t i = blockIdx.x * kProbeBlock + threadIdx.x;
    const bool has = i < n;
    const uint32_t root = P.root_count ? (kLeafBit | P.root_link | (P.root_count << 24)) : P.root_link;
    const uint32_t ytab = YT ? (threadIdx.x >> 5) * P.n_yiv * kYEntryStride + (threadIdx.x & 31u) * 8u : 0u;
    V3 ori = mk(0.0f, 0.0f, 0.0f), dir = mk(1.0f, 1.0f, 1.0f);
    float t = 1e30f;
    uint32_t slot = 0xFFFFFFFFu;
    bool alive = false;
    if (has) {
        const float *r = rays + 8 * (size_t)i;
        ori = mk(r[0], r[1], r[2]); dir = mk(r[3], r[4], r[5]); t = r[6];
        alive = r[7] != 0.0f;
        if (slots) slot = slots[i];
    }
    Tally tl = {0u, 0u, 0u, 0u};
    bool lit;
    uint32_t form;
    const Hit h = warp_traverse<true, YT, true>(P, root, alive, ori, dir, t, slot, tl, ytab, lit, form);
    if (has) {
        t_out[i] = h.t;
        index_out[i] = h.slot == 0xFFFFFFFFu ? 0xFFFFFFFFu : __float_as_uint(__ldg(reinterpret_cast<const float4 *>(P.shade + h.slot) + 1).w);
        uint32_t *o = tally_out + 6 * (size_t)i;
        o[0] = tl.inner; o[1] = tl.leaf; o[2] = tl.rect; o[3] = tl.max_stack; o[4] = lit ? 1u : 0u; o[5] = form;
    }
}

// ---- trace_kernel_rg: the same kernel with the block's paths RE-FORMED INTO WARPS at every segment boundary ---------------------
// After the first diffuse bounce the rays of a warp have nothing in common, and the warp runs every segment for as long as
// its slowest ray needs (17.4 of 32 lanes busy in the interior body).  How long a ray travels — and with it how many nodes it
// visits — correlates with how steeply it points at the floor or the roof (|dir.y|: the maze is a 10-unit-high slab, rays near
// the vertical end after a few nodes, near-horizontal ones cross many cells; trace replays in tools/sched_sim_r2.py).  So at
// the end of every segment the block pushes the state of its live paths through shared memory, ordered by a 5-bit key on
// |dir.y| (a counting sort: one shared-memory atomic per path, one warp scan), and each warp continues with 32 paths of similar
// steepness; ended paths drop out, so the tail segments (paths kept alive by mirror hits) run in fewer, fuller warps.  Which lane
// traces which path changes, nothing else: every path keeps its own RNG state, counters and home thread (the thread it started
// on, where its sample is delivered for the pixel reduction), so every observable stays bit-identical.
template <bool CNT, bool DBG, int kBlockThreads>
__global__ void __launch_bounds__(kBlockThreads, 1024 / kBlockThreads)
trace_kernel_rg(const __grid_constant__ KParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *red = reinterpret_cast<float *>(smem_raw);                                  // 3 * kBlockThreads floats: samples by home thread
    float4 *xch = reinterpret_cast<float4 *>(smem_raw + 3 * kBlockThreads * sizeof(float));   // 4 planes of kBlockThreads float4: path state in flight
    uint32_t *hist = reinterpret_cast<uint32_t *>(xch + 4 * kBlockThreads);            // 2 x 32 bin counters (double-buffered)

    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint64_t path = (uint64_t)blockIdx.x * kBlockThreads + tid;
    const bool active = path < P.total_paths;
    Tally tl = {0u, 0u, 0u, 0u};
    uint32_t seg = 0, nhits = 0, nliteral = 0;                                         // per-lane event counts (summed over the grid at the end)
    uint32_t pxx = 0, pxy = 0, k = 0, flat = 0;                                        // of the path this thread STARTED (its home pixel)
    const uint32_t root = P.root_count ? (kLeafBit | P.root_link | (P.root_count << 24)) : P.root_link;
    // the path this lane currently carries
    V3 ori = mk(0.0f, 0.0f, 0.0f), dir = mk(1.0f, 1.0f, 1.0f), color = mk(1.0f, 1.0f, 1.0f), light = mk(0.0f, 0.0f, 0.0f);
    uint32_t state = 0u, first_hit = 0xFFFFFFFFu, home = tid, pseg = 0;
    int n = 0, mirror_hits = 0;
    bool has = false;

    if (active) {
        const PathStart ps = start_path(P, path);
        k = ps.k; flat = ps.flat; pxx = ps.pxx; pxy = ps.pxy;
        ori = ps.ori; dir = ps.dir; state = ps.state;
        has = 0 < P.bounce_limit;                                                      // :306, n = 0
    }
    red[tid] = 0.0f; red[kBlockThreads + tid] = 0.0f; red[2 * kBlockThreads + tid] = 0.0f;   // sqrt(max(0, 0)) of a path that never runs (:344)
    if (DBG && active && !has) {
        if (P.dbg_first_hit) P.dbg_first_hit[path] = 0xFFFFFFFFu;
        if (P.dbg_segments) P.dbg_segments[path] = 0u;
        if (P.dbg_mirror_hits) P.dbg_mirror_hits[path] = 0u;
        if (P.dbg_radiance) { P.dbg_radiance[3 * path] = 0.0f; P.dbg_radiance[3 * path + 1] = 0.0f; P.dbg_radiance[3 * path + 2] = 0.0f; }
    }
    if (tid < 64) hist[tid] = 0u;          // kBlockThreads >= 64
    uint32_t live = (uint32_t)__syncthreads_count(has);                                // paths of the block still running
    uint32_t round = 0, n_rg = 0;
    // P.rg_mask: bit r set = re-form the warps after segment r.  After the mask's last round the warps run on independently.
    const uint32_t last_rg = P.rg_mask ? 32u - (uint32_t)__clz(P.rg_mask) : 0u;        // first round index without any later regroup

    while (live > 0u) {
        // ---- one segment for the lanes that carry a path (whole warps without one skip it) ----
        if (__any_sync(0xFFFFFFFFu, has)) {
            const bool lit = ray_is_literal(P, ori, dir);
            const bool any_lit = __any_sync(0xFFFFFFFFu, has && lit) || !P.rect_fast_ok;
            Hit h;
            if (P.rcp_mode) {
                if (!any_lit) h = traverse<false, CNT, true>(P.pairs, P.rects, root, has, false, ori, dir, 1e30f, 0xFFFFFFFFu, &tl);
                else h = traverse<true, CNT, true>(P.pairs, P.rects, root, has, lit, ori, dir, 1e30f, 0xFFFFFFFFu, &tl);
            } else {
                if (!any_lit) h = traverse<false, CNT, false>(P.pairs, P.rects, root, has, false, ori, dir, 1e30f, 0xFFFFFFFFu, &tl);
                else h = traverse<true, CNT, false>(P.pairs, P.rects, root, has, lit, ori, dir, 1e30f, 0xFFFFFFFFu, &tl);
            }
            if (has) {
                if (lit) nliteral++;
                seg++; pseg++;
                bool alive = false;
                if (h.t < 1e30f) {                                                     // :308, :336-339 (sky term is * 0.0)
                    nhits++;
                    uint32_t orig = 0xFFFFFFFFu;
                    alive = shade_hit(P, h.slot, h.t, ori, dir, color, light, state, mirror_hits, (DBG && n == 0) ? &orig : nullptr);
                    if (DBG && n == 0) first_hit = orig;
                    n++;
                    alive = alive && (n < P.bounce_limit + mirror_hits);               // :306
                }
                if (!alive) {                                                          // the path is over: its sample goes home (:344)
                    red[home] = fsqrt(fmaxf(light.x, 0.0f)); red[kBlockThreads + home] = fsqrt(fmaxf(light.y, 0.0f));
                    red[2 * kBlockThreads + home] = fsqrt(fmaxf(light.z, 0.0f));
                    if (DBG) {
                        const uint64_t hp = (uint64_t)blockIdx.x * kBlockThreads + home;
                        if (P.dbg_first_hit) P.dbg_first_hit[hp] = first_hit;
                        if (P.dbg_segments) P.dbg_segments[hp] = pseg;
                        if (P.dbg_mirror_hits) P.dbg_mirror_hits[hp] = (uint32_t)mirror_hits;
                        if (P.dbg_radiance) { P.dbg_radiance[3 * hp] = light.x; P.dbg_radiance[3 * hp + 1] = light.y; P.dbg_radiance[3 * hp + 2] = light.z; }
                    }
                    has = false;
                }
            }
        }
        if (round >= 32u || !((P.rg_mask >> round) & 1u)) {                            // no regroup after this segment
            round++;
            if (round >= last_rg && !__any_sync(0xFFFFFFFFu, has)) break;              // nothing left to wait for: this warp is done
            continue;
        }
        // ---- re-form the warps: counting sort of the live paths by |dir.y| (dir is normalised: :321, :329) ----
        uint32_t *h_now = hist + 32u * (n_rg & 1u), *h_next = hist + 32u * ((n_rg + 1u) & 1u);
        n_rg++;
        const uint32_t bin = min(31u, (uint32_t)(fabsf(dir.y) * 32.0f));
        uint32_t pos = 0;
        if (has) pos = atomicAdd(h_now + bin, 1u);
        if (tid < 32) h_next[tid] = 0u;
        __syncthreads();
        const uint32_t c = h_now[lane];
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += v;
        }
        live = __shfl_sync(0xFFFFFFFFu, incl, 31);
        const uint32_t start = __shfl_sync(0xFFFFFFFFu, incl - c, bin);
        if (has) {
            const uint32_t r = start + pos;
            xch[r] = make_float4(ori.x, ori.y, ori.z, dir.x);
            xch[kBlockThreads + r] = make_float4(dir.y, dir.z, color.x, color.y);
            xch[2 * kBlockThreads + r] = make_float4(color.z, light.x, light.y, light.z);
            xch[3 * kBlockThreads + r] = make_float4(__uint_as_float(state), __uint_as_float((uint32_t)n | ((uint32_t)mirror_hits << 16)),
                                                     __uint_as_float(home | (pseg << 12)), __uint_as_float(first_hit));
        }
        __syncthreads();
        has = tid < live;
        if (has) {
            const float4 a = xch[tid], b = xch[kBlockThreads + tid], cc = xch[2 * kBlockThreads + tid], d = xch[3 * kBlockThreads + tid];
            ori = mk(a.x, a.y, a.z); dir = mk(a.w, b.x, b.y); color = mk(b.z, b.w, cc.x); light = mk(cc.y, cc.z, cc.w);
            state = __float_as_uint(d.x);
            const uint32_t nm = __float_as_uint(d.y), hs = __float_as_uint(d.z);
            n = (int)(nm & 0xFFFFu); mirror_hits = (int)(nm >> 16);
            home = hs & 0xFFFu; pseg = hs >> 12;
            first_hit = __float_as_uint(d.w);
        }
        round++;
    }
    __syncthreads();
    block_epilogue<CNT, false, kBlockThreads>(P, red, active, flat, pxx, pxy, k, seg, nhits, nliteral, tl, 0xFFFFFFFFu);
}

// De-interleave gathered tiles into the frame (consumer side of the multi-GPU tile gather).
__global__ void scatter_kernel(const float4 *__restrict__ tiles, float4 *__restrict__ image, const mm_chunk *__restrict__ chunks,
                               uint32_t group_first, uint32_t group_step, uint32_t group_count, uint32_t chunk, uint32_t ppc,
                               uint32_t W, uint32_t H) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)group_count * ppc) return;
    const uint32_t k = (uint32_t)(i / ppc), pn = (uint32_t)(i % ppc);
    const mm_chunk ch = chunks[group_first + k * group_step];
    const uint32_t x = ch.x + pn / chunk, y = ch.y + pn % chunk;
    if (x < W && y < H) image[(size_t)y * W + x] = tiles[i];
}

// The whole all-gather result in one launch: rank r's tile k is group r + k*world (the interleaved partition).
__global__ void scatter_all_kernel(const float4 *__restrict__ gathered, float4 *__restrict__ image, const mm_chunk *__restrict__ chunks,
                                   uint32_t world, uint32_t max_count, uint32_t n_groups, uint32_t chunk, uint32_t ppc, uint32_t W, uint32_t H) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)world * max_count * ppc) return;
    const uint32_t pn = (uint32_t)(i % ppc);
    const uint64_t tile = i / ppc;
    const uint32_t r = (uint32_t)(tile / max_count), k = (uint32_t)(tile % max_count);
    const uint64_t g = (uint64_t)r + (uint64_t)k * world;
    if (g >= n_groups) return;                         // padding rows of ranks that own one group less
    const mm_chunk ch = chunks[g];
    const uint32_t x = ch.x + pn / chunk, y = ch.y + pn % chunk;
    if (x < W && y < H) image[(size_t)y * W + x] = gathered[i];
}

// Self-test of the shared-reciprocal quotient against __fdiv_rn, through the scalar quot<true> and through quot2, the packed
// sequence the traversal runs (b + (-o), then mul, fma, fma, fma).  Pseudo-random operands inside the guarded ranges
// (|d| in [2^-60, 2^60], x = RN(b - o) = 0 or |x| in [2^-40, 2^31]); half of the samples are built to land within a few
// 2^-24 ulp of a rounding midpoint, the only place where a faithful-but-not-exact quotient could differ, with quotient
// exponents over the whole [-100, 91] the ranges allow.  A deterministic pass then covers the edge operands (below).
__device__ __forceinline__ uint32_t mix32(uint64_t &s) {
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    uint32_t x = (uint32_t)(((s >> 18) ^ s) >> 27), r = (uint32_t)(s >> 59);
    return (x >> r) | (x << ((32 - r) & 31));
}
__device__ __forceinline__ float with_exp(uint32_t bits, int e) { return __uint_as_float((bits & 0x807FFFFFu) | ((uint32_t)(e + 127) << 23)); }
__device__ __forceinline__ bool d_guarded(float d) { return fabsf(d) >= 8.673617379884035e-19f /*2^-60*/ && fabsf(d) <= 1.152921504606847e18f /*2^60*/; }
__device__ __forceinline__ bool x_guarded(float x) { return x == 0.0f || (fabsf(x) >= 9.094947017729282e-13f /*2^-40*/ && fabsf(x) <= 2147483648.0f /*2^31*/); }

// One pseudo-random sample (x, d); false when it falls outside the guarded ranges.  keep_d: build x for the d given.
__device__ __forceinline__ bool quot_sample(uint64_t &s, float &x, float &d, bool keep_d) {
    const uint32_t a = mix32(s), b = mix32(s), c = mix32(s);
    if (c & 1u) {
        // adversarial: x ~ (q + half ulp(q)) * d for a random q, so x/d sits next to a rounding midpoint
        const int eq = (int)(a % 192u) - 100;                              // quotient exponent in [-100, 91]
        if (!keep_d) {                                                     // d's exponent such that |q d| can lie in [2^-40, 2^31]
            const int lo = max(-60, -41 - eq), hi = min(60, 31 - eq);
            d = with_exp(b, lo + (int)(mix32(s) % (uint32_t)(hi - lo + 1)));
        }
        const float q = with_exp(mix32(s), eq);
        double mid = (double)q + 0.5 * (double)(__uint_as_float(__float_as_uint(fabsf(q)) + 1u) - fabsf(q)) * (q < 0 ? -1.0 : 1.0);
        x = (float)(mid * (double)d);
        if ((c >> 1) & 1u) x = __uint_as_float(__float_as_uint(x) + ((c >> 2) & 3u) - 1u);   // +-1 ulp neighbours
    } else {
        if (!keep_d) d = with_exp(b, (int)(a % 121u) - 60);
        x = with_exp(mix32(s), (int)((c >> 1) % 72u) - 40);
        if (((c >> 8) & 63u) == 0u) x = 0.0f;
    }
    return d_guarded(d) && x_guarded(x);
}

// An origin o for which b = RN(x + o) and RN(b - o) = x hold exactly: 0, or -sign(x) y with y = |x| with its low mantissa
// bits masked and scaled by 2^-k, a multiple of ulp(x) not above |x|, so that |b| = |x| - y lies on x's grid.
__device__ __forceinline__ float origin_for(float x, uint32_t salt) {
    if ((salt & 3u) == 0u || x == 0.0f) return 0.0f;
    const uint32_t k = (salt >> 2) & 7u;
    const uint32_t keep = 0xFF800000u | ((salt >> 5) & 0x7FFFFFu & ~((1u << k) - 1u));
    const float y = fmul(__uint_as_float(__float_as_uint(fabsf(x)) & keep), __uint_as_float((uint32_t)(127 - k) << 23));
    return x > 0.0f ? -y : y;
}

__device__ __forceinline__ bool same_quot(float a, float b) { return __float_as_uint(a) == __float_as_uint(b) || (a == 0.0f && b == 0.0f); }

// Mismatches of three samples against __fdiv_rn: (x0, d0) and (x1, d1) through the scalar form (o = 0) and as the two halves
// of one packed quotient with their own origins (the interior visit's x|y pair); (x0, d0) and (x2, d0) as the halves of the
// y-table fill's form, one origin and one direction duplicated (has2: x2 is a sample).
__device__ uint32_t quot_check(float x0, float d0, float x1, float d1, float x2, bool has2, uint32_t salt) {
    Axis a0, a1;
    a0.o = 0.0f; a0.d = d0; a0.r = __frcp_rn(d0); a0.rl = fmul(__fmaf_rn(-d0, a0.r, 1.0f), a0.r);
    a1.o = 0.0f; a1.d = d1; a1.r = __frcp_rn(d1); a1.rl = fmul(__fmaf_rn(-d1, a1.r, 1.0f), a1.r);
    uint32_t bad = 0;
    bad += !same_quot(quot<true>(x0, a0), quot<false>(x0, a0));
    bad += !same_quot(quot<true>(x1, a1), quot<false>(x1, a1));
    const float o0 = origin_for(x0, salt), o1 = origin_for(x1, salt >> 10);
    const float b0 = fadd(x0, o0), b1 = fadd(x1, o1);
    const f2 q = quot2<false>(pack2(b0, b1), pack2(-o0, -o1), pack2(-d0, -d1), pack2(a0.r, a1.r), pack2(a0.rl, a1.rl));
    bad += !same_quot(lo2f(q), fdiv(fsub(b0, o0), d0));
    bad += !same_quot(hi2f(q), fdiv(fsub(b1, o1), d1));
    const float b2 = fadd(x2, o0);
    if (has2 && x_guarded(fsub(b2, o0))) {
        const f2 qy = quot2<false>(pack2(b0, b2), pack2(-o0, -o0), pack2(-d0, -d0), pack2(a0.r, a0.r), pack2(a0.rl, a0.rl));
        bad += !same_quot(lo2f(qy), fdiv(fsub(b0, o0), d0));
        bad += !same_quot(hi2f(qy), fdiv(fsub(b2, o0), d0));
    }
    return bad;
}

// Edge operands of the deterministic pass: d = +-m 2^k for k in [-60, 60] and x = +-m 2^k for k in [-40, 31], m = 1 (powers of
// two: rho = rl = 0), 1 + 2^-23 or 2 - 2^-23 (all-ones mantissa), plus x = 0; those past 2^60 or 2^31 are skipped.  The
// pairs include |d| = 2^-60 and 2^60 with their inside neighbours, |x| = 2^-40 and 2^31 with theirs, and the tiny-x, huge-d
// combinations whose p = x rl and e r are subnormal.
constexpr uint32_t kEdgeD = 2u * 3u * 121u, kEdgeX = 2u * 3u * 72u + 1u;
__device__ __forceinline__ float edge_operand(uint32_t i, int k0) {
    const uint32_t m = (i >> 1) % 3u, mant = m == 0u ? 0u : (m == 1u ? 1u : 0x7FFFFFu);
    return __uint_as_float(((i & 1u) << 31) | ((uint32_t)((int)((i >> 1) / 3u) + k0 + 127) << 23) | mant);
}

__global__ void quot_selftest_kernel(uint64_t n, uint64_t seed, unsigned long long *mismatches) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t s = seed ^ (tid * 0x9E3779B97F4A7C15ull);
    unsigned long long bad = 0;
    for (uint64_t i = tid; i < n; i += stride) {
        float x0, d0, x1, d1, x2;
        const bool ok0 = quot_sample(s, x0, d0, false), ok1 = quot_sample(s, x1, d1, false);
        float d2 = d0;
        const bool ok2 = quot_sample(s, x2, d2, true);
        if (ok0 && ok1) bad += quot_check(x0, d0, x1, d1, x2, ok2, mix32(s));
    }
    for (uint64_t i = tid; i < (uint64_t)kEdgeD * kEdgeX; i += stride) {
        const uint32_t id = (uint32_t)(i / kEdgeX), ix = (uint32_t)(i % kEdgeX);
        const float d = edge_operand(id, -60), x = ix == kEdgeX - 1u ? 0.0f : edge_operand(ix, -40);
        if (d_guarded(d) && x_guarded(x)) bad += quot_check(x, d, x, -d, -x, true, (uint32_t)i * 2654435761u);
    }
    if (bad) atomicAdd(mismatches, bad);
}

// fragment_shader's 5-tap blur (shaders.metal:214-225), ping-pong: one thread per pixel, one float4 per tap.  HBM-bound:
// 16 B read + 16 B written per pixel (the four neighbour taps hit L1/L2).
// x / 3 without the divide: q0 = RN(x * r), e = x - 3 q0 (exact by FMA), q = RN(q0 + e * r) with r = RN(1/3).  Equal to __fdiv_rn(x, 3)
// for every float whose quotient is a normal number — established by exhaustion over all 2^32 bit patterns (div3_selftest_kernel,
// mm_selftest_div3; tests/test_next_rows.py) — and guarded for the rest (tiny values take the IEEE divide).  x / 2 is x * 0.5: the
// same real number, hence the same rounding.
__device__ __forceinline__ float div3(float x) {
    if (!(fabsf(x) >= 1e-30f && fabsf(x) <= 3.4028234663852886e38f)) return fdiv(x, 3.0f);   // zeros, denormal quotients, infinities, NaN: the literal divide
    const float r = 0.3333333432674407958984375f;                          // RN(1/3)
    const float q0 = fmul(x, r);
    return __fmaf_rn(__fmaf_rn(-3.0f, q0, x), r, q0);
}
__global__ void div3_selftest_kernel(unsigned long long *mismatches) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    for (uint64_t i = tid; i < (1ull << 32); i += stride) {
        const float x = __uint_as_float((uint32_t)i);
        const float a = div3(x), b = fdiv(x, 3.0f);
        if (__float_as_uint(a) != __float_as_uint(b) && !(a != a && b != b)) bad++;   // NaN payloads aside, bit for bit
    }
    if (bad) atomicAdd(mismatches, bad);
}

// fragment_shader's 5-tap blur (shaders.metal:214-225), ping-pong.  HBM-bound: 16 B read + 16 B written per pixel (the four
// neighbour taps hit L1/L2).  One thread handles two horizontally adjacent pixels (8 loads for 2 pixels instead of 10).
__global__ void __launch_bounds__(256) blur_kernel(const float4 *__restrict__ src, float4 *__restrict__ dst, uint32_t W, uint32_t H, bool q8,
                                                   uchar4 *__restrict__ bytes) {
    const uint32_t x0 = 2u * (blockIdx.x * blockDim.x + threadIdx.x), y = blockIdx.y;
    if (x0 >= W || y >= H) return;
    const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const size_t row = (size_t)y * W;
    const bool two = x0 + 1 < W;
    const float4 c0 = __ldg(src + row + x0), c1 = two ? __ldg(src + row + x0 + 1) : zero;
    const float4 l0 = x0 > 0 ? __ldg(src + row + x0 - 1) : zero, r1 = x0 + 2 < W ? __ldg(src + row + x0 + 2) : zero;
    const float4 d0 = y + 1 < H ? __ldg(src + row + W + x0) : zero, u0 = y > 0 ? __ldg(src + row - W + x0) : zero;
    const float4 d1 = (two && y + 1 < H) ? __ldg(src + row + W + x0 + 1) : zero, u1 = (two && y > 0) ? __ldg(src + row - W + x0 + 1) : zero;
    auto tap = [](float c, float r, float l, float d, float u) {             // :217-222, one channel
        return div3(fadd(fadd(c, fmul(fadd(r, l), 0.5f)), fmul(fadd(d, u), 0.5f)));
    };
    float4 o0 = make_float4(tap(c0.x, c1.x, l0.x, d0.x, u0.x), tap(c0.y, c1.y, l0.y, d0.y, u0.y), tap(c0.z, c1.z, l0.z, d0.z, u0.z), 1.0f);
    float4 o1 = make_float4(tap(c1.x, r1.x, c0.x, d1.x, u1.x), tap(c1.y, r1.y, c0.y, d1.y, u1.y), tap(c1.z, r1.z, c0.z, d1.z, u1.z), 1.0f);
    if (q8) { o0 = quant8(o0); o1 = quant8(o1); }
    dst[row + x0] = o0;
    if (two) dst[row + x0 + 1] = o1;
    if (bytes) {
        bytes[row + x0] = make_uchar4((unsigned char)unorm8(o0.x), (unsigned char)unorm8(o0.y), (unsigned char)unorm8(o0.z), (unsigned char)unorm8(o0.w));
        if (two) bytes[row + x0 + 1] = make_uchar4((unsigned char)unorm8(o1.x), (unsigned char)unorm8(o1.y), (unsigned char)unorm8(o1.z), (unsigned char)unorm8(o1.w));
    }
}

// Micro-benchmarks for the two rooflines the path is measured against (SURVEY §8 d): how fast can this GPU fetch 56 useful
// bytes (a 32-B, a 16-B and an 8-B load, the traversal's per-visit pattern) from random 128-B records of a table of the
// scene's size, and how fast can it issue FP32 FMAs.  Independent addresses / chains: these are peaks, not models.
__global__ void __launch_bounds__(256) mb_gather_kernel(const float4 *__restrict__ table, uint32_t n_records, uint32_t iters,
                                                        float *__restrict__ sink) {
    uint32_t idx = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u;
    float acc = 0.0f;
    for (uint32_t i = 0; i < iters; i++) {
        idx = idx * 747796405u + 2891336453u;
        const float4 *rec = table + (size_t)((idx >> 8) % n_records) * 12;
        const uint32_t sxy = (idx & 3u) * 2u, sz = ((idx >> 2) & 1u) * 2u;      // any travel order, like the kernel
        const Line32 ab = ldg256(rec + sxy);
        const float4 z = __ldg(rec + 8 + sz);
        const float2 l = __ldg(reinterpret_cast<const float2 *>(rec + 9 + sz));
        acc += lo2f(ab.x) + hi2f(ab.y) + lo2f(ab.w) + z.z + l.x;
    }
    if (acc == 12345.678f) sink[0] = acc;                                       // keep the loads alive
}
__global__ void __launch_bounds__(256) mb_ffma_kernel(uint32_t iters, float *__restrict__ sink) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.0f, a2 = a0 + 2.0f, a3 = a0 + 3.0f, a4 = a0 + 4.0f, a5 = a0 + 5.0f, a6 = a0 + 6.0f, a7 = a0 + 7.0f;
    const float m = 1.000001f, c = 1e-7f;
    for (uint32_t i = 0; i < iters; i++) {
        a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
        a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
    }
    const float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678f) sink[0] = s;
}

template <bool C, bool D>
const void *kptr_rg(int bt) {
    if (bt == 64) return reinterpret_cast<const void *>(&trace_kernel_rg<C, D, 64>);
    if (bt == 128) return reinterpret_cast<const void *>(&trace_kernel_rg<C, D, 128>);
    return reinterpret_cast<const void *>(&trace_kernel_rg<C, D, kLargeBlock>);
}

template <bool C, bool D>
const void *kptr(int bt) {
    return bt == kSmallBlock ? reinterpret_cast<const void *>(&trace_kernel<C, D, kSmallBlock>)
                             : reinterpret_cast<const void *>(&trace_kernel<C, D, kLargeBlock>);
}

template <bool C, bool D>
const void *kptr_yt(int bt) {
    return bt == kSmallBlock ? reinterpret_cast<const void *>(&trace_ytab_kernel<C, D, kSmallBlock>)
                             : reinterpret_cast<const void *>(&trace_ytab_kernel<C, D, kLargeBlock>);
}

template <bool C, bool D>
const void *tail_ptr(bool yt) {
    return yt ? reinterpret_cast<const void *>(&trace_tail_kernel<C, D, true>) : reinterpret_cast<const void *>(&trace_tail_kernel<C, D, false>);
}

}  // namespace

const void *kernel_ptr(KernelChoice c) {
    if (c.regroup) {
        if (c.debug) return kptr_rg<true, true>(c.block_threads);
        return c.counters ? kptr_rg<true, false>(c.block_threads) : kptr_rg<false, false>(c.block_threads);
    }
    if (c.ytab) {
        if (c.debug) return kptr_yt<true, true>(c.block_threads);
        return c.counters ? kptr_yt<true, false>(c.block_threads) : kptr_yt<false, false>(c.block_threads);
    }
    if (c.debug) return kptr<true, true>(c.block_threads);
    return c.counters ? kptr<true, false>(c.block_threads) : kptr<false, false>(c.block_threads);
}

cudaError_t launch_trace(const KParams &p, KernelChoice c, unsigned blocks, size_t smem_bytes, cudaStream_t stream) {
    const void *fn = kernel_ptr(c);
    void *args[] = {const_cast<KParams *>(&p)};
    return cudaLaunchKernel(fn, dim3(blocks), dim3(c.block_threads), args, smem_bytes, stream);
}

cudaError_t launch_tail(const KParams &p, KernelChoice c, unsigned blocks, size_t smem_bytes, cudaStream_t stream) {
    const void *fn = c.debug ? tail_ptr<true, true>(c.ytab) : (c.counters ? tail_ptr<true, false>(c.ytab) : tail_ptr<false, false>(c.ytab));
    void *args[] = {const_cast<KParams *>(&p)};
    return cudaLaunchKernel(fn, dim3(blocks), dim3(kTailBlock), args, smem_bytes, stream);
}

cudaError_t launch_probe(const KParams &p, bool ytab, const float *rays, const uint32_t *slots, uint32_t n, float *t_out, uint32_t *index_out,
                         uint32_t *tally_out, cudaStream_t stream) {
    const unsigned blocks = (n + kProbeBlock - 1) / kProbeBlock;
    if (ytab)
        probe_rays_kernel<true><<<blocks, kProbeBlock, (size_t)(kProbeBlock / 32) * p.n_yiv * kYEntryStride, stream>>>(p, rays, slots, n, t_out, index_out, tally_out);
    else
        probe_rays_kernel<false><<<blocks, kProbeBlock, 0, stream>>>(p, rays, slots, n, t_out, index_out, tally_out);
    return cudaGetLastError();
}

cudaError_t launch_mb_gather(const void *table, uint32_t n_records, uint32_t iters, unsigned blocks, float *sink, cudaStream_t stream) {
    mb_gather_kernel<<<blocks, 256, 0, stream>>>(reinterpret_cast<const float4 *>(table), n_records, iters, sink);
    return cudaGetLastError();
}
cudaError_t launch_mb_ffma(uint32_t iters, unsigned blocks, float *sink, cudaStream_t stream) {
    mb_ffma_kernel<<<blocks, 256, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}

cudaError_t launch_scatter_all(const float *gathered, float *image, const mm_chunk *chunks, uint32_t world, uint32_t max_count,
                               uint32_t n_groups, uint32_t chunk, uint32_t W, uint32_t H, cudaStream_t stream) {
    const uint32_t ppc = chunk * chunk;
    const uint64_t n = (uint64_t)world * max_count * ppc;
    if (n == 0) return cudaSuccess;
    scatter_all_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const float4 *>(gathered),
                                                                       reinterpret_cast<float4 *>(image), chunks, world, max_count,
                                                                       n_groups, chunk, ppc, W, H);
    return cudaGetLastError();
}

cudaError_t launch_blur(const float *src, float *dst, uint32_t W, uint32_t H, cudaStream_t stream, bool quant8, uint8_t *bytes) {
    if (W == 0 || H == 0) return cudaSuccess;
    dim3 grid((W + 511) / 512, H);                                            // two pixels per thread
    blur_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const float4 *>(src), reinterpret_cast<float4 *>(dst), W, H, quant8,
                                          reinterpret_cast<uchar4 *>(bytes));
    return cudaGetLastError();
}

cudaError_t launch_div3_selftest(unsigned long long *d_mismatches, cudaStream_t stream) {
    div3_selftest_kernel<<<148 * 16, 256, 0, stream>>>(d_mismatches);
    return cudaGetLastError();
}

cudaError_t launch_quot_selftest(uint64_t n, uint64_t seed, unsigned long long *d_mismatches, cudaStream_t stream) {
    quot_selftest_kernel<<<148 * 8, 256, 0, stream>>>(n, seed, d_mismatches);
    return cudaGetLastError();
}

cudaError_t launch_scatter(const float *tiles, float *image, const mm_chunk *chunks, uint32_t /*grid_groups*/, uint32_t group_first,
                           uint32_t group_step, uint32_t group_count, uint32_t chunk, uint32_t W, uint32_t H, cudaStream_t stream) {
    const uint32_t ppc = chunk * chunk;
    const uint64_t n = (uint64_t)group_count * ppc;
    if (n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    scatter_kernel<<<blocks, 256, 0, stream>>>(reinterpret_cast<const float4 *>(tiles), reinterpret_cast<float4 *>(image), chunks,
                                               group_first, group_step, group_count, chunk, ppc, W, H);
    return cudaGetLastError();
}

}  // namespace mmk
