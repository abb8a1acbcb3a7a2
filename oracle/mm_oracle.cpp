// mm_oracle.cpp — CPU ORACLE for mirror-maze's per-pixel render kernel.  TEST INFRASTRUCTURE, NOT PRODUCT:
// only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this.
//
// A literal scalar fp32 restatement of the reference's Metal kernel, function by function:
//   random()                  reference src/shaders.metal:181-186
//   quat_inv/quat_dot/quat_mult                         :159-172
//   intersect_aabb                                       :87-95
//   ray_rect_intersect                                   :51-67
//   intersect_bvh_iterative                              :115-156
//   compute_shader (mapping, ray-gen, seed, bounce loop, tone-map, reduction, store)   :245-368
//
// PARITY PIN: the reference has no tests, golden vectors or fixtures for this path (SURVEY §4, §8 c) and its binary only
// runs on Apple GPUs (fast-math + FTZ AIR).  But its device SOURCE is a C++ dialect: oracle/ref_shader/ compiles reference
// src/shaders.metal, unmodified, with g++ (msl_shim.h stands in for <metal_stdlib>) into oracle/_ref/libref_shader.so and
// runs the reference's own compute_shader on the CPU.  tests/test_ref_shader.py pins this file to it — random(),
// intersect_aabb, ray_rect_intersect, quat_mult on random and edge inputs, and whole dispatches image for image (every
// shape the unmodified shader can address: its literal limits 5 / 15, spp 8..256, chunk 1..8); the digests of its images
// are committed under tests/golden/.  What the reference cannot pin stays this file's decision, shared with the shim: the
// arithmetic of Metal's library functions (below) and everything the shader hard-wires (other limits, spp < 8, full
// frames) — for those: the known-answer vectors of SURVEY Appendix E, the independent numpy-float32 transcription
// (oracle/np_oracle.py) compared path by path, and the committed fixtures.
//
// Canonical arithmetic (SURVEY §8 a-0) — the kernel under test obeys the same rules:
//   fp32 only; every + - * / sqrt is one IEEE-754 round-to-nearest-even operation (build with
//   -ffp-contract=off, never -ffast-math); dot(a,b) = (a.x*b.x + a.y*b.y) + a.z*b.z; cross as maths.rs:130-136;
//   length = sqrt(dot(v,v)); normalize(v) = v / length(v) component-wise; reflect(I,N) = I - (2*dot(N,I))*N;
//   sign(x) in {1,-1,0} with sign(NaN) = 0; min/max return the non-NaN operand; float->uint truncates toward
//   zero and saturates to [0, 2^32-1] with NaN -> 0; uint->float rounds to nearest even.
//   The literal slab test divides by the direction (no reciprocal) and the literal rect test recomputes the
//   normal and edge lengths per call; both are kept.
//
// Build: g++ -O2 -ffp-contract=off -fopenmp -shared -fPIC (oracle/Makefile).
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "../include/mirror_maze_cuda.h"

namespace {

struct f3 { float x, y, z; };

inline f3 mk(float x, float y, float z) { f3 r = {x, y, z}; return r; }
inline f3 ld(const mm_float3 &a) { return mk(a.x, a.y, a.z); }
inline f3 add(f3 a, f3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
// Store into an RGBA8Unorm texture and read back (reference src/main.rs:702-709 creates the screen as RGBA8Unorm): Metal converts
// float -> unorm8 as round-to-nearest-even of clamp(v, 0, 1) * 255 (NaN -> 0) and unorm8 -> float as k / 255.
inline float quant8(float v) {
    float c = v > 0.0f ? v : 0.0f;                 // also maps NaN to 0
    c = c < 1.0f ? c : 1.0f;
    return std::nearbyintf(c * 255.0f) / 255.0f;   // default rounding mode: to nearest even
}
inline f3 sub(f3 a, f3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
inline f3 mul(f3 a, f3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
inline f3 scale(f3 a, float s) { return mk(a.x * s, a.y * s, a.z * s); }
inline float dot(f3 a, f3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
inline f3 cross(f3 a, f3 b) { return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
inline float length(f3 a) { return std::sqrt(dot(a, a)); }
inline f3 normalize(f3 a) { float l = length(a); return mk(a.x / l, a.y / l, a.z / l); }
inline f3 reflect(f3 i, f3 n) { return sub(i, scale(n, 2.0f * dot(n, i))); }
inline float sign(float x) { return x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f); }
inline float fmin_c(float a, float b) { return (b < a || a != a) ? b : a; }   // non-NaN operand
inline float fmax_c(float a, float b) { return (b > a || a != a) ? b : a; }
inline uint32_t f2u_sat(float f) {
    if (!(f > 0.0f)) return 0u;                 // NaN, negatives, zero
    if (f >= 4294967296.0f) return 0xFFFFFFFFu;
    return (uint32_t)f;                         // in range: C++ truncation toward zero
}

struct Ray { f3 ori, dir; float t; uint32_t index; };   // shaders.metal:12-17

struct Scene {
    const mm_plane *rects; uint32_t n_rects;
    const mm_bvh_node *nodes; uint32_t n_nodes;
    const uint32_t *indices;
    const uint8_t *materials;
    const mm_float4 *emissions;
};

struct Counts {
    uint64_t rays = 0, inner = 0, leaf = 0, rect = 0, hits = 0, max_stack = 0; bool overflow = false;
    bool rcp = false;                          // MM_FLAG_RCP_SLAB
    std::vector<uint16_t> *trace = nullptr;   // optional event trace for scheduling studies (tools/sched_sim.py)
};

// shaders.metal:181-186
inline float random_f(uint32_t &state) {
    state = state * 747796405u + 291336453u;
    uint32_t result = ((state >> ((state >> 28) + 4u)) ^ state) * 277803737u;
    result = (result >> 22) ^ result;
    return (float)result / 4294967296.0f;      // MSL literal 4294967295.0 is a float: rounds to 2^32
}

// shaders.metal:159-172
struct f4 { float x, y, z, w; };
inline f4 quat_dot(f4 q1, f4 q2) {
    f3 a = mk(q1.x, q1.y, q1.z), b = mk(q2.x, q2.y, q2.z);
    float s = q1.w * q2.w - dot(a, b);
    f3 v = add(add(cross(a, b), scale(b, q1.w)), scale(a, q2.w));
    f4 r = {v.x, v.y, v.z, s};
    return r;
}
inline f3 quat_mult(f3 vec, f4 quat) {
    f4 inv = {-quat.x, -quat.y, -quat.z, quat.w};
    f4 v4 = {vec.x, vec.y, vec.z, 0.0f};
    f4 r = quat_dot(quat_dot(inv, v4), quat);
    return mk(r.x, r.y, r.z);
}

// shaders.metal:87-95
inline float intersect_aabb(const Ray &beam, f3 bmin, f3 bmax) {
    float tx1 = (bmin.x - beam.ori.x) / beam.dir.x, tx2 = (bmax.x - beam.ori.x) / beam.dir.x;
    float tmin = fmin_c(tx1, tx2), tmax = fmax_c(tx1, tx2);
    float ty1 = (bmin.y - beam.ori.y) / beam.dir.y, ty2 = (bmax.y - beam.ori.y) / beam.dir.y;
    tmin = fmax_c(tmin, fmin_c(ty1, ty2)); tmax = fmin_c(tmax, fmax_c(ty1, ty2));
    float tz1 = (bmin.z - beam.ori.z) / beam.dir.z, tz2 = (bmax.z - beam.ori.z) / beam.dir.z;
    tmin = fmax_c(tmin, fmin_c(tz1, tz2)); tmax = fmin_c(tmax, fmax_c(tz1, tz2));
    if (tmax >= tmin && tmin < beam.t && tmax > 0.0f) return tmin; else return 1e30f;
}

// Opt-in variant (MM_FLAG_RCP_SLAB): the same test with t = (b - o) * (1/d), one IEEE reciprocal per axis — what a
// fast-math compile of :88-93 amounts to.  Not the default; only used when the caller asks for it.
inline float intersect_aabb_rcp(const Ray &beam, f3 bmin, f3 bmax) {
    float ix = 1.0f / beam.dir.x, iy = 1.0f / beam.dir.y, iz = 1.0f / beam.dir.z;
    float tx1 = (bmin.x - beam.ori.x) * ix, tx2 = (bmax.x - beam.ori.x) * ix;
    float tmin = fmin_c(tx1, tx2), tmax = fmax_c(tx1, tx2);
    float ty1 = (bmin.y - beam.ori.y) * iy, ty2 = (bmax.y - beam.ori.y) * iy;
    tmin = fmax_c(tmin, fmin_c(ty1, ty2)); tmax = fmin_c(tmax, fmax_c(ty1, ty2));
    float tz1 = (bmin.z - beam.ori.z) * iz, tz2 = (bmax.z - beam.ori.z) * iz;
    tmin = fmax_c(tmin, fmin_c(tz1, tz2)); tmax = fmin_c(tmax, fmax_c(tz1, tz2));
    if (tmax >= tmin && tmin < beam.t && tmax > 0.0f) return tmin; else return 1e30f;
}

// shaders.metal:51-67
inline void ray_rect_intersect(Ray &beam, const mm_plane &mirror, uint32_t index) {
    f3 mo = ld(mirror.origin), mv = ld(mirror.v), mu = ld(mirror.u);
    f3 rect_norm = normalize(cross(mv, mu));
    float norm_check = dot(beam.dir, rect_norm);
    float a = dot(sub(mo, beam.ori), rect_norm) / norm_check;
    f3 intersection = add(beam.ori, scale(beam.dir, a));
    f3 rect_vect = sub(intersection, mo);
    float d1 = dot(rect_vect, mv) / length(mv);
    float d2 = dot(rect_vect, mu) / length(mu);
    if ((0.0f <= d1 && d1 <= length(mv)) && (0.0f <= d2 && d2 <= length(mu)) && norm_check != 0.0f && a > 0.1f && a < beam.t) {
        beam.t = a;
        beam.index = index;
    }
}

// shaders.metal:115-156
inline void intersect_bvh_iterative(Ray &beam, const Scene &sc, Counts &c) {
    uint32_t node = 0;                // &nodes[0]; the root box is never tested
    uint32_t stack[50];
    uint32_t head = 0;
    uint32_t run = 0;
    c.rays++;
    if (c.trace) {   // segment header: 0xFFF0 | octant, then |dir.y| / |dir| quantised to 0..255 (a cheap predictor of traversal length)
        c.trace->push_back((uint16_t)(0xFFF0u | (beam.dir.x < 0.0f ? 1u : 0u) | (beam.dir.y < 0.0f ? 2u : 0u) | (beam.dir.z < 0.0f ? 4u : 0u)));
        float l = std::sqrt(beam.dir.x * beam.dir.x + beam.dir.y * beam.dir.y + beam.dir.z * beam.dir.z);
        float q = l > 0.0f ? std::fabs(beam.dir.y) / l * 255.0f : 0.0f;
        c.trace->push_back((uint16_t)(q < 0.0f ? 0.0f : (q > 255.0f ? 255.0f : q)));
    }
    while (true) {
        const mm_bvh_node &nd = sc.nodes[node];
        if (nd.tri_count > 0) {
            c.leaf++;
            if (c.trace) { c.trace->push_back((uint16_t)run); c.trace->push_back((uint16_t)nd.tri_count); run = 0; }
            for (uint32_t i = 0; i < nd.tri_count; i++) {
                uint32_t pi = sc.indices[nd.left_first + i];
                ray_rect_intersect(beam, sc.rects[pi], pi);
                c.rect++;
            }
            if (head == 0) break; else node = stack[--head];
            continue;
        }
        c.inner++;
        run++;
        uint32_t left = nd.left_first, right = nd.left_first + 1;
        float dist1 = c.rcp ? intersect_aabb_rcp(beam, ld(sc.nodes[left].aabb_min), ld(sc.nodes[left].aabb_max))
                            : intersect_aabb(beam, ld(sc.nodes[left].aabb_min), ld(sc.nodes[left].aabb_max));
        float dist2 = c.rcp ? intersect_aabb_rcp(beam, ld(sc.nodes[right].aabb_min), ld(sc.nodes[right].aabb_max))
                            : intersect_aabb(beam, ld(sc.nodes[right].aabb_min), ld(sc.nodes[right].aabb_max));
        if (dist1 > dist2) {
            float temp = dist1; dist1 = dist2; dist2 = temp;
            uint32_t nemp = left; left = right; right = nemp;
        }
        if (dist1 == 1e30f) {
            if (head == 0) break; else node = stack[--head];
        } else {
            node = left;
            if (dist2 != 1e30f) {
                if (head >= 50) { c.overflow = true; break; }   // the reference would write past its array
                stack[head++] = right;
                if (head > c.max_stack) c.max_stack = head;
            }
        }
    }
    if (c.trace) { c.trace->push_back((uint16_t)run); c.trace->push_back(0xFFFFu); }   // trailing interior run, end of segment
}

struct Job {
    Scene sc;
    const uint8_t *noise; uint32_t nw, nh;
    mm_uniform uni;
    mm_params par;
    const mm_chunk *chunks; uint32_t n_chunks;
};

// noise.sample(s, float2(gid)) with sampler(address::repeat, filter::nearest), normalised coordinates
// (shaders.metal:288,291): wrap = x - floor(x), texel = min(int(wrap * size), size - 1).  Integer-valued
// coordinates therefore always address texel (0,0); the rule is implemented, not the constant.
inline void sample_noise(const Job &j, float u, float v, float out[4]) {
    float fu = u - std::floor(u), fv = v - std::floor(v);
    int ix = (int)std::floor(fu * (float)j.nw), iy = (int)std::floor(fv * (float)j.nh);
    if (ix > (int)j.nw - 1) ix = (int)j.nw - 1;
    if (iy > (int)j.nh - 1) iy = (int)j.nh - 1;
    if (ix < 0) ix = 0;
    if (iy < 0) iy = 0;
    const uint8_t *t = j.noise + 4 * ((size_t)iy * j.nw + (size_t)ix);
    for (int c = 0; c < 4; c++) out[c] = (float)t[c] / 255.0f;   // RGBA8Unorm -> float
}

// One thread of compute_shader (shaders.metal:261-344).  Returns the tone-mapped sample.
inline f3 trace_thread(const Job &j, uint32_t tgx, uint32_t tgy, uint32_t flat, uint32_t dimx, uint32_t dimy,
                       Counts &c, uint32_t *first_hit, uint32_t *segments, uint32_t *mirror_out, float *radiance,
                       uint32_t *pixel_out /*x,y*/) {
    const mm_uniform &U = j.uni;
    float width = U.view_width, height = U.view_height;
    uint32_t chunk = U.chunk_width;
    uint32_t ppc = chunk * chunk;
    uint32_t pixel_buffer_index = tgx + tgy * j.par.grid_x;            // :266, row stride = grid width
    mm_chunk px = j.chunks[pixel_buffer_index];                        // :267
    uint32_t total_threads = dimx * dimy;                              // :269
    uint32_t gx = flat % dimx, gy = flat / dimx;                       // inverse of :271
    uint32_t pixel_number = flat / (total_threads / ppc);              // :272
    uint32_t pixel_y_add = pixel_number % chunk;                       // :273
    uint32_t pixel_x_add = pixel_number / chunk;                       // :274
    uint32_t pxx = px.x + pixel_x_add, pxy = px.y + pixel_y_add;       // :275
    pixel_out[0] = pxx; pixel_out[1] = pxy;
    uint32_t texid_x = tgx * dimx + gx, texid_y = tgy * dimy + gy;     // thread_position_in_grid

    const mm_camera &cam = U.cam;
    f3 center = ld(cam.camera_center);
    float pnx = (float)pxx / width, pny = (float)pxy / height;         // :281
    f3 viewport_corner = sub(center, mk(cam.viewport.x / 2.0f, cam.viewport.y / 2.0f, -cam.focal_length));   // :282
    f3 ray_dir = normalize(sub(add(viewport_corner, mk(pnx * cam.viewport.x, pny * cam.viewport.y, 0.0f)), center));   // :283
    f4 rot = {cam.rotation.x, cam.rotation.y, cam.rotation.z, cam.rotation.w};
    ray_dir = quat_mult(ray_dir, rot);                                 // :284

    Ray beam;
    f3 color = mk(1.0f, 1.0f, 1.0f);                                   // :289
    f3 incoming_light = mk(0.0f, 0.0f, 0.0f);                          // :290
    float ns[4];
    sample_noise(j, (float)gx, (float)gy, ns);                         // :291
    int bounce_limit = (int)j.par.bounce_limit;                        // :294 (uniform instead of 5)
    int mirror_limit = (int)j.par.mirror_limit;                        // :295 (uniform instead of 15)
    // :298 — float + uint promotes to float; products wrap in u32 first; evaluated left to right.
    float seed_f = (((ns[0] + ns[1]) + (float)(texid_x * 15823u)) + (float)(texid_y * 9737333u)) + (float)U.time;
    uint32_t state = f2u_sat(seed_f);

    beam.ori = center;                                                 // :302
    float r1 = random_f(state), r2 = random_f(state);
    beam.dir = add(ray_dir, scale(mk((r1 - 0.5f) * 2.0f, (r2 - 0.5f) * 2.0f, 0.0f), 0.001f));   // :303
    beam.t = 1e30f;
    beam.index = 0xFFFFFFFFu;
    int mirror_hits = 0;
    uint32_t seg = 0, fh = 0xFFFFFFFFu;
    for (int n = 0; n < bounce_limit + mirror_hits; n++) {             // :306
        intersect_bvh_iterative(beam, j.sc, c);                        // :307
        seg++;
        if (c.overflow) break;
        if (beam.t < 1e30f) {                                          // :308
            c.hits++;
            if (n == 0) fh = beam.index;
            const mm_plane &m = j.sc.rects[beam.index];
            f3 mirror_norm = normalize(cross(ld(m.v), ld(m.u)));       // :309
            float beam_side = -sign(dot(beam.dir, mirror_norm));       // :310
            if (j.sc.materials[beam.index] == 0 || beam_side == -1.0f) {   // :311
                const mm_float4 &e = j.sc.emissions[beam.index];
                f3 emitted_light = scale(mk(e.x, e.y, e.z), e.w);      // :312
                incoming_light = add(incoming_light, mul(emitted_light, color));   // :313
                color = mul(color, ld(m.color));                       // :314
                f3 random_dir;
                {
                    float a = random_f(state), b = random_f(state), d = random_f(state);   // :315
                    random_dir = mk((a - 0.5f) * 2.0f, (b - 0.5f) * 2.0f, (d - 0.5f) * 2.0f);
                }
                while (length(random_dir) > 1.0f) {                    // :316-318
                    float a = random_f(state), b = random_f(state), d = random_f(state);
                    random_dir = mk((a - 0.5f) * 2.0f, (b - 0.5f) * 2.0f, (d - 0.5f) * 2.0f);
                }
                random_dir = normalize(random_dir);                    // :319
                beam.ori = add(beam.ori, scale(beam.dir, beam.t));     // :320
                beam.dir = normalize(add(random_dir, scale(mirror_norm, beam_side)));   // :321
                beam.t = 1e30f;                                        // :323
            } else {
                mirror_hits++;                                         // :325
                if (mirror_hits < mirror_limit) {                      // :326
                    incoming_light = add(incoming_light, scale(ld(m.color), 0.005f));   // :327
                    beam.ori = add(beam.ori, scale(beam.dir, beam.t)); // :328
                    beam.dir = normalize(reflect(beam.dir, mirror_norm));   // :329
                    beam.t = 1e30f;                                    // :330
                } else {
                    break;                                             // :333
                }
            }
        } else {
            break;   // :337-338: the sky term is multiplied by 0.0 — adds nothing
        }
    }
    if (c.trace) c.trace->push_back(0xFFFEu);   // end of path
    if (first_hit) *first_hit = fh;
    if (segments) *segments = seg;
    if (mirror_out) *mirror_out = (uint32_t)mirror_hits;
    if (radiance) { radiance[0] = incoming_light.x; radiance[1] = incoming_light.y; radiance[2] = incoming_light.z; }
    // :344
    return mk(std::sqrt(fmax_c(incoming_light.x, 0.0f)), std::sqrt(fmax_c(incoming_light.y, 0.0f)),
              std::sqrt(fmax_c(incoming_light.z, 0.0f)));
}

int validate(const mm_uniform *uni, const mm_params *p, uint32_t n_chunks, uint32_t *T_out) {
    if (!uni || !p) return MM_ERR_INVALID;
    uint32_t spp = p->spp, chunk = uni->chunk_width;
    if (spp == 0 || (spp & (spp - 1)) || spp > 256) return MM_ERR_UNSUPPORTED;
    if (chunk == 0 || chunk > 64) return MM_ERR_UNSUPPORTED;
    uint64_t T = (uint64_t)chunk * chunk * spp;
    if (T > (1u << 20)) return MM_ERR_UNSUPPORTED;
    if (T > 32 && (T % 32) != 0) return MM_ERR_UNSUPPORTED;   // the virtual threadgroup is (32, T/32): Metal groups are rows of the execution width
    if (p->grid_x == 0 || p->grid_y == 0 || (uint64_t)p->grid_x * p->grid_y != n_chunks) return MM_ERR_INVALID;
    if (p->bounce_limit > 4096 || p->mirror_limit > 4096) return MM_ERR_INVALID;
    *T_out = (uint32_t)T;
    return MM_OK;
}

}  // namespace

extern "C" {

// Same contract as mm_render (include/mirror_maze_cuda.h) with the scene passed by pointer.
int mmo_render(const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes,
               const uint32_t *indices, const uint8_t *materials, const mm_float4 *emissions,
               const uint8_t *noise_rgba8, uint32_t noise_w, uint32_t noise_h,
               const mm_uniform *uni, const mm_params *params, const mm_chunk *chunks, uint32_t n_chunks,
               float *out_rgba, mm_counters *counters, const mm_debug *debug, int n_threads) {
    if (!planes || !nodes || !indices || !materials || !emissions || !noise_rgba8 || !chunks || !out_rgba) return MM_ERR_INVALID;
    if (n_planes == 0 || n_nodes == 0 || noise_w == 0 || noise_h == 0) return MM_ERR_INVALID;
    uint32_t T = 0;
    int rc = validate(uni, params, n_chunks, &T);
    if (rc != MM_OK) return rc;
    Job j;
    j.sc = {planes, n_planes, nodes, n_nodes, indices, materials, emissions};
    j.noise = noise_rgba8; j.nw = noise_w; j.nh = noise_h;
    j.uni = *uni; j.par = *params; j.chunks = chunks; j.n_chunks = n_chunks;
    const uint32_t n_groups = params->grid_x * params->grid_y;
    uint32_t first = params->group_first, step = params->group_step ? params->group_step : 1, count = params->group_count;
    if (count == 0) { first = 0; step = 1; count = n_groups; }
    if ((uint64_t)first + (uint64_t)(count - 1) * step >= n_groups) return MM_ERR_INVALID;
    const uint32_t dimx = T < 32 ? T : 32, dimy = T / dimx;
    const uint32_t spp = params->spp, ppc = uni->chunk_width * uni->chunk_width;
    const uint32_t W = (uint32_t)uni->view_width, H = (uint32_t)uni->view_height;
    Counts total;
    int overflow = 0;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel
    {
        Counts c;
        c.rcp = (params->flags & MM_FLAG_RCP_SLAB) != 0;
        std::vector<f3> test(T);
        std::vector<uint32_t> pix(2 * (size_t)T);
#pragma omp for schedule(dynamic, 8)
        for (int64_t k = 0; k < (int64_t)count; k++) {
            uint32_t g = first + (uint32_t)k * step;
            uint32_t tgx = g % params->grid_x, tgy = g / params->grid_x;
            for (uint32_t flat = 0; flat < T; flat++) {
                size_t e = (size_t)k * T + flat;
                test[flat] = trace_thread(j, tgx, tgy, flat, dimx, dimy, c,
                                          debug && debug->first_hit ? debug->first_hit + e : nullptr,
                                          debug && debug->segments ? debug->segments + e : nullptr,
                                          debug && debug->mirror_hits ? debug->mirror_hits + e : nullptr,
                                          debug && debug->radiance ? debug->radiance + 3 * e : nullptr, &pix[2 * (size_t)flat]);
            }
            // shaders.metal:347-358 — three barrier-separated pairwise phases over the whole group.  For spp < 8
            // only the phases whose stride stays inside one pixel are run (SURVEY §8 D12 generalisation).
            for (uint32_t stride = 1; stride <= 4 && stride < spp; stride *= 2)
                for (uint32_t flat = 0; flat < T; flat += 2 * stride) test[flat] = add(test[flat], test[flat + stride]);
            // :360-366 — first thread of each pixel: serial sum of the octets, divide by max_index, store.
            for (uint32_t pn = 0; pn < ppc; pn++) {
                uint32_t base = pn * spp;
                for (uint32_t i = 1; i < spp / 8; i++) test[base] = add(test[base], test[base + 8 * i]);
                float d = (float)(int)spp;
                f3 r = mk(test[base].x / d, test[base].y / d, test[base].z / d);
                float alpha = 1.0f;
                if (params->flags & MM_FLAG_SCREEN_RGBA8) {   // main.rs:702-709: the screen is RGBA8Unorm; a store quantises, a read returns k / 255
                    r = mk(quant8(r.x), quant8(r.y), quant8(r.z));
                    alpha = quant8(alpha);
                }
                uint32_t x = pix[2 * (size_t)base], y = pix[2 * (size_t)base + 1];
                if (x < W && y < H) {
                    float *o = out_rgba + 4 * ((size_t)y * W + x);
                    o[0] = r.x; o[1] = r.y; o[2] = r.z; o[3] = alpha;
                }
            }
        }
#pragma omp critical
        {
            total.rays += c.rays; total.inner += c.inner; total.leaf += c.leaf; total.rect += c.rect; total.hits += c.hits;
            if (c.max_stack > total.max_stack) total.max_stack = c.max_stack;
            if (c.overflow) overflow = 1;
        }
    }
    if (counters) {
        counters->paths = (uint64_t)count * T;
        counters->rays = total.rays; counters->inner_visits = total.inner; counters->leaf_visits = total.leaf;
        counters->rect_tests = total.rect; counters->hits = total.hits; counters->literal_rays = 0;
        counters->max_stack = total.max_stack;
    }
    return overflow ? MM_ERR_BVH : MM_OK;
}

// Event trace of a render (single-threaded): per path, per segment, 0xFFF0|octant then (interior-run, leaf-count) pairs, 0xFFFF after the
// trailing interior run of a segment, 0xFFFE after a path.  Returns the number of u16 written (or needed if cap is small).
uint64_t mmo_trace(const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes, const uint32_t *indices,
                   const uint8_t *materials, const mm_float4 *emissions, const uint8_t *noise_rgba8, uint32_t noise_w, uint32_t noise_h,
                   const mm_uniform *uni, const mm_params *params, const mm_chunk *chunks, uint32_t n_chunks, uint16_t *out, uint64_t cap) {
    uint32_t T = 0;
    if (validate(uni, params, n_chunks, &T) != MM_OK) return 0;
    Job j;
    j.sc = {planes, n_planes, nodes, n_nodes, indices, materials, emissions};
    j.noise = noise_rgba8; j.nw = noise_w; j.nh = noise_h;
    j.uni = *uni; j.par = *params; j.chunks = chunks; j.n_chunks = n_chunks;
    uint32_t first = params->group_first, step = params->group_step ? params->group_step : 1, count = params->group_count;
    if (count == 0) { first = 0; step = 1; count = params->grid_x * params->grid_y; }
    const uint32_t dimx = T < 32 ? T : 32, dimy = T / dimx;
    std::vector<uint16_t> tr;
    Counts c;
    c.trace = &tr;
    uint32_t pix[2];
    for (uint32_t k = 0; k < count; k++) {
        uint32_t g = first + k * step;
        for (uint32_t flat = 0; flat < T; flat++)
            trace_thread(j, g % params->grid_x, g / params->grid_x, flat, dimx, dimy, c, nullptr, nullptr, nullptr, nullptr, pix);
    }
    if (out && tr.size() <= cap) std::memcpy(out, tr.data(), tr.size() * sizeof(uint16_t));
    return tr.size();
}

// intersect_bvh_iterative ray by ray, the reference for mm_trace_rays: rays n x 8 floats (ori.xyz, dir.xyz, starting t, alive),
// index_in the starting beam.index (plane index; null: 0xFFFFFFFF), flags & MM_FLAG_RCP_SLAB selects the reciprocal-multiply
// slab test.  Per ray: t, index and counts n x 5 (inner, leaf, rect, max_stack, stack overflow).  A dead ray (alive == 0)
// keeps its t and index and counts nothing.  Returns MM_ERR_BVH when some ray overflowed the reference's 50-entry stack.
int mmo_trace_rays(const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes, const uint32_t *indices,
                   uint32_t flags, const float *rays, const uint32_t *index_in, uint32_t n, float *t_out, uint32_t *index_out,
                   uint64_t *counts_out, int n_threads) {
    if (!planes || !nodes || !indices || !rays || !t_out || !index_out || !counts_out || n_planes == 0 || n_nodes == 0) return MM_ERR_INVALID;
    const Scene sc = {planes, n_planes, nodes, n_nodes, indices, nullptr, nullptr};
    int overflow = 0;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel for schedule(dynamic, 256) reduction(| : overflow)
    for (int64_t i = 0; i < (int64_t)n; i++) {
        const float *r = rays + 8 * i;
        Ray beam;
        beam.ori = mk(r[0], r[1], r[2]); beam.dir = mk(r[3], r[4], r[5]); beam.t = r[6];
        beam.index = index_in ? index_in[i] : 0xFFFFFFFFu;
        Counts c;
        c.rcp = (flags & MM_FLAG_RCP_SLAB) != 0;
        if (r[7] != 0.0f) intersect_bvh_iterative(beam, sc, c);
        t_out[i] = beam.t;
        index_out[i] = beam.index;
        uint64_t *o = counts_out + 5 * i;
        o[0] = c.inner; o[1] = c.leaf; o[2] = c.rect; o[3] = c.max_stack; o[4] = c.overflow ? 1u : 0u;
        overflow |= c.overflow ? 1 : 0;
    }
    return overflow ? MM_ERR_BVH : MM_OK;
}

// Unit-level entry points for known-answer tests.
float mmo_random(uint32_t *state) { return random_f(*state); }
uint32_t mmo_random_word(uint32_t *state) {   // the u32 `result` before the float conversion
    *state = *state * 747796405u + 291336453u;
    uint32_t result = ((*state >> ((*state >> 28) + 4u)) ^ *state) * 277803737u;
    return (result >> 22) ^ result;
}
uint32_t mmo_seed(float nx, float ny, uint32_t texid_x, uint32_t texid_y, uint32_t time) {
    float s = (((nx + ny) + (float)(texid_x * 15823u)) + (float)(texid_y * 9737333u)) + (float)time;
    return f2u_sat(s);
}
float mmo_intersect_aabb(const float ori[3], const float dir[3], float t, const float bmin[3], const float bmax[3]) {
    Ray b; b.ori = mk(ori[0], ori[1], ori[2]); b.dir = mk(dir[0], dir[1], dir[2]); b.t = t; b.index = 0;
    return intersect_aabb(b, mk(bmin[0], bmin[1], bmin[2]), mk(bmax[0], bmax[1], bmax[2]));
}
// returns 1 and writes t when the rect is hit
int mmo_ray_rect(const float ori[3], const float dir[3], float t, const mm_plane *rect, float *t_out) {
    Ray b; b.ori = mk(ori[0], ori[1], ori[2]); b.dir = mk(dir[0], dir[1], dir[2]); b.t = t; b.index = 0xFFFFFFFFu;
    ray_rect_intersect(b, *rect, 7u);
    if (t_out) *t_out = b.t;
    return b.index == 7u ? 1 : 0;
}
void mmo_quat_mult(const float v[3], const float q[4], float out[3]) {
    f4 qq = {q[0], q[1], q[2], q[3]};
    f3 r = quat_mult(mk(v[0], v[1], v[2]), qq);
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}
int mmo_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

}  // extern "C"
