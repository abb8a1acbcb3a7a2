// trace_device.cuh — device code shared by the two trace kernels (render_kernel.cu: one thread per path, segment-synchronous
// warps; pool_kernel.cu: persistent warps over a ray pool in shared memory): the IEEE arithmetic helpers, the RNG, the packed
// exact slab test, the rect test, the warp-voted traversal, ray generation and shading.  Everything here follows reference
// src/shaders.metal line by line (citations inline) under the arithmetic contract of SURVEY 8 a-0; both kernels call the same
// functions, so their results are the same bits by construction.  Included inside an anonymous namespace of each .cu file.
#pragma once
#include "render_kernel.cuh"

namespace mmk {
namespace {

struct V3 { float x, y, z; };

__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fsqrt(float a) { return __fsqrt_rn(a); }

__device__ __forceinline__ V3 mk(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ V3 add3(V3 a, V3 b) { return mk(fadd(a.x, b.x), fadd(a.y, b.y), fadd(a.z, b.z)); }
__device__ __forceinline__ V3 sub3(V3 a, V3 b) { return mk(fsub(a.x, b.x), fsub(a.y, b.y), fsub(a.z, b.z)); }
__device__ __forceinline__ V3 mul3(V3 a, V3 b) { return mk(fmul(a.x, b.x), fmul(a.y, b.y), fmul(a.z, b.z)); }
__device__ __forceinline__ V3 scale3(V3 a, float s) { return mk(fmul(a.x, s), fmul(a.y, s), fmul(a.z, s)); }
__device__ __forceinline__ float dot3(V3 a, V3 b) { return fadd(fadd(fmul(a.x, b.x), fmul(a.y, b.y)), fmul(a.z, b.z)); }
__device__ __forceinline__ V3 cross3(V3 a, V3 b) {
    return mk(fsub(fmul(a.y, b.z), fmul(a.z, b.y)), fsub(fmul(a.z, b.x), fmul(a.x, b.z)), fsub(fmul(a.x, b.y), fmul(a.y, b.x)));
}
__device__ __forceinline__ float length3(V3 a) { return fsqrt(dot3(a, a)); }
__device__ __forceinline__ V3 normalize3(V3 a) { float l = length3(a); return mk(fdiv(a.x, l), fdiv(a.y, l), fdiv(a.z, l)); }
__device__ __forceinline__ V3 reflect3(V3 i, V3 n) { return sub3(i, scale3(n, fmul(2.0f, dot3(n, i)))); }
__device__ __forceinline__ float sign1(float x) { return x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f); }

// random() of shaders.metal:181-186 (state = state * 747796405 + 291336453; PCG output hash; float(result) / 2^32) is only
// ever used as (random(state) - 0.5) * 2.0 (:303, :315-317), evaluated here as one FMA: float(r) * 2^-32 is an exact scaling, and so is the
// final * 2, hence 2 * RN(f * 2^-32 - 0.5) == RN(f * 2^-31 - 1), which is what the FMA's single rounding returns
// (tests/test_oracle.py checks the identity over 2^24 random words and the edge words).
__device__ __forceinline__ float rnd_pm1(uint32_t &state) {
    state = state * 747796405u + 291336453u;
    uint32_t result = ((state >> ((state >> 28) + 4u)) ^ state) * 277803737u;
    result = (result >> 22) ^ result;
    return __fmaf_rn(__uint2float_rn(result), 4.656612873077393e-10f /*2^-31*/, -1.0f);
}

// shaders.metal:163-172
struct Q4 { float x, y, z, w; };
__device__ __forceinline__ Q4 quat_dot(Q4 q1, Q4 q2) {
    V3 a = mk(q1.x, q1.y, q1.z), b = mk(q2.x, q2.y, q2.z);
    float s = fsub(fmul(q1.w, q2.w), dot3(a, b));
    V3 v = add3(add3(cross3(a, b), scale3(b, q1.w)), scale3(a, q2.w));
    Q4 r = {v.x, v.y, v.z, s};
    return r;
}
__device__ __forceinline__ V3 quat_mult(V3 vec, Q4 q) {
    Q4 inv = {-q.x, -q.y, -q.z, q.w};
    Q4 v4 = {vec.x, vec.y, vec.z, 0.0f};
    Q4 r = quat_dot(quat_dot(inv, v4), q);
    return mk(r.x, r.y, r.z);
}

struct Axis { float o, d, r, rl; };

// RCP (MM_FLAG_RCP_SLAB): the opt-in reciprocal-multiply slab arithmetic t = (b - o) * RN(1/d) — what a fast-math compile
// of the reference's divide amounts to; the oracle implements the same rule under the same flag.
template <bool FAST, bool RCP = false>
__device__ __forceinline__ float quot(float b, const Axis &a) {
    float x = fsub(b, a.o);
    if (RCP) return fmul(x, a.r);
    if (FAST) {
        float p = fmul(x, a.rl);
        float q1 = __fmaf_rn(x, a.r, p);
        float e = __fmaf_rn(-a.d, q1, x);
        return __fmaf_rn(e, a.r, q1);
    } else {
        return fdiv(x, a.d);
    }
}

__device__ __forceinline__ bool axis_safe(float o, float d) {
    float ad = fabsf(d), ao = fabsf(o);
    bool dok = ad >= 8.673617379884035e-19f /*2^-60*/ && ad <= 1.152921504606847e18f /*2^60*/;
    bool ook = ao == 0.0f || (ao >= 9.094947017729282e-13f /*2^-40*/ && ao <= 1073741824.0f /*2^30*/);
    return dok && ook;
}

// Reciprocal-multiply mode: the travel-ordered form needs finite operands and a finite non-zero reciprocal (no NaN from
// 0 * inf, monotone products); anything else takes the general min/max form.
__device__ __forceinline__ bool rcp_safe(float o, float d) {
    const float ad = fabsf(d);
    return ad >= 1.1754943508222875e-38f /*2^-126*/ && ad <= 8.507059173023462e37f /*2^126*/ && fabsf(o) <= 3.4028234663852886e38f;
}

struct Tally { uint32_t inner, leaf, rect, max_stack; };

constexpr uint32_t CUR_END = 0xFFFFFFFFu;   // traversal finished

// ---- packed FP32 (Blackwell FADD2 / FMUL2 / FFMA2: two IEEE-RN fp32 operations per issued instruction) ------------------
// The kernel is bound by instruction issue, not by the FMA pipe (ncu: issue slots 85 % busy, FMA pipe 43 %), and the
// twelve slab quotients of a visit are six pairs of identical, independent operation chains — so they are issued as
// add.rn.f32x2 / mul.rn.f32x2 / fma.rn.f32x2 on register pairs: per lane the results are the bits of the scalar
// instructions, at half the issue slots.
typedef unsigned long long f2;   // two fp32 in a 64-bit register pair (low word = first component)
__device__ __forceinline__ f2 pack2(float lo, float hi) {
    f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float lo2f(f2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); (void)b; return a; }
__device__ __forceinline__ float hi2f(f2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); (void)a; return b; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

// 8-byte shared-memory store / load at a 32-bit shared-window address (the y-table).  Through a generic pointer into dynamic
// shared memory, every access rebuilds the window base (S2UR SR_CgaCtaId, UMOV, UIADD3, ULEA).  Both are volatile, so they
// keep their program order: a visit's load of a table entry never moves above the fill's store of it.
__device__ __forceinline__ void sts64(uint32_t a, f2 v) { asm volatile("st.shared.b64 [%0], %1;" : : "r"(a), "l"(v)); }
__device__ __forceinline__ f2 lds64(uint32_t a) { f2 v; asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(a)); return v; }

// 32-byte read-only load (LDG.E.256, sm_100+): one instruction and one L1 request per half record.
struct Line32 { f2 x, y, z, w; };
__device__ __forceinline__ Line32 ldg256(const void *p) {
    Line32 q;
    asm("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(q.x), "=l"(q.y), "=l"(q.z), "=l"(q.w) : "l"(p));
    return q;
}

// Per-ray constants of the packed slab test: x and y share register pairs, z is duplicated.
struct RayK {
    f2 no_xy, nd_xy, r_xy, rl_xy;   // (-o.x, -o.y), (-d.x, -d.y), (r.x, r.y), (rl.x, rl.y)
    f2 no_zz, nd_zz, r_zz, rl_zz;
};

// Two slab quotients at once: x = b - o, then either the exact shared-reciprocal sequence (== RN(x/d), see the file header
// and docs/exact_quotient.md) or, in the opt-in MM_FLAG_RCP_SLAB arithmetic, x * RN(1/d).
template <bool RCP>
__device__ __forceinline__ f2 quot2(f2 b, f2 no, f2 nd, f2 r, f2 rl) {
    const f2 x = add2(b, no);                  // b + (-o) == b - o
    if (RCP) return mul2(x, r);
    const f2 p = mul2(x, rl);
    const f2 q1 = fma2(x, r, p);
    const f2 e = fma2(nd, q1, x);              // x - d*q1, exact
    return fma2(e, r, q1);
}

// The decisions of one interior visit (shaders.metal:140-154) from the children's [lo, hi] slab intervals.
// The literal `dist` values are never materialised: with hit_k = (hi_k >= lo_k && lo_k < t && hi_k > 0) and
// dist_k = hit_k ? lo_k : 1e30 (lo_k < t <= 1e30 when hit), `dist1 > dist2` is hit2 && (!hit1 || lo1 > lo2),
// `dist_near == 1e30` is !hit1 && !hit2 and `dist_far != 1e30` is hit1 && hit2 — the same decisions, fewer instructions.
template <bool CNT>
__device__ __forceinline__ void descend(float lo1, float hi1, float lo2, float hi2, const uint2 &lk, float t, uint32_t &cur, uint32_t *&sp,
                                        const uint32_t *stack, Tally &tl) {
    const bool hit1 = (hi1 >= lo1) & (lo1 < t) & (hi1 > 0.0f);          // :94
    const bool hit2 = (hi2 >= lo2) & (lo2 < t) & (hi2 > 0.0f);
    const bool swap = hit2 & (!hit1 | (lo1 > lo2));                     // :140, ties keep the left child first
    if (!(hit1 | hit2)) {                                               // :149-150
        cur = *--sp;                                                    // the bottom entry is the CUR_END sentinel
    } else {                                                            // :151-154
        cur = swap ? lk.y : lk.x;
        if (hit1 & hit2) {
            *sp++ = swap ? lk.x : lk.y;
            if (CNT) tl.max_stack = max(tl.max_stack, (uint32_t)(sp - stack) - 1u);   // entries above the sentinel
        }
    }
}

// One interior visit, fast form (guarded operand ranges: no zero / NaN / inf anywhere).  The quotients are the exact
// RN((b - o)/d) of the literal code; the record is loaded in the ray's travel order on every axis, so each axis' near
// plane is the first and its far plane the second value (rounding is monotone: min(t1,t2) is the near plane's quotient):
//   A = (c0.near.x, c0.near.y | c0.far.x, c0.far.y)   B likewise for child 1   Z = (c0.near.z, c1.near.z | c0.far.z, c1.far.z)
template <bool CNT, bool RCP>
__device__ __forceinline__ void inner_step_packed(const ulonglong2 &A, const ulonglong2 &B, const ulonglong2 &Z, const uint2 &lk,
                                                  const RayK &k, float t, uint32_t &cur, uint32_t *&sp, const uint32_t *stack, Tally &tl) {
    const f2 an = quot2<RCP>(A.x, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy), af = quot2<RCP>(A.y, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy);
    const f2 bn = quot2<RCP>(B.x, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy), bf = quot2<RCP>(B.y, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy);
    const f2 zn = quot2<RCP>(Z.x, k.no_zz, k.nd_zz, k.r_zz, k.rl_zz), zf = quot2<RCP>(Z.y, k.no_zz, k.nd_zz, k.r_zz, k.rl_zz);
    const float lo1 = fmaxf(fmaxf(lo2f(an), hi2f(an)), lo2f(zn));
    const float hi1 = fminf(fminf(lo2f(af), hi2f(af)), lo2f(zf));
    const float lo2 = fmaxf(fmaxf(lo2f(bn), hi2f(bn)), hi2f(zn));
    const float hi2 = fminf(fminf(lo2f(bf), hi2f(bf)), hi2f(zf));
    descend<CNT>(lo1, hi1, lo2, hi2, lk, t, cur, sp, stack, tl);
}

// One interior visit of the y-table traversal (PairRecY): the same quotients, with the two children's y pairs read from the
// per-lane table (y0 = child 0's (near.y, far.y), y1 = child 1's) instead of recomputed.  k holds x in both halves of its
// first four pairs.  XZ = (c0.near.x, c1.near.x | c0.far.x, c1.far.x | c0.near.z, c1.near.z | c0.far.z, c1.far.z).
template <bool CNT>
__device__ __forceinline__ void inner_step_ytab(const Line32 &XZ, f2 y0, f2 y1, const uint2 &lk, const RayK &k, float t, uint32_t &cur,
                                                uint32_t *&sp, const uint32_t *stack, Tally &tl) {
    const f2 xn = quot2<false>(XZ.x, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy), xf = quot2<false>(XZ.y, k.no_xy, k.nd_xy, k.r_xy, k.rl_xy);
    const f2 zn = quot2<false>(XZ.z, k.no_zz, k.nd_zz, k.r_zz, k.rl_zz), zf = quot2<false>(XZ.w, k.no_zz, k.nd_zz, k.r_zz, k.rl_zz);
    const float lo1 = fmaxf(fmaxf(lo2f(xn), lo2f(y0)), lo2f(zn));
    const float hi1 = fminf(fminf(lo2f(xf), hi2f(y0)), lo2f(zf));
    const float lo2 = fmaxf(fmaxf(hi2f(xn), lo2f(y1)), hi2f(zn));
    const float hi2 = fminf(fminf(hi2f(xf), hi2f(y1)), hi2f(zf));
    descend<CNT>(lo1, hi1, lo2, hi2, lk, t, cur, sp, stack, tl);
}

// One interior visit, general form: the literal min/max of shaders.metal:88-93 with NaN-dropping fmin/fmax, for rays whose
// operands are outside the guarded ranges (zero / subnormal / huge / NaN components) or under MM_FLAG_FORCE_LITERAL.
// Reads the record in its "up" order: a = (c0.min.x, c0.min.y, c0.max.x, c0.max.y), zu = (c0.min.z, c1.min.z, c0.max.z, c1.max.z).
template <bool CNT, bool RCP>
__device__ __forceinline__ void inner_step_general(const float4 &a, const float4 &b, const float4 &zu, const uint2 &lk, const Axis &ax,
                                                   const Axis &ay, const Axis &az, float t, uint32_t &cur, uint32_t *&sp,
                                                   const uint32_t *stack, Tally &tl) {
    float t1 = quot<false, RCP>(a.x, ax), t2 = quot<false, RCP>(a.z, ax);
    float lo1 = fminf(t1, t2), hi1 = fmaxf(t1, t2);
    t1 = quot<false, RCP>(a.y, ay); t2 = quot<false, RCP>(a.w, ay);
    lo1 = fmaxf(lo1, fminf(t1, t2)); hi1 = fminf(hi1, fmaxf(t1, t2));
    t1 = quot<false, RCP>(zu.x, az); t2 = quot<false, RCP>(zu.z, az);
    lo1 = fmaxf(lo1, fminf(t1, t2)); hi1 = fminf(hi1, fmaxf(t1, t2));
    t1 = quot<false, RCP>(b.x, ax); t2 = quot<false, RCP>(b.z, ax);
    float lo2 = fminf(t1, t2), hi2 = fmaxf(t1, t2);
    t1 = quot<false, RCP>(b.y, ay); t2 = quot<false, RCP>(b.w, ay);
    lo2 = fmaxf(lo2, fminf(t1, t2)); hi2 = fminf(hi2, fmaxf(t1, t2));
    t1 = quot<false, RCP>(zu.y, az); t2 = quot<false, RCP>(zu.w, az);
    lo2 = fmaxf(lo2, fminf(t1, t2)); hi2 = fminf(hi2, fmaxf(t1, t2));
    descend<CNT>(lo1, hi1, lo2, hi2, lk, t, cur, sp, stack, tl);
}

// One leaf visit (shaders.metal:127-129 with ray_rect_intersect :51-67 inlined), then pop / finish.
// LITERAL = false: the two edge tests `0 <= RN(x / L) <= L` are evaluated as the equivalent interval test on x stored in
// the record (render_kernel.cuh, RectI) — no divides by the edge lengths.  LITERAL = true (scenes with an edge length
// outside the guarded range, or MM_FLAG_FORCE_LITERAL): the literal divides, with the lengths recomputed by the same
// operations the upload used.
template <bool CNT, bool LITERAL>
__device__ __forceinline__ void leaf_step(const RectI *__restrict__ rects, V3 ori, V3 dir, float &t, uint32_t &slot, uint32_t &cur,
                                          uint32_t *&sp, Tally &tl) {
    const uint32_t first = cur & 0xFFFFFFu, count = (cur >> 24) & 0x7Fu;
#pragma unroll 1                               // leaves hold one rect almost always (leaf visits ~ rect tests): no unrolled copy, -1.3 %
    for (uint32_t i = 0; i < count; i++) {
        const float4 *rp = reinterpret_cast<const float4 *>(rects + first + i);
        const float4 r0 = __ldg(rp), r1 = __ldg(rp + 1), r2 = __ldg(rp + 2), r3 = __ldg(rp + 3);
        if (CNT) tl.rect++;
        const V3 ro = mk(r0.x, r0.y, r0.z), n = mk(r1.x, r1.y, r1.z), v = mk(r2.x, r2.y, r2.z), u = mk(r3.x, r3.y, r3.z);
        const float norm_check = dot3(dir, n);                                   // :53
        const float a = fdiv(dot3(sub3(ro, ori), n), norm_check);                // :55
        const V3 isect = add3(ori, scale3(dir, a));                              // :56
        const V3 rv = sub3(isect, ro);                                           // :58
        const float xv = dot3(rv, v), xu = dot3(rv, u);
        bool inside;
        if (LITERAL) {
            const float len_v = length3(v), len_u = length3(u);
            const float d1 = fdiv(xv, len_v);                                    // :60
            const float d2 = fdiv(xu, len_u);                                    // :61
            inside = (0.0f <= d1 && d1 <= len_v) && (0.0f <= d2 && d2 <= len_u);
        } else {
            inside = (r2.w <= xv) & (xv <= r0.w) & (r3.w <= xu) & (xu <= r1.w);
        }
        if (inside && norm_check != 0.0f && a > 0.1f && a < t) {                 // :63
            t = a;
            slot = first + i;
        }
    }
    cur = *--sp;
}

// One leaf visit for scenes whose rects are all axis-aligned (render_kernel.cuh, RectA): the literal test of
// shaders.metal:51-67 collapsed to one subtraction, one IEEE divide, two multiply-adds and interval tests on the intersection
// point's two in-plane coordinates — the same accept / reject decisions and the same beam.t, bit for bit (see RectA).
template <bool CNT>
__device__ __forceinline__ void leaf_step_axis(const RectA *__restrict__ rects, V3 ori, V3 dir, float &t, uint32_t &slot, uint32_t &cur,
                                               uint32_t *&sp, Tally &tl) {
    const uint32_t first = cur & 0xFFFFFFu, count = (cur >> 24) & 0x7Fu;
#pragma unroll 1
    for (uint32_t i = 0; i < count; i++) {
        const Line32 q = ldg256(rects + first + i);
        if (CNT) tl.rect++;
        const float c = lo2f(q.x), lo_a = hi2f(q.x), hi_a = lo2f(q.y), lo_b = hi2f(q.y), hi_b = lo2f(q.z);
        const uint32_t k = __float_as_uint(hi2f(q.z));
        const bool k0 = k == 0u, k2 = k == 2u;
        const float o_k = k0 ? ori.x : (k2 ? ori.z : ori.y), d_k = k0 ? dir.x : (k2 ? dir.z : dir.y);
        const float o_a = k0 ? ori.y : ori.x, d_a = k0 ? dir.y : dir.x;       // in-plane axes in increasing order
        const float o_b = k2 ? ori.y : ori.z, d_b = k2 ? dir.y : dir.z;
        const float a = fdiv(fsub(c, o_k), d_k);                                 // :53-55 with n = +-e_k
        const float pa = fadd(o_a, fmul(d_a, a)), pb = fadd(o_b, fmul(d_b, a));  // :56, the two in-plane coordinates
        const bool inside = (lo_a <= pa) & (pa <= hi_a) & (lo_b <= pb) & (pb <= hi_b);   // :58-63 as intervals on the point itself
        if (inside && d_k != 0.0f && a > 0.1f && a < t) {                        // :63
            t = a;
            slot = first + i;
        }
    }
    cur = *--sp;
}

// intersect_bvh_iterative (shaders.metal:115-156) for the rays of one warp.  Every lane of the warp calls this together
// (lanes without a ray pass alive = false) and the warp votes on which body to execute: the interior body runs (kInnerReps
// visits per vote) while the lanes standing at an interior node outweigh the lanes waiting at a leaf
// (nI >= kLeafWeight * nL), otherwise the waiting lanes test their rects.  Each lane still performs exactly the
// reference's sequence of visits for its own ray; only the interleaving between lanes changes.  (A plain while-while
// loop — all lanes descend to a leaf, then all test — left 12 of 32 lanes active in the interior body; see profiles/.)
// `lit` lanes (operands outside the guarded ranges, or MM_FLAG_FORCE_LITERAL) use the general slab form.
#ifndef MM_LEAF_WEIGHT
#define MM_LEAF_WEIGHT 8
#endif
constexpr uint32_t kLeafWeight = MM_LEAF_WEIGHT;   // measured best on B200 (r1: 6; 8 since the axis-aligned leaf test made the leaf body cheaper)
#ifndef MM_INNER_REPS
#define MM_INNER_REPS 4
#endif
constexpr uint32_t kInnerReps = MM_INNER_REPS;
constexpr int kRepUnroll = 2;                      // visits per loop trip: 2 measured best (1: +0.6 %, 4: +1.3 %)

// MIXED = false: no lane of the warp is literal (the common case; the loop then contains no general-form code).
// Not inlined on purpose: the call boundary parks the path state that the traversal does not touch (throughput,
// radiance, RNG state, counters, pixel bookkeeping) in the caller's frame, so the traversal loop has the whole 64-register
// budget for its per-ray constants.
struct Hit { float t; uint32_t slot; };
// AX = true: the scene's rects are all axis-aligned and `rects` points at RectA records (leaf_step_axis).
// YT = true (only with MIXED = false, RCP = false): `pairs` points at PairRecY records, and the ray's y quotients of the scene's
// n_yiv y-intervals y_ivals are first written to the lane's column of the y-table, at shared-window address `ytab` (entry i at
// ytab + i * kYEntryStride), with the same operations a visit of the other form performs on them.  The caller converts the
// column to that address once per thread (table_column): converted here, at every call, it would cost the y-table kernels a
// register across the call and a spill.
extern __shared__ __align__(16) unsigned char mm_dyn_smem[];
// The shared-window address of byte `offset` of the dynamic shared memory (the y-table column of a lane).
__device__ __forceinline__ uint32_t table_column(uint32_t offset) { return (uint32_t)__cvta_generic_to_shared(mm_dyn_smem) + offset; }
template <bool MIXED, bool CNT, bool RCP, bool AX = false, bool YT = false>
__device__ __noinline__ Hit traverse(const void *__restrict__ pairs, const void *__restrict__ rects, uint32_t root, bool alive,
                                     bool lit, V3 ori, V3 dir, float beam_t, uint32_t beam_slot, Tally *tlp,
                                     uint32_t ytab = 0u, const float4 *__restrict__ y_ivals = nullptr, uint32_t n_yiv = 0u) {
    static_assert(!YT || (!MIXED && !RCP), "the y-table traversal is the exact fast form only");
    Tally tl = {0u, 0u, 0u, 0u};
    uint32_t stack[MM_MAX_STACK];              // local memory (L1); BVH depth is validated against it at upload
    const float rx = __frcp_rn(dir.x), ry = __frcp_rn(dir.y), rz = __frcp_rn(dir.z);
    const float rlx = fmul(__fmaf_rn(-dir.x, rx, 1.0f), rx), rly = fmul(__fmaf_rn(-dir.y, ry, 1.0f), ry),
                rlz = fmul(__fmaf_rn(-dir.z, rz, 1.0f), rz);
    RayK k;
    if (YT) {
        const f2 no_yy = pack2(-ori.y, -ori.y), nd_yy = pack2(-dir.y, -dir.y), r_yy = pack2(ry, ry), rl_yy = pack2(rly, rly);
        const uint32_t sy = dir.y < 0.0f ? 8u : 0u;
        // A branch out, not a predicate per slot: the warp issues only the scene's n_yiv slots (5 for every maze).
#pragma unroll
        for (uint32_t i = 0; i < kMaxYIntervals; i++) {
            if (i >= n_yiv) break;
            const f2 b = __ldg(reinterpret_cast<const f2 *>(reinterpret_cast<const char *>(y_ivals + i) + sy));   // (near.y, far.y)
            sts64(ytab + i * kYEntryStride, quot2<false>(b, no_yy, nd_yy, r_yy, rl_yy));
        }
        k.no_xy = pack2(-ori.x, -ori.x); k.nd_xy = pack2(-dir.x, -dir.x); k.r_xy = pack2(rx, rx); k.rl_xy = pack2(rlx, rlx);
    } else {
        k.no_xy = pack2(-ori.x, -ori.y); k.nd_xy = pack2(-dir.x, -dir.y); k.r_xy = pack2(rx, ry); k.rl_xy = pack2(rlx, rly);
    }
    k.no_zz = pack2(-ori.z, -ori.z); k.nd_zz = pack2(-dir.z, -dir.z); k.r_zz = pack2(rz, rz); k.rl_zz = pack2(rlz, rlz);
    // per-ray record pointers with the travel order folded in: ab[sx + 2 sy] at +32 (sx + 2 sy), z|link[sz] at +128 + 32 sz;
    // YT: xz[sx + 2 sz] at +32 (sx + 2 sz), link at +128
    const char *base = reinterpret_cast<const char *>(pairs);
    const char *pAB = YT ? base + (dir.x < 0.0f ? 32 : 0) + (dir.z < 0.0f ? 64 : 0)
                         : base + (lit ? 0 : (dir.x < 0.0f ? 32 : 0) + (dir.y < 0.0f ? 64 : 0));
    const char *pZ = YT ? base + 128 : base + 128 + ((!lit && dir.z < 0.0f) ? 32 : 0);
    asm("" : "+l"(pAB)); asm("" : "+l"(pZ));      // keep them live: ptxas otherwise re-derives them from sign(dir) at every node
    // The pair table lies inside one 4-GB-aligned window (checked at upload), so a record address is {hi, lo + offset} with
    // no carry: one 32-bit add per pointer instead of a 64-bit add (two instructions).
    uint32_t ab_lo = (uint32_t)reinterpret_cast<uintptr_t>(pAB), z_lo = (uint32_t)reinterpret_cast<uintptr_t>(pZ);
    uint32_t hi_a = (uint32_t)(reinterpret_cast<uintptr_t>(pAB) >> 32), hi_z = (uint32_t)(reinterpret_cast<uintptr_t>(pZ) >> 32);   // two registers on purpose
    asm("" : "+r"(ab_lo)); asm("" : "+r"(z_lo)); asm("" : "+r"(hi_a)); asm("" : "+r"(hi_z));
    stack[0] = CUR_END;                        // sentinel: popping an empty stack ends the traversal, no emptiness test
    uint32_t *sp = stack + 1;                  // next free entry; a pointer, so push and pop need no address arithmetic
    uint32_t cur = alive ? root : CUR_END, slot = beam_slot;
    float t = beam_t;
    while (true) {
        const bool isI = (cur & kLeafBit) == 0u;
        const bool isL = !isI && cur != CUR_END;
        const unsigned mI = __ballot_sync(0xFFFFFFFFu, isI), mL = __ballot_sync(0xFFFFFFFFu, isL);
        if ((mI | mL) == 0u) break;
        if (mI != 0u && __popc(mI) >= kLeafWeight * __popc(mL)) {
#pragma unroll kRepUnroll
            for (uint32_t rep = 0; rep < kInnerReps; rep++) {
                if ((cur & kLeafBit) == 0u) {
                    const size_t off = cur;                      // interior descriptors are byte offsets
                    if (CNT) tl.inner++;
                    if (YT) {
                        uint64_t aXZ, aL;
                        asm("mov.b64 %0, {%1, %2};" : "=l"(aXZ) : "r"(ab_lo + cur), "r"(hi_a));
                        asm("mov.b64 %0, {%1, %2};" : "=l"(aL) : "r"(z_lo + cur), "r"(hi_z));
                        const Line32 xz = ldg256(reinterpret_cast<const void *>(aXZ));
                        const uint4 lk = __ldg(reinterpret_cast<const uint4 *>(aL));
                        const f2 y0 = lds64(ytab + lk.z), y1 = lds64(ytab + lk.w);
                        inner_step_ytab<CNT>(xz, y0, y1, make_uint2(lk.x, lk.y), k, t, cur, sp, stack, tl);
                    } else if (!MIXED || !lit) {
                        // 32-B load for (A, B): measured 1.5 % faster than two 16-B loads; folding (Z, link) into a second
                        // 32-B load gave nothing (profiles/r1_block_shape.txt)
                        uint64_t aAB, aZ;
                        asm("mov.b64 %0, {%1, %2};" : "=l"(aAB) : "r"(ab_lo + cur), "r"(hi_a));
                        asm("mov.b64 %0, {%1, %2};" : "=l"(aZ) : "r"(z_lo + cur), "r"(hi_z));
                        const Line32 ab = ldg256(reinterpret_cast<const void *>(aAB));
                        ulonglong2 A, B;
                        A.x = ab.x; A.y = ab.y; B.x = ab.z; B.y = ab.w;
                        const ulonglong2 Z = __ldg(reinterpret_cast<const ulonglong2 *>(aZ));
                        const uint2 lk = __ldg(reinterpret_cast<const uint2 *>(aZ + 16));
                        inner_step_packed<CNT, RCP>(A, B, Z, lk, k, t, cur, sp, stack, tl);
                    } else {
                        const uint2 lk = __ldg(reinterpret_cast<const uint2 *>(base + 144 + off));
                        const float4 a = __ldg(reinterpret_cast<const float4 *>(base + off)), b = __ldg(reinterpret_cast<const float4 *>(base + off + 16));
                        const float4 zu = __ldg(reinterpret_cast<const float4 *>(base + off + 128));
                        Axis ax, ay, az;
                        ax.o = ori.x; ax.d = dir.x; ax.r = rx; ax.rl = rlx;
                        ay.o = ori.y; ay.d = dir.y; ay.r = ry; ay.rl = rly;
                        az.o = ori.z; az.d = dir.z; az.r = rz; az.rl = rlz;
                        inner_step_general<CNT, RCP>(a, b, zu, lk, ax, ay, az, t, cur, sp, stack, tl);
                    }
                }
            }
        } else {
            if (isL) {
                if (CNT) tl.leaf++;
                if (AX) leaf_step_axis<CNT>(static_cast<const RectA *>(rects), ori, dir, t, slot, cur, sp, tl);
                else leaf_step<CNT, MIXED>(static_cast<const RectI *>(rects), ori, dir, t, slot, cur, sp, tl);
            }
        }
    }
    if (CNT) { tlp->inner += tl.inner; tlp->leaf += tl.leaf; tlp->rect += tl.rect; tlp->max_stack = max(tlp->max_stack, tl.max_stack); }
    Hit h;
    h.t = t; h.slot = slot;
    return h;
}

// noise.sample(s, float2(gid)): normalised coordinates, address::repeat, filter::nearest (shaders.metal:288,291).
__device__ __forceinline__ void sample_noise_xy(const uint8_t *noise, uint32_t nw, uint32_t nh, float u, float v, float &nx, float &ny) {
    float fu = fsub(u, floorf(u)), fv = fsub(v, floorf(v));
    int ix = (int)floorf(fmul(fu, (float)nw)), iy = (int)floorf(fmul(fv, (float)nh));
    ix = min(max(ix, 0), (int)nw - 1);
    iy = min(max(iy, 0), (int)nh - 1);
    const uint8_t *tx = noise + 4 * ((size_t)iy * nw + (size_t)ix);
    uchar4 c = *reinterpret_cast<const uchar4 *>(tx);
    nx = fdiv((float)c.x, 255.0f);
    ny = fdiv((float)c.y, 255.0f);
}


// ---- one path's start (shaders.metal:261-303): thread -> pixel mapping of the virtual dispatch, camera ray, seed, jitter ------
struct PathStart {
    V3 ori, dir;
    uint32_t state;            // RNG state after the two jitter draws
    uint32_t pxx, pxy;         // pixel
    uint32_t k, flat;          // group index within the launch, thread index within the group
};
// Thread s.flat of grid group g under camera cam at frame `time`, chunk list `chunks` (s.k and s.flat set by the caller).
__device__ __forceinline__ void start_at(const KParams &P, PathStart &s, uint32_t g, const mm_chunk *chunks, const mm_camera &cam, uint32_t time) {
    const uint32_t tgx = g % P.grid_x, tgy = g / P.grid_x;
    const mm_chunk ch = chunks[g];                                     // :266-267
    const uint32_t gx = s.flat % P.dim_x, gy = s.flat / P.dim_x;       // inverse of :271
    const uint32_t chunk = P.uni.chunk_width;
    const uint32_t pixel_number = s.flat >> P.log2_spp;                // :272
    s.pxx = ch.x + pixel_number / chunk;                               // :274-275
    s.pxy = ch.y + pixel_number % chunk;                               // :273,275
    const uint32_t texid_x = tgx * P.dim_x + gx, texid_y = tgy * P.dim_y + gy;

    const V3 center = mk(cam.camera_center.x, cam.camera_center.y, cam.camera_center.z);
    const float pnx = fdiv(__uint2float_rn(s.pxx), P.uni.view_width), pny = fdiv(__uint2float_rn(s.pxy), P.uni.view_height);   // :281
    const V3 corner = sub3(center, mk(fdiv(cam.viewport.x, 2.0f), fdiv(cam.viewport.y, 2.0f), -cam.focal_length));        // :282
    V3 ray_dir = normalize3(sub3(add3(corner, mk(fmul(pnx, cam.viewport.x), fmul(pny, cam.viewport.y), 0.0f)), center));  // :283
    const Q4 rot = {cam.rotation.x, cam.rotation.y, cam.rotation.z, cam.rotation.w};
    ray_dir = quat_mult(ray_dir, rot);                                 // :284

    float nx, ny;
    sample_noise_xy(P.noise, P.noise_w, P.noise_h, __uint2float_rn(gx), __uint2float_rn(gy), nx, ny);   // :291
    // :298 — float + uint promotes to float, products wrap in u32, left to right; float->uint saturates.
    const float seed_f = fadd(fadd(fadd(fadd(nx, ny), __uint2float_rn(texid_x * 15823u)), __uint2float_rn(texid_y * 9737333u)),
                              __uint2float_rn(time));
    uint32_t state = __float2uint_rz(seed_f);
    s.ori = center;                                                    // :302
    const float j1 = rnd_pm1(state), j2 = rnd_pm1(state);
    s.dir = add3(ray_dir, scale3(mk(j1, j2, 0.0f), 0.001f));           // :303
    s.state = state;
}
__device__ __forceinline__ PathStart start_path(const KParams &P, uint64_t path) {
    PathStart s;
    s.k = (uint32_t)(path / P.T);
    s.flat = (uint32_t)(path - (uint64_t)s.k * P.T);
    start_at(P, s, P.group_first + s.k * P.group_step, P.chunks, P.uni.cam, P.uni.time);
    return s;
}
// The same for a multi-view launch (mm_render_views): the launch's group k is group k mod group_count of view
// k / group_count, which starts exactly as that group of a single-view dispatch with the view's camera, time and chunks.
__device__ __forceinline__ PathStart start_view_path(const KParams &P, const ViewRec *views, uint64_t path) {
    PathStart s;
    s.k = (uint32_t)(path / P.T);
    s.flat = (uint32_t)(path - (uint64_t)s.k * P.T);
    const uint32_t v = s.k / P.group_count, kv = s.k - v * P.group_count;
    const ViewRec &V = views[v];
    const mm_camera cam = V.uni.cam;
    start_at(P, s, P.group_first + kv * P.group_step, P.chunks + V.chunk_off, cam, V.uni.time);
    return s;
}

// ---- one hit's shading (shaders.metal:308-335) after a traversal returned (t < 1e30, slot): updates the path state and sets up
// the next segment's ray.  Returns false when the path ends inside the mirror branch (:333).
__device__ __forceinline__ bool shade_hit(const KParams &P, uint32_t slot, float t, V3 &ori, V3 &dir, V3 &color, V3 &light, uint32_t &state,
                                          int &mirror_hits, uint32_t *orig_id) {
    const float4 *rp = reinterpret_cast<const float4 *>(P.rects + slot);
    const float4 r1 = __ldg(rp + 1);
    const V3 nrm = mk(r1.x, r1.y, r1.z);                   // :309 (per-rect constant, same operations)
    const float side = -sign1(dot3(dir, nrm));             // :310
    const float4 *sp4 = reinterpret_cast<const float4 *>(P.shade + slot);
    const float4 col = __ldg(sp4);                         // albedo, material bits in .w
    if (orig_id) *orig_id = __float_as_uint(__ldg(sp4 + 1).w);
    if (__float_as_uint(col.w) == 0u || side == -1.0f) {   // :311
        const float4 emi = __ldg(sp4 + 1);
        light = add3(light, mul3(mk(emi.x, emi.y, emi.z), color));   // :312-313
        color = mul3(color, mk(col.x, col.y, col.z));      // :314
        // :315-318 rejection loop `while (length(rd) > 1)`.  RN(sqrt(s)) > 1 <=> s > 1 + 2^-23: sqrt is
        // monotone, sqrt(1 + 2^-23) = 1 + 2^-24 - ... lies below the midpoint and rounds to 1, and
        // sqrt(1 + 2^-22) rounds above 1 (checked over every float in [0.5, 2) in tests/test_oracle.py),
        // so the loop compares the squared length and the square root is taken once, after it.
        V3 rd;
        float s2;
        do {
            const float a = rnd_pm1(state), b = rnd_pm1(state), c = rnd_pm1(state);
            rd = mk(a, b, c);
            s2 = dot3(rd, rd);
        } while (s2 > 1.00000011920928955f);
        const float rl = fsqrt(s2);                        // :319 normalize = v / length(v)
        rd = mk(fdiv(rd.x, rl), fdiv(rd.y, rl), fdiv(rd.z, rl));
        ori = add3(ori, scale3(dir, t));                   // :320
        dir = normalize3(add3(rd, scale3(nrm, side)));     // :321
        return true;
    }
    mirror_hits++;                                         // :325
    if (mirror_hits < P.mirror_limit) {                    // :326
        light = add3(light, scale3(mk(col.x, col.y, col.z), 0.005f));   // :327
        ori = add3(ori, scale3(dir, t));                   // :328
        dir = normalize3(reflect3(dir, nrm));              // :329
        return true;
    }
    return false;                                          // :333
}

// lit: this ray must use the general slab form (operands outside the guarded ranges of the shared-reciprocal quotient)
__device__ __forceinline__ bool ray_is_literal(const KParams &P, V3 ori, V3 dir) {
    return P.force_literal || !P.scene_fast_ok ||
           !(P.rcp_mode ? (rcp_safe(ori.x, dir.x) && rcp_safe(ori.y, dir.y) && rcp_safe(ori.z, dir.z))
                        : (axis_safe(ori.x, dir.x) && axis_safe(ori.y, dir.y) && axis_safe(ori.z, dir.z)));
}

// Store into an RGBA8Unorm texture and read back (main.rs:702-709): rte(clamp(v, 0, 1) * 255) / 255; NaN stores 0.
__device__ __forceinline__ uint32_t unorm8(float v) { return min(__float2uint_rn(fmul(fminf(fmaxf(v, 0.0f), 1.0f), 255.0f)), 255u); }
__device__ __forceinline__ float quant8(float v) { return fdiv(__uint2float_rn(unorm8(v)), 255.0f); }
__device__ __forceinline__ float4 quant8(float4 p) { return make_float4(quant8(p.x), quant8(p.y), quant8(p.z), quant8(p.w)); }

// Per-pixel reduction of spp tone-mapped samples in the reference's order (shaders.metal:343-364): pairs, quads, octets (the
// phases whose stride is < spp), then the octets serially.  v[i * stride] is sample i.
__device__ __forceinline__ float reduce_samples(const float *v, uint32_t spp, uint32_t stride) {
    if (spp >= 8) {
        float acc = 0.0f;
        for (uint32_t o = 0; o < spp; o += 8) {
            const float *w = v + o * stride;
            const float oct = fadd(fadd(fadd(w[0], w[stride]), fadd(w[2 * stride], w[3 * stride])),
                                   fadd(fadd(w[4 * stride], w[5 * stride]), fadd(w[6 * stride], w[7 * stride])));
            acc = o == 0 ? oct : fadd(acc, oct);
        }
        return acc;
    }
    if (spp == 4) return fadd(fadd(v[0], v[stride]), fadd(v[2 * stride], v[3 * stride]));
    if (spp == 2) return fadd(v[0], v[stride]);
    return v[0];
}

}  // namespace
}  // namespace mmk
