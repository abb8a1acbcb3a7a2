// scene_prep.cpp — turns the reference's buffers (rect[], bvh_node[], indices[], materials[], emissions[];
// reference src/shaders.metal:249-254) into the device layout of render_kernel.cuh.  Host code, compiled by g++
// with -ffp-contract=off: the per-rect constants are computed with exactly the operations ray_rect_intersect
// performs per call (shaders.metal:52,60-61: normalize(cross(v,u)), length(v), length(u)) and the shader performs
// per hit (:312 emissions.rgb * emissions.a), one IEEE rounding each, so the kernel sees the literal values.
#include <climits>
#include <cmath>
#include <cstring>
#include "scene_prep.h"

namespace mmk {

namespace {
inline float dot3(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
inline float as_float(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }
inline bool coord_ok(float b) {
    float a = std::fabs(b);
    return a == 0.0f || (a >= 9.765625e-4f /*2^-10*/ && a <= 1073741824.0f /*2^30*/);
}
}  // namespace

// The literal edge test computes d = RN(x / L) and accepts 0 <= d <= L (shaders.metal:60-63).  Both comparisons are
// monotone in x, so each is a threshold on x; the thresholds follow from round-to-nearest-even:
//   d <= L  <=>  x / L < m, or x / L == m and L's last mantissa bit is 0 (the tie goes to L), m = midpoint(L, next(L)).
//       T = m * L is exact in double (25 x 24 bits).  With th = RN_f32(T) and tl = T - th: a float x satisfies x < T iff
//       x <= th (tl > 0) or x < th (tl < 0); for tl == 0, x == T is the tie.  So `x <= up` with up = th when tl > 0 or
//       (tl == 0 and L even), else the float below th.
//   0 <= d  <=>  x >= 0, or x < 0 and the quotient rounds to -0: |x| / L <= 2^-150 (2^-150 is the tie between 0 and the
//       smallest denormal and goes to 0).  With x = -k * 2^-149 that is k <= L / 2, so lo = -floor(L / 2) * 2^-149.
// NaN x fails both forms, +-inf behaves the same in both.  L == +0 (a degenerate edge) never accepts in the literal form
// (x / 0 is +-inf or NaN): NaN bounds reproduce that.  Guarded range otherwise: 2^-20 <= L <= 2^23 (quotients near L are
// normal numbers, floor(L / 2) * 2^-149 is an exact denormal); anything else — denormal, huge, inf, NaN — reports false.
bool edge_thresholds(float L, float *lo, float *up) {
    const float nan = std::nanf("");
    *lo = nan; *up = nan;
    uint32_t bits;
    std::memcpy(&bits, &L, 4);
    if (bits == 0u) return true;                                  // +0: never accepts
    if (!(L >= 9.5367431640625e-07f /*2^-20*/ && L <= 8388608.0f /*2^23*/)) return false;
    const float next = std::nextafterf(L, INFINITY);
    const double m = ((double)L + (double)next) * 0.5;            // exact
    const double T = m * (double)L;                               // exact: 25 x 24 significant bits
    const float th = (float)T;                                    // round to nearest even
    const double tl = T - (double)th;                             // exact
    *up = (tl > 0.0 || (tl == 0.0 && (bits & 1u) == 0u)) ? th : std::nextafterf(th, -INFINITY);
    *lo = -(float)(std::floor((double)L * 0.5) * 1.401298464324817e-45 /*2^-149*/);
    return true;
}

namespace {
// floats in their total order as integers (finite values and infinities; NaN never gets here)
inline int64_t fkey(float f) {
    uint32_t b; std::memcpy(&b, &f, 4);
    return (b & 0x80000000u) ? -(int64_t)(b & 0x7FFFFFFFu) : (int64_t)b;      // -0 and +0 share key 0
}
inline float fkey_inv(int64_t k) {
    const uint32_t b = k >= 0 ? (uint32_t)k : ((uint32_t)(-k) | 0x80000000u);
    float f; std::memcpy(&f, &b, 4); return f;
}
// The edge test as the literal code evaluates it for an in-plane coordinate p of the intersection point:
// x = RN(RN(p - origin_j) * edge_j), accepted iff lo <= x <= up (the interval form of 0 <= RN(x / L) <= L, edge_thresholds).
inline bool edge_accepts(float p, float origin_j, float edge_j, float lo, float up) {
    const float rv = p - origin_j;
    const float x = rv * edge_j;
    return lo <= x && x <= up;
}
// Interval [lo_p, hi_p] of floats p with edge_accepts(p): the test is a monotone chain (p -> p - origin_j -> * edge_j) followed
// by an interval, so the accepted set is contiguous; its ends are found by bisection over the float order from one accepted
// point.  Returns false when no float is accepted.
bool edge_interval(float origin_j, float edge_j, float lo, float up, float *lo_p, float *hi_p) {
    if (!(lo <= up) || edge_j == 0.0f) return false;
    // a point inside: the middle of the edge, then its neighbourhood, then the ends
    const float cand[5] = {origin_j + 0.5f * edge_j, origin_j, origin_j + edge_j, origin_j + 0.25f * edge_j, origin_j + 0.75f * edge_j};
    float seed = 0.0f;
    bool found = false;
    for (float c : cand)
        if (edge_accepts(c, origin_j, edge_j, lo, up)) { seed = c; found = true; break; }
    if (!found) return false;
    const int64_t ks = fkey(seed);
    int64_t a = fkey(-3.4028234663852886e38f), b = ks;          // lowest accepted: first key in [a, ks] that accepts
    while (a < b) {
        const int64_t m = a + (b - a) / 2;
        if (edge_accepts(fkey_inv(m), origin_j, edge_j, lo, up)) b = m; else a = m + 1;
    }
    *lo_p = fkey_inv(a);
    a = ks; b = fkey(3.4028234663852886e38f);                   // highest accepted: last key in [ks, b] that accepts
    while (a < b) {
        const int64_t m = a + (b - a + 1) / 2;
        if (edge_accepts(fkey_inv(m), origin_j, edge_j, lo, up)) a = m; else b = m - 1;
    }
    *hi_p = fkey_inv(a);
    return true;
}
inline int single_axis(const mm_float3 &v) {       // index of the only non-zero component, or -1
    const float c[3] = {v.x, v.y, v.z};
    int k = -1;
    for (int i = 0; i < 3; i++)
        if (c[i] != 0.0f) { if (k >= 0) return -1; k = i; }
    return k;
}
}  // namespace

bool axis_rect(const mm_plane &m, RectA *out) {
    RectA r;
    std::memset(&r, 0, sizeof(r));
    const float nan = std::nanf("");
    const float v[3] = {m.v.x, m.v.y, m.v.z}, u[3] = {m.u.x, m.u.y, m.u.z}, o[3] = {m.origin.x, m.origin.y, m.origin.z};
    for (int i = 0; i < 3; i++)
        if (!std::isfinite(v[i]) || !std::isfinite(u[i]) || !std::isfinite(o[i])) return false;
    const int jv = single_axis(m.v), ju = single_axis(m.u);
    const bool v_zero = v[0] == 0.0f && v[1] == 0.0f && v[2] == 0.0f, u_zero = u[0] == 0.0f && u[1] == 0.0f && u[2] == 0.0f;
    if (v_zero || u_zero) {                         // zero-length edge: cross = 0, normal = NaN, the literal test never accepts
        r.c = nan; r.lo_a = r.lo_b = nan; r.hi_a = r.hi_b = nan; r.k = 3u;
        *out = r;
        return true;
    }
    if (jv < 0 || ju < 0 || jv == ju) return false;
    const int k = 3 - jv - ju;                      // normal axis
    // the normal must come out as exactly +-e_k: normalize(cross(v, u)) with the operations of the upload / the shader
    const float c3[3] = {v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]};
    const float lc = std::sqrt(dot3(c3, c3));
    const float n[3] = {c3[0] / lc, c3[1] / lc, c3[2] / lc};
    for (int i = 0; i < 3; i++)
        if (!(i == k ? (n[i] == 1.0f || n[i] == -1.0f) : n[i] == 0.0f)) return false;
    const float lv = std::sqrt(dot3(v, v)), lu = std::sqrt(dot3(u, u));
    float lo_v, up_v, lo_u, up_u;
    if (!edge_thresholds(lv, &lo_v, &up_v) || !edge_thresholds(lu, &lo_u, &up_u)) return false;
    const int a = k == 0 ? 1 : 0, b = k == 2 ? 1 : 2;           // in-plane axes in increasing order
    float lo[3], hi[3];
    const bool okv = edge_interval(o[jv], v[jv], lo_v, up_v, &lo[jv], &hi[jv]);
    const bool oku = edge_interval(o[ju], u[ju], lo_u, up_u, &lo[ju], &hi[ju]);
    r.c = o[k]; r.k = (uint32_t)k;
    if (!okv || !oku) { r.c = nan; r.lo_a = r.lo_b = nan; r.hi_a = r.hi_b = nan; r.k = 3u; *out = r; return true; }   // nothing ever accepted
    r.lo_a = lo[a]; r.hi_a = hi[a]; r.lo_b = lo[b]; r.hi_b = hi[b];
    *out = r;
    return true;
}

int prepare_scene(const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes,
                  const uint32_t *indices, const uint8_t *materials, const mm_float4 *emissions, Prepared &out,
                  std::string &err) {
    uint32_t depth = 0, max_leaf = 0;
    std::vector<uint8_t> reachable;   // nodes the traversal can reach; a caller may pass a capacity-sized array with a garbage tail
    if (!mmh::bvh_stats(nodes, n_nodes, n_planes, &depth, &max_leaf, &reachable)) {
        err = "malformed BVH: child or leaf range out of bounds, shared child or cycle";
        return MM_ERR_BVH;
    }
    if (depth > MM_MAX_BVH_DEPTH) {   // stack occupancy <= depth - 1 <= 50 (the reference's stack), plus the kernel's bottom sentinel
        err = "BVH depth " + std::to_string(depth) + " exceeds MM_MAX_BVH_DEPTH";
        return MM_ERR_BVH;
    }
    if (max_leaf > kMaxLeafCount || n_planes >= (1u << 24) || n_nodes >= (1u << 24)) {
        err = "scene exceeds packed-descriptor limits (leaf > 126 planes or >= 2^24 planes/nodes)";
        return MM_ERR_UNSUPPORTED;
    }
    for (uint32_t i = 0; i < n_planes; i++)
        if (indices[i] >= n_planes) { err = "index out of range"; return MM_ERR_BVH; }

    // pair ids: reachable interior nodes in node-index order (the root, node 0, gets pair 0); unreachable entries are never read
    std::vector<uint32_t> pair_id(n_nodes, 0xFFFFFFFFu);
    uint32_t n_pairs = 0;
    for (uint32_t i = 0; i < n_nodes; i++)
        if (reachable[i] && nodes[i].tri_count == 0) pair_id[i] = n_pairs++;
    auto desc = [&](uint32_t c) -> uint32_t {
        const mm_bvh_node &nd = nodes[c];
        return nd.tri_count > 0 ? (kLeafBit | nd.left_first | (nd.tri_count << 24)) : pair_id[c] * (uint32_t)sizeof(PairRec);
    };
    out.pairs.assign(n_pairs ? n_pairs : 1, PairRec());
    std::memset(out.pairs.data(), 0, out.pairs.size() * sizeof(PairRec));
    bool fast_ok = true;
    for (uint32_t i = 0; i < n_nodes; i++) {
        if (!reachable[i] || nodes[i].tri_count != 0) continue;
        const mm_bvh_node &a = nodes[nodes[i].left_first], &b = nodes[nodes[i].left_first + 1];
        PairRec &p = out.pairs[pair_id[i]];
        for (int sy = 0; sy < 2; sy++)
            for (int sx = 0; sx < 2; sx++) {
                const mm_bvh_node *ch[2] = {&a, &b};
                for (int k = 0; k < 2; k++) {
                    const mm_float3 &mn = ch[k]->aabb_min, &mx = ch[k]->aabb_max;
                    p.ab[sx + 2 * sy][k] = make_float4(sx ? mx.x : mn.x, sy ? mx.y : mn.y, sx ? mn.x : mx.x, sy ? mn.y : mx.y);
                }
            }
        p.zl[0].z = make_float4(a.aabb_min.z, b.aabb_min.z, a.aabb_max.z, b.aabb_max.z);
        p.zl[1].z = make_float4(a.aabb_max.z, b.aabb_max.z, a.aabb_min.z, b.aabb_min.z);
        p.zl[0].link = p.zl[1].link = make_uint4(desc(nodes[i].left_first), desc(nodes[i].left_first + 1), 0u, 0u);
        const float c[12] = {a.aabb_min.x, a.aabb_min.y, a.aabb_min.z, a.aabb_max.x, a.aabb_max.y, a.aabb_max.z,
                             b.aabb_min.x, b.aabb_min.y, b.aabb_min.z, b.aabb_max.x, b.aabb_max.y, b.aabb_max.z};
        for (int k = 0; k < 12; k++) fast_ok = fast_ok && coord_ok(c[k]);
        // the travel-ordered fast path also needs min <= max on every axis (true for every box the builder emits)
        for (int k = 0; k < 3; k++) fast_ok = fast_ok && c[k] <= c[k + 3] && c[k + 6] <= c[k + 9];
    }
    out.n_pairs = n_pairs;
    // y-table records (render_kernel.cuh, PairRecY): only for the exact fast form, and only while the children's distinct
    // (min.y, max.y) intervals fit the table.  Intervals are told apart by their bits, so an entry's operands are exactly the
    // bounds a PairRec of the same child holds.  A scene whose root is a leaf has no interior visit and keeps PairRec only.
    if (fast_ok) {
        out.pairs_y.assign(n_pairs ? n_pairs : 1, PairRecY());
        std::memset(out.pairs_y.data(), 0, out.pairs_y.size() * sizeof(PairRecY));
        auto y_index = [&](const mm_bvh_node &c) -> uint32_t {
            const float4 iv = make_float4(c.aabb_min.y, c.aabb_max.y, c.aabb_max.y, c.aabb_min.y);
            for (uint32_t j = 0; j < out.y_ivals.size(); j++)
                if (std::memcmp(&out.y_ivals[j], &iv, sizeof(iv)) == 0) return j;
            out.y_ivals.push_back(iv);
            return (uint32_t)out.y_ivals.size() - 1u;
        };
        auto desc_y = [&](uint32_t c) -> uint32_t {
            const mm_bvh_node &nd = nodes[c];
            return nd.tri_count > 0 ? (kLeafBit | nd.left_first | (nd.tri_count << 24)) : pair_id[c] * (uint32_t)sizeof(PairRecY);
        };
        for (uint32_t i = 0; i < n_nodes && out.y_ivals.size() <= kMaxYIntervals; i++) {
            if (!reachable[i] || nodes[i].tri_count != 0) continue;
            const mm_bvh_node &a = nodes[nodes[i].left_first], &b = nodes[nodes[i].left_first + 1];
            PairRecY &p = out.pairs_y[pair_id[i]];
            for (int sz = 0; sz < 2; sz++)
                for (int sx = 0; sx < 2; sx++) {
                    p.xz[sx + 2 * sz][0] = make_float4(sx ? a.aabb_max.x : a.aabb_min.x, sx ? b.aabb_max.x : b.aabb_min.x,
                                                       sx ? a.aabb_min.x : a.aabb_max.x, sx ? b.aabb_min.x : b.aabb_max.x);
                    p.xz[sx + 2 * sz][1] = make_float4(sz ? a.aabb_max.z : a.aabb_min.z, sz ? b.aabb_max.z : b.aabb_min.z,
                                                       sz ? a.aabb_min.z : a.aabb_max.z, sz ? b.aabb_min.z : b.aabb_max.z);
                }
            const uint32_t ya = y_index(a), yb = y_index(b);
            p.link = make_uint4(desc_y(nodes[i].left_first), desc_y(nodes[i].left_first + 1), ya * kYEntryStride, yb * kYEntryStride);
        }
        if (out.y_ivals.empty() || out.y_ivals.size() > kMaxYIntervals) { out.pairs_y.clear(); out.y_ivals.clear(); }
    }
    out.root_link = nodes[0].tri_count > 0 ? nodes[0].left_first : 0u;
    out.root_count = nodes[0].tri_count;
    out.depth = depth;
    out.max_leaf = max_leaf;
    out.fast_ok = fast_ok;

    out.rects.resize(n_planes);
    bool rect_fast_ok = true;
    out.shade.resize(n_planes);
    for (uint32_t s = 0; s < n_planes; s++) {
        const uint32_t id = indices[s];
        const mm_plane &m = planes[id];
        const float v[3] = {m.v.x, m.v.y, m.v.z}, u[3] = {m.u.x, m.u.y, m.u.z};
        const float c[3] = {v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]};   // cross(v,u)
        const float lc = std::sqrt(dot3(c, c));
        const float n[3] = {c[0] / lc, c[1] / lc, c[2] / lc};                                                   // normalize
        const float lv = std::sqrt(dot3(v, v)), lu = std::sqrt(dot3(u, u));
        RectI &r = out.rects[s];
        float lo_v, up_v, lo_u, up_u;
        rect_fast_ok = edge_thresholds(lv, &lo_v, &up_v) && rect_fast_ok;
        rect_fast_ok = edge_thresholds(lu, &lo_u, &up_u) && rect_fast_ok;
        r.o_upv = make_float4(m.origin.x, m.origin.y, m.origin.z, up_v);
        r.n_upu = make_float4(n[0], n[1], n[2], up_u);
        r.v_lov = make_float4(v[0], v[1], v[2], lo_v);
        r.u_lou = make_float4(u[0], u[1], u[2], lo_u);
        const mm_float4 &e = emissions[id];
        RectS &sh = out.shade[s];
        sh.color = make_float4(m.color.x, m.color.y, m.color.z, as_float(materials[id] ? 1u : 0u));
        sh.emitted = make_float4(e.x * e.w, e.y * e.w, e.z * e.w, as_float(id));
    }
    out.rect_fast_ok = rect_fast_ok;
    // axis-aligned form (every rect of a maze scene): used by the kernel's leaf test when ALL rects have it
    out.rects_axis.resize(n_planes);
    bool axis_ok = rect_fast_ok;
    for (uint32_t s = 0; s < n_planes && axis_ok; s++) axis_ok = axis_rect(planes[indices[s]], &out.rects_axis[s]);
    if (!axis_ok) out.rects_axis.clear();
    out.axis_ok = axis_ok;
    return MM_OK;
}

}  // namespace mmk
