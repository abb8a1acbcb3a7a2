"""The BVH traversal ray by ray (mm_trace_rays, probe_rays_kernel) against the oracle's intersect_bvh_iterative (mmo_trace_rays),
for rays chosen to sit on the edges that frames never reach.

Frames only produce unit directions, and in a maze every bounce direction component is 0 or at least about 2^-25.  So the
guards that pick the exact shared-reciprocal slab form (axis_safe, rcp_safe), the ties of the interior visit and the warp's
choice of traversal form are never approached by a frame.  Here every ray's t, plane index and traversal counts must equal the
oracle's bit for bit, every ray's `lit` bit must equal a CPU restatement of the guards, and every warp's form must equal a CPU
restatement of the selection in warp_traverse (render_kernel.cu).  The ray sets, each seeded and built here:

- guard edges: one direction component at +-0, the smallest and largest subnormal, 2^-126, 2^-60 and 2^60 with both float
  neighbours, 2^126, FLT_MAX, +-inf and NaN; or one origin component at +-0, 2^-40 and 2^30 with both neighbours, +-inf and
  NaN, aimed at a point inside the scene;
- bulk: direction components with exponents uniform in [-64, 64] (not normalised), origins inside the scene, on box faces and
  at rect corners;
- ties: power-of-two directions from points on child box faces (x = +-0, hi = +-0), through box corners shared by siblings
  (lo1 == lo2), grazing corners (hi == lo), and with a starting t equal to a box's near quotient or a rect's distance;
- midpoints: (b - o) / d within a few 2^-48 (relative) of a rounding midpoint for a real child plane b, in all eight travel
  octants and on every axis, the y-table's included;
- warps: all-fast warps, one literal lane at each of the 32 positions, that lane dead, all lanes dead and a partial last warp.

Each set runs under 0, NO_Y_TABLE, GENERAL_RECTS, GENERAL_RECTS | NO_Y_TABLE, RCP_SLAB and FORCE_LITERAL, on mazes 10, 32 and
256, shelf scenes with 8 and 9 child y-intervals, a tilted cloud, a wide-leaf BVH, a scene with fast_slab_ok = 0 and the
maze scaled by 2^-3 and 2^20 and the far cloud at 2^22.  The CPU tests check the oracle entry against oracle/np_oracle.py on
every set, the rule restatements at their edges, the midpoint construction and the probe kernel's instruction mix."""
import functools
import os

import numpy as np
import pytest

from test_general_scenes import build_scene as general_scene
from test_general_scenes import classify
from test_y_table import scene_with_intervals

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
NONE = 0xFFFFFFFF
FORCE_LITERAL, RCP_SLAB, GENERAL_RECTS, NO_Y_TABLE = 2, 64, 2048, 8192          # include/mirror_maze_cuda.h
MIXED, RCP, AXIS, YTAB = 1, 2, 4, 8                                             # mm_trace_rays form bits
FLAGS = {"default": 0, "no_ytab": NO_Y_TABLE, "general": GENERAL_RECTS, "general_no_ytab": GENERAL_RECTS | NO_Y_TABLE,
         "rcp": RCP_SLAB, "literal": FORCE_LITERAL}
SCENES = ["maze10", "maze32", "maze256", "shelves8", "shelves9", "tilted_0", "wide_tilted_two_levels", "tiny_coord",
          "scaled_eighth", "scaled_2p20", "far_0"]
BULK_SCENES = ["maze32", "maze256", "shelves9", "tilted_0", "wide_tilted_two_levels", "scaled_2p20", "far_0"]
BULK_N = 1 << 20


def f32(x):
    return F32(x)


def up(x):
    return np.nextafter(F32(x), F32(np.inf))


def down(x):
    return np.nextafter(F32(x), F32(-np.inf))


FLT_MAX = np.finfo(F32).max
D_EDGES = [F32(0.0), F32(-0.0), F32(2.0 ** -149), F32(2.0 ** -126 - 2.0 ** -149), F32(2.0 ** -126), down(2.0 ** -60),
           f32(2.0 ** -60), up(2.0 ** -60), down(2.0 ** 60), f32(2.0 ** 60), up(2.0 ** 60), f32(2.0 ** 126), FLT_MAX,
           F32(np.inf), F32(-np.inf), F32(np.nan)]
O_EDGES = [F32(0.0), F32(-0.0), down(2.0 ** -40), f32(2.0 ** -40), up(2.0 ** -40), down(2.0 ** 30), f32(2.0 ** 30),
           up(2.0 ** 30), F32(np.inf), F32(-np.inf), F32(np.nan)]


# ---- scenes -----------------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _scene(name):
    import mirror_maze_b200 as mm

    if name.startswith("maze"):
        return mm.MazeScene(int(name[4:]), 0)
    if name.startswith("shelves"):
        return scene_with_intervals(mm, lambda n: mm.MazeScene(n, 0), int(name[7:]))
    return general_scene(mm, name)


def scene(mm, name):
    mm.load_library()
    return _scene(name)


@functools.lru_cache(maxsize=None)
def _classification(name):
    return classify(_scene(name))


# ---- CPU restatement of the rules ---------------------------------------------------------------------------------------------

def axis_safe(o, d):
    """trace_device.cuh axis_safe: 2^-60 <= |d| <= 2^60, and o = 0 or 2^-40 <= |o| <= 2^30 (NaN fails)."""
    ad, ao = np.abs(d), np.abs(o)
    return (ad >= F32(2.0 ** -60)) & (ad <= F32(2.0 ** 60)) & ((ao == 0) | ((ao >= F32(2.0 ** -40)) & (ao <= F32(2.0 ** 30))))


def rcp_safe(o, d):
    """rcp_safe: 2^-126 <= |d| <= 2^126 and |o| finite."""
    ad = np.abs(d)
    return (ad >= F32(2.0 ** -126)) & (ad <= F32(2.0 ** 126)) & (np.abs(o) <= FLT_MAX)


def lit(rays, flags, cls):
    """A ray takes the literal-divide slab form under FORCE_LITERAL, in a scene without fast_slab_ok, or when a component
    fails the guard of its arithmetic (rcp_safe under RCP_SLAB, axis_safe otherwise)."""
    o, d = rays[:, 0:3], rays[:, 3:6]
    with np.errstate(invalid="ignore"):
        safe = (rcp_safe(o, d) if flags & RCP_SLAB else axis_safe(o, d)).all(axis=1)
    return bool(flags & FORCE_LITERAL) | (not cls["slab"]) | ~safe


def warp_form(rays, lit_bits, flags, cls):
    """The traversal each ray's warp runs (32 rays to a warp): the mixed form when a live lane is literal or the scene lacks
    the divide-free rect test, else the y-table form where the scene has the table and the flags allow it, the
    reciprocal-multiply form under RCP_SLAB, or the plain packed form; with the axis-aligned rect test where the scene has it
    (never under RCP_SLAB, GENERAL_RECTS or FORCE_LITERAL)."""
    n = len(rays)
    w = (n + 31) // 32
    live_lit = np.zeros(w * 32, bool)
    live_lit[:n] = (rays[:, 7] != 0) & lit_bits
    rect_fast = cls["rect"] and not flags & FORCE_LITERAL
    rcp = bool(flags & RCP_SLAB)
    any_lit = live_lit.reshape(w, 32).any(axis=1) | (not rect_fast)
    axis = rect_fast and cls["axis"] and not flags & GENERAL_RECTS and not rcp
    ytab = cls["y_table"] > 0 and not flags & (FORCE_LITERAL | RCP_SLAB | NO_Y_TABLE)
    form = np.where(any_lit, MIXED, 0) | (RCP if rcp else 0) | np.where(~any_lit & axis, AXIS, 0) | np.where(~any_lit & ytab, YTAB, 0)
    return np.repeat(form.astype(np.uint32), 32)[:n]


# ---- ray sets ---------------------------------------------------------------------------------------------------------------

def _rays(o, d, t=None, alive=None):
    n = len(o)
    r = np.empty((n, 8), F32)
    r[:, 0:3], r[:, 3:6] = o, d
    r[:, 6] = F32(1e30) if t is None else t
    r[:, 7] = 1.0 if alive is None else alive
    return r


def _bounds(sc):
    return sc.nodes[0]["aabb_min"].astype(F32), sc.nodes[0]["aabb_max"].astype(F32)


def _inside(rng, sc, n):
    lo, hi = _bounds(sc)
    return (lo + (hi - lo) * rng.random((n, 3))).astype(F32)


def _unit(rng, n):
    d = rng.normal(size=(n, 3))
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F32)


def _children(sc):
    """Indices of the nodes that are some interior node's child (the boxes the traversal slab-tests)."""
    nd = sc.nodes
    inner = np.nonzero(nd["tri_count"] == 0)[0]
    if len(inner) == 0:
        return np.zeros(0, np.int64)
    lf = nd["left_first"][inner].astype(np.int64)
    return np.unique(np.concatenate([lf, lf + 1]))


def _face_points(rng, sc, n):
    ch = _children(sc)
    if len(ch) == 0:
        return _inside(rng, sc, n)
    pick = ch[rng.integers(len(ch), size=n)]
    mn, mx = sc.nodes["aabb_min"][pick].astype(F32), sc.nodes["aabb_max"][pick].astype(F32)
    p = (mn + (mx - mn) * rng.random((n, 3))).astype(F32)
    k = rng.integers(3, size=n)
    side = rng.random(n) < 0.5
    p[np.arange(n), k] = np.where(side, mn[np.arange(n), k], mx[np.arange(n), k])
    return p


def _rect_corners(rng, sc, n):
    pl = sc.planes[rng.integers(len(sc.planes), size=n)]
    o, v, u = pl["origin"].astype(F32), pl["v"].astype(F32), pl["u"].astype(F32)
    a, b = rng.integers(2, size=(n, 1)).astype(F32), rng.integers(2, size=(n, 1)).astype(F32)
    return (o + a * v + b * u).astype(F32)


def guard_edge_rays(sc, rng, per=48):
    """One direction component at each D_EDGES value (random sign), or one origin component at each O_EDGES value (random sign)
    with the direction aimed at a point inside the scene; the other components ordinary."""
    out = []
    for k in range(3):
        for v in D_EDGES:
            o, d = _inside(rng, sc, per), _unit(rng, per)
            d[:, k] = v * np.where(rng.random(per) < 0.5, F32(-1), F32(1))
            out.append(_rays(o, d))
        for v in O_EDGES:
            target, o = _inside(rng, sc, per), _inside(rng, sc, per)
            o[:, k] = v * np.where(rng.random(per) < 0.5, F32(-1), F32(1))
            with np.errstate(invalid="ignore"):
                d = (target - o).astype(F32)
            bad = ~np.isfinite(d).all(axis=1)
            d[bad] = _unit(rng, int(bad.sum()))
            out.append(_rays(o, d))
    return np.concatenate(out)


def bulk_rays(sc, rng, n):
    """Direction components with exponents uniform in [-64, 64], random mantissas and signs (not normalised); origins inside the
    scene's bounds, on child box faces and at rect corners in equal parts."""
    e = rng.integers(-64, 65, size=(n, 3))
    m = rng.integers(0, 1 << 23, size=(n, 3))
    bits = (rng.integers(2, size=(n, 3)).astype(np.uint32) << 31) | ((e + 127).astype(np.uint32) << 23) | m.astype(np.uint32)
    d = bits.view(F32)
    third = n // 3
    o = np.concatenate([_inside(rng, sc, third), _face_points(rng, sc, third), _rect_corners(rng, sc, n - 2 * third)])
    return _rays(o, d)


def _pow2_dirs(rng, n):
    return (np.exp2(rng.integers(-3, 4, size=(n, 3))) * np.where(rng.random((n, 3)) < 0.5, -1.0, 1.0)).astype(F32)


def tie_rays(sc, rng, per=1024):
    """Exact ties from the scene's own boxes, power-of-two directions (exact quotients): origins on child box faces (x = +-0,
    and hi = +-0 on a far face moving away); rays through box corners, which siblings often share (lo1 == lo2) and which grazing
    rays only touch (hi == lo), a third of them starting at t = the corner's quotient (lo == t); and rays whose starting t and
    slot are a rect's own distance and slot (a == t).  Returns (rays, slots)."""
    ch = _children(sc)
    face = _rays(_face_points(rng, sc, per), _pow2_dirs(rng, per))
    if len(ch):
        pick = ch[rng.integers(len(ch), size=per)]
        mn, mx = sc.nodes["aabb_min"][pick].astype(F32), sc.nodes["aabb_max"][pick].astype(F32)
        corner = np.where(rng.random((per, 3)) < 0.5, mn, mx).astype(F32)
    else:
        corner = _rect_corners(rng, sc, per)
    d = _pow2_dirs(rng, per)
    t0 = np.exp2(rng.integers(-2, 5, size=per)).astype(F32)
    o = (corner - d * t0[:, None]).astype(F32)
    t = np.where(rng.random(per) < 1 / 3, t0, F32(1e30)).astype(F32)
    through = _rays(o, d, t)
    # a rect's own distance as the starting t: p = origin + v/2 + u/4 on the rect, the ray reaches p at t0
    pid = rng.integers(len(sc.planes), size=per)
    pl = sc.planes[pid]
    p = (pl["origin"] + F32(0.5) * pl["v"] + F32(0.25) * pl["u"]).astype(F32)
    d = _pow2_dirs(rng, per)
    t0 = np.exp2(rng.integers(-1, 4, size=per)).astype(F32)
    rect = _rays((p - d * t0[:, None]).astype(F32), d, t0)
    slot_of = np.empty(len(sc.indices), np.uint32)
    slot_of[sc.indices] = np.arange(len(sc.indices), dtype=np.uint32)
    slots = np.concatenate([np.full(2 * per, NONE, np.uint32), slot_of[pid]])
    return np.concatenate([face, through, rect]), slots


def midpoint_operands(rng, b, sign_d):
    """(o, d, x) with x = RN(b - o) exact and x / d within 6 * 2^-48 (relative) of a rounding midpoint, d of sign sign_d.
    x = X 2^ex and |d| = D 2^ed with M D = X 2^K + r for an odd 25-bit M and r in {-3, -1, 1, 3}: M = r D^-1 mod 2^K, so
    x / d = (M - r / D) 2^(ex - ed - K), at r / (M D) <= 3 * 2^-47 from the midpoint M 2^(ex - ed - K)."""
    while True:
        D = int(rng.integers(1 << 23, 1 << 24)) | 1
        r = int(rng.choice([-3, -1, 1, 3]))
        for K in (24, 25, 26):
            M = (r * pow(D, -1, 1 << K)) % (1 << K)
            if not ((1 << 24) <= M < (1 << 25)):
                continue
            X, rem = divmod(M * D - r, 1 << K)
            if rem == 0 and (1 << 23) <= X < (1 << 24):
                break
        else:
            continue
        if b != 0:                                    # x in b's binade and of its sign: b - x is exact
            ex = int(np.floor(np.log2(abs(float(b))))) - 23
            x = F32(np.copysign(X * 2.0 ** ex, float(b)))
            o = F32(b) - x
        else:
            x = F32(X * 2.0 ** int(rng.integers(-25, -19)) * (1 if rng.random() < 0.5 else -1))
            o = -x
        d = F32(sign_d * D * 2.0 ** int(rng.integers(-25, -21)))
        return o, d, x


def midpoint_rays(sc, rng, per=48):
    """For every axis and each of the eight travel octants: a real child plane b of the scene, an origin and a direction whose
    quotient (b - o) / d on that axis lies within a few 2^-48 of a rounding midpoint.  The other components are ordinary."""
    ch = _children(sc)
    if len(ch) == 0:
        ch = np.array([0])
    out = []
    for k in range(3):
        for octant in range(8):
            signs = np.array([1.0 if (octant >> j) & 1 == 0 else -1.0 for j in range(3)], F32)
            o, d = _inside(rng, sc, per), (np.abs(_unit(rng, per)) + F32(0.05)) * signs
            for i in range(per):
                node = ch[rng.integers(len(ch))]
                b = F32(sc.nodes[node]["aabb_min" if rng.random() < 0.5 else "aabb_max"][k])
                o[i, k], d[i, k], _ = midpoint_operands(rng, b, float(signs[k]))
            out.append(_rays(o, d.astype(F32)))
    return np.concatenate(out)


def warp_rays(sc, rng):
    """All-fast warps; warp j with one literal lane (d.x = 0) at position j; the same with that lane dead; two dead warps;
    a partial last warp of 13 lanes with one literal lane."""
    def ordinary(n):
        return _rays(_inside(rng, sc, n), _unit(rng, n))

    parts = [ordinary(4 * 32)]
    for dead in (False, True):
        for j in range(32):
            w = ordinary(32)
            w[j, 3] = 0.0
            if dead:
                w[j, 7] = 0.0
            parts.append(w)
    dead = ordinary(64)
    dead[:, 7] = 0.0
    dead[::7, 4] = 0.0
    tail = ordinary(13)
    tail[5, 5] = 0.0
    parts += [dead, tail]
    return np.concatenate(parts)


SETS = {"guard": lambda sc, rng: (guard_edge_rays(sc, rng), None), "ties": tie_rays,
        "midpoint": lambda sc, rng: (midpoint_rays(sc, rng), None), "warps": lambda sc, rng: (warp_rays(sc, rng), None)}


def ray_set(sc, name, seed):
    return SETS[name](sc, np.random.default_rng([21, seed, len(name)]))


def start_index(sc, slots):
    """The oracle's starting beam.index for starting slots (the plane the slot holds)."""
    if slots is None:
        return None
    return np.where(slots == NONE, NONE, sc.indices[np.minimum(slots, len(sc.indices) - 1)]).astype(np.uint32)


def first_bad(mask, rays, *cols):
    i = np.nonzero(mask)[0]
    if len(i) == 0:
        return ""
    j = int(i[0])
    return (f"{len(i)} rays, first #{j}: ray {rays[j].view(np.uint32).tolist()} = {rays[j].tolist()}; "
            + "; ".join(f"{name} {a[j]} vs {b[j]}" for name, a, b in cols))


def compare(got, ref, rays, what):
    """Bit-for-bit agreement of the GPU probe with the oracle: t, index and the four traversal counts."""
    assert not ref["overflow"].any(), what
    cols = [("t bits", got["t"].view(np.uint32), ref["t"].view(np.uint32)), ("index", got["index"], ref["index"])]
    cols += [(k, got[k].astype(np.uint64), ref[k]) for k in ("inner", "leaf", "rect", "max_stack")]
    bad = np.zeros(len(rays), bool)
    for _, a, b in cols:
        bad |= a != b
    assert not bad.any(), f"{what}: {first_bad(bad, rays, *cols)}"


def probe_and_check(renderer, oracle, sc, cls, rays, slots, flags, what, refs):
    got = renderer.trace_rays(rays, slots, flags)
    want_lit = lit(rays, flags, cls)
    bad = got["lit"] != want_lit
    assert not bad.any(), f"{what} lit: {first_bad(bad, rays, ('lit', got['lit'], want_lit))}"
    want_form = warp_form(rays, want_lit, flags, cls)
    bad = got["form"] != want_form
    assert not bad.any(), f"{what} form: {first_bad(bad, rays, ('form', got['form'], want_form))}"
    key = flags & RCP_SLAB
    if key not in refs:
        refs[key] = oracle.trace_rays(sc, rays, start_index(sc, slots), flags=key)
    compare(got, refs[key], rays, what)
    dead = rays[:, 7] == 0
    assert (got["t"][dead].view(np.uint32) == rays[dead, 6].view(np.uint32)).all(), what
    assert not (got["inner"][dead] | got["leaf"][dead] | got["rect"][dead] | got["max_stack"][dead]).any(), what
    return got


# ---- without a GPU ----------------------------------------------------------------------------------------------------------

def test_guard_restatement_on_its_edges():
    o0 = F32(1.0)
    assert axis_safe(o0, F32(2.0 ** -60)) and axis_safe(o0, F32(-(2.0 ** 60))) and axis_safe(o0, up(2.0 ** -60))
    assert not axis_safe(o0, down(2.0 ** -60)) and not axis_safe(o0, up(2.0 ** 60)) and not axis_safe(o0, F32(0.0))
    assert not axis_safe(o0, F32(np.nan)) and not axis_safe(o0, F32(np.inf))
    d0 = F32(1.0)
    assert axis_safe(F32(0.0), d0) and axis_safe(F32(-0.0), d0) and axis_safe(F32(2.0 ** -40), d0) and axis_safe(F32(-(2.0 ** 30)), d0)
    assert not axis_safe(down(2.0 ** -40), d0) and not axis_safe(up(2.0 ** 30), d0) and not axis_safe(F32(np.nan), d0)
    assert rcp_safe(F32(1e38), F32(2.0 ** -126)) and rcp_safe(FLT_MAX, F32(2.0 ** 126))
    assert not rcp_safe(o0, F32(2.0 ** -126 - 2.0 ** -149)) and not rcp_safe(o0, up(2.0 ** 126)) and not rcp_safe(F32(np.inf), d0)
    assert not rcp_safe(o0, F32(0.0)) and not rcp_safe(F32(np.nan), d0)


def test_warp_form_restatement():
    cls = dict(slab=True, rect=True, axis=True, y_table=5)
    rng = np.random.default_rng(3)
    r = _rays(rng.uniform(-1, 1, (40, 3)).astype(F32), _unit(rng, 40))
    r[3, 3] = 0.0                                         # literal lane in warp 0
    r[35, 7], r[35, 4] = 0.0, 0.0                          # dead literal lane in the partial warp 1
    lb = lit(r, 0, cls)
    assert lb[3] and lb[35] and lb.sum() == 2
    f = warp_form(r, lb, 0, cls)
    assert (f[:32] == MIXED).all() and (f[32:] == AXIS | YTAB).all()
    assert (warp_form(r, lit(r, NO_Y_TABLE, cls), NO_Y_TABLE, cls)[32:] == AXIS).all()
    assert (warp_form(r, lit(r, GENERAL_RECTS, cls), GENERAL_RECTS, cls)[32:] == YTAB).all()
    assert (warp_form(r, lit(r, RCP_SLAB, cls), RCP_SLAB, cls) == np.r_[[MIXED | RCP] * 32, [RCP] * 8]).all()
    assert (warp_form(r, lit(r, FORCE_LITERAL, cls), FORCE_LITERAL, cls) == MIXED).all()
    assert (warp_form(r, lb, 0, dict(cls, rect=False)) == MIXED).all()
    assert (lit(r, 0, dict(cls, slab=False))).all()


def test_midpoint_construction_is_exact_and_close():
    """RN(b - o) is x exactly, and x / d lies within 6 * 2^-48 (relative) of the midpoint between its two float neighbours."""
    from fractions import Fraction

    rng = np.random.default_rng(5)
    for b in (F32(5.0), F32(-45.0), F32(0.0), F32(3.0e-3), F32(-2.0 ** 21), F32(7.25e6)):
        for s in (1.0, -1.0):
            for _ in range(20):
                o, d, x = midpoint_operands(rng, b, s)
                assert F32(b - o) == x and np.sign(d) == s
                q = Fraction(float(x)) / Fraction(float(d))
                below = F32(float(q))
                if Fraction(float(below)) > q:
                    below = np.nextafter(below, F32(-np.inf))
                mid = (Fraction(float(below)) + Fraction(float(np.nextafter(below, F32(np.inf))))) / 2
                assert abs(q - mid) <= 6 * Fraction(1, 2 ** 48) * abs(q), (b, o, d, x)


def test_ray_sets_reach_their_edges(mm):
    sc = scene(mm, "maze10")
    rng = np.random.default_rng(1)
    g = guard_edge_rays(sc, rng, per=4)
    for k in range(3):
        dk = np.abs(g[:, 3 + k]).view(np.uint32)
        for v in D_EDGES:
            assert (dk == np.abs(v).view(np.uint32)).any() if v == v else np.isnan(g[:, 3 + k]).any()
        ok = np.abs(g[:, k]).view(np.uint32)
        for v in O_EDGES:
            assert (ok == np.abs(v).view(np.uint32)).any() if v == v else np.isnan(g[:, k]).any()
    b = bulk_rays(sc, rng, 1 << 14)
    e = ((b[:, 3:6].view(np.uint32) >> 23) & 0xFF).astype(int) - 127
    assert e.min() == -64 and e.max() == 64
    t, slots = tie_rays(sc, rng, per=256)
    q = t[:, 3:6]
    assert ((np.abs(q).view(np.uint32) & 0x7FFFFF) == 0).all()    # power-of-two directions
    assert (slots != NONE).sum() == 256 and (t[slots != NONE, 6] < 1e30).all()
    w = warp_rays(sc, rng)
    assert len(w) % 32 == 13
    lb = lit(w, 0, _classification("maze10"))
    assert lb[128:128 + 32 * 32].reshape(32, 32).nonzero()[1].tolist() == list(range(32))


@pytest.mark.parametrize("name", ["maze10", "shelves8", "tilted_0", "wide_tilted_two_levels", "tiny_coord", "far_0"])
@pytest.mark.parametrize("rcp", [False, True])
def test_oracle_entry_matches_numpy_transcription(mm, oracle, name, rcp):
    """mmo_trace_rays against np_oracle._traverse on every ray set: t and index per ray, counters summed."""
    from oracle import np_oracle

    sc = scene(mm, name)
    rng = np.random.default_rng([22, len(name), int(rcp)])
    rays = np.concatenate([guard_edge_rays(sc, rng, per=8), bulk_rays(sc, rng, 1500), tie_rays(sc, rng, per=200)[0],
                           midpoint_rays(sc, rng, per=2), warp_rays(sc, rng)])
    flags = RCP_SLAB if rcp else 0
    ref = oracle.trace_rays(sc, rays, flags=flags)
    alive = rays[:, 7] != 0
    a = rays[alive]
    cnt = {"rays": 0, "inner_visits": 0, "leaf_visits": 0, "rect_tests": 0, "max_stack": 0}
    np_oracle.RCP_SLAB = rcp
    try:
        with np.errstate(all="ignore"):
            t, idx = np_oracle._traverse(sc, [a[:, i].copy() for i in range(3)], [a[:, 3 + i].copy() for i in range(3)],
                                         a[:, 6].copy(), np.full(len(a), NONE, np.uint32), cnt)
    finally:
        np_oracle.RCP_SLAB = False
    assert (t.view(np.uint32) == ref["t"][alive].view(np.uint32)).all()
    assert (idx == ref["index"][alive]).all()
    assert cnt["inner_visits"] == ref["inner"].sum() and cnt["leaf_visits"] == ref["leaf"].sum()
    assert cnt["rect_tests"] == ref["rect"].sum() and cnt["max_stack"] == ref["max_stack"].max()
    assert (ref["t"][~alive].view(np.uint32) == rays[~alive, 6].view(np.uint32)).all() and not ref["inner"][~alive].any()
    assert not ref["overflow"].any() and (ref["t"] < 1e30).any()


def _sass_counts():
    import shutil
    import subprocess
    obj = os.path.join(ROOT, "mirror_maze_b200", "build", "render_kernel.o")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not (os.path.exists(obj) and os.path.exists(tool)):
        pytest.skip("needs the built render_kernel.o and cuobjdump")
    sass = subprocess.run([tool, "-sass", obj], capture_output=True, text=True, check=True).stdout
    counts, name = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            counts[name] = [0, 0, 0]
        elif name:
            for i, op in enumerate(("FADD2", "FMUL2", "FFMA2")):
                if f" {op} " in line:
                    counts[name][i] += 1
    return counts


def test_probe_instruction_mix_matches_the_trace_kernels():
    """probe_rays_kernel compiles its own copies of traverse: without the y-table the five of trace_kernel (60 : 60 : 108),
    with it the three of trace_ytab_kernel (44 : 44 : 132).  A fused, dropped or extra packed instruction changes the counts."""
    counts = _sass_counts()
    probes = {n: tuple(c) for n, c in counts.items() if "probe_rays_kernel" in n}
    assert len(probes) == 2
    for n, c in probes.items():
        assert c == ((44, 44, 132) if "probe_rays_kernelILb1E" in n else (60, 60, 108)), (n, c)


# ---- on the GPU -------------------------------------------------------------------------------------------------------------

def _upload(mm, renderer, noise, name):
    sc = scene(mm, name)
    renderer.upload_scene(sc, noise)
    cls = _classification(name)
    info = renderer.scene_info()
    assert (info["fast_slab_ok"], info["fast_rect_ok"], info["axis_rects"]) == (int(cls["slab"]), int(cls["rect"]), int(cls["axis"]))
    return sc, cls


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("which", sorted(SETS))
def test_rays_match_oracle_in_every_form(mm, oracle, noise, renderer, which, name):
    sc, cls = _upload(mm, renderer, noise, name)
    rays, slots = ray_set(sc, which, SCENES.index(name))
    refs = {}
    for label, flags in FLAGS.items():
        got = probe_and_check(renderer, oracle, sc, cls, rays, slots, flags, f"{name} {which} {label}", refs)
        if which == "warps" and flags == 0 and cls["slab"] and cls["rect"]:     # both sides of the vote
            assert set(np.unique(got["form"]).tolist()) == {MIXED, warp_form(rays[:1], np.zeros(1, bool), 0, cls)[0]}


@pytest.mark.gpu
@pytest.mark.parametrize("name", BULK_SCENES)
def test_wide_range_directions_in_bulk(mm, oracle, noise, renderer, name):
    sc, cls = _upload(mm, renderer, noise, name)
    rays = bulk_rays(sc, np.random.default_rng([23, SCENES.index(name)]), BULK_N)
    refs = {}
    for label, flags in FLAGS.items():
        got = probe_and_check(renderer, oracle, sc, cls, rays, None, flags, f"{name} bulk {label}", refs)
        if flags == 0:
            assert 0 < got["lit"].sum() < len(rays) and (got["t"] < 1e30).any()


@pytest.mark.gpu
def test_probe_refuses_bad_arguments(mm, noise, renderer):
    _upload(mm, renderer, noise, "maze10")
    r = _rays(np.zeros((4, 3), F32), np.ones((4, 3), F32))
    with pytest.raises(mm.MMError):
        renderer.trace_rays(r, flags=mm.FLAG_COUNTERS)
    with pytest.raises(mm.MMError):
        renderer.trace_rays(r, slots=np.full(4, 1 << 20, np.uint32))
    assert renderer.trace_rays(r)["inner"].sum() > 0
