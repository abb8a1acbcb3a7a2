"""Scenes the mazes never produce, rendered against the oracle: tilted rects, wide leaves, 1 to 9 child y-intervals and
every classification the upload makes.

A maze has 5 child y-intervals, axis-aligned rects and leaves of at most 2 rects, so the general rect test on tilted
geometry, leaf loops past their second rect, the y-table at other interval counts and the fallbacks of scenes outside the
guarded ranges are not exercised by the maze cases.  The seeded scene families here reach each of those:

- tilted: 40-80 rects of random orientation around the camera (v and u not perpendicular, lengths 1-30); "far" puts an
  integer-edged cloud at 2^22, where every coordinate is a multiple of 0.5, so edge tests land exactly on their thresholds;
- walls: vertical walls rotated about y, their heights drawn from k bands, with exactly 1, 2, 3, 5, 6, 7, 8 and 9 child
  y-intervals: general rects with (and, at 9, without) the y-table;
- maze_mirrors: the 10x10 maze plus three tilted mirrors, so the whole scene takes the general rect test;
- wide: hand-built BVHs with leaves of 3, 7, 31 and 126 rects and a root that is a leaf of 126, axis-aligned (RectA) and
  tilted (RectI), shuffled indices (slot != plane id) and coplanar overlapping rects at equal distance (the strict
  `a < t` tie rule decides the hit);
- scaled: the 10x10 maze times 2^-3, 3.7 and 2^20, and the maze plus one coordinate in (0, 2^-10) (fast_slab_ok = 0);
- degenerate: rotated walls plus zero-length edges, rects whose plane holds the camera, rects nearer than the 0.1
  self-hit epsilon, bit-distinct +-0 y-bounds and a y-bound equal to the camera's y; signed_zero: the last two in a scene
  few enough y-intervals for the y-table, which tells +-0 apart by bits.

The CPU tests check each family's classification with an independent restatement of the upload's rules and compare the
C++ oracle with oracle/np_oracle.py.  The GPU tests check scene_info() against that classification and compare every
kernel variant bit for bit with the oracle: per-path arrays, image, counters and the tail's mm_last_tail."""
import functools
import types

import numpy as np
import pytest

from test_tail_and_shapes import assert_same, assert_tail, gpu_render, with_flags
from test_y_table import MAX_Y_INTERVALS, y_intervals

F32 = np.float32
MAX_LEAF = 126                        # render_kernel.cuh: kMaxLeafCount (7-bit count field of a leaf descriptor)
ERR_UNSUPPORTED = -5
# integer edge vectors with integer lengths (a^2 + b^2 + c^2 = L^2): their thresholds are exactly L^2
QUADS = [(1, 2, 2), (2, 3, 6), (1, 4, 8), (4, 4, 7), (2, 6, 9), (6, 6, 7), (3, 4, 12), (2, 10, 11), (2, 5, 14), (8, 9, 12)]
# y-bands of the wall scenes; several share min.y, so intervals that differ only in max.y are common
BANDS = [(-8.0, 2.0), (-8.0, 6.0), (-4.0, 2.0), (-8.0, -1.0), (-2.0, 4.0), (-6.0, 3.0), (-8.0, 0.5), (-3.0, 6.0)]
# (k bands, seed) with exactly the named number of child y-intervals (searched once, pinned by a CPU test)
WALLS = {1: (1, 0), 2: (2, 0), 3: (3, 0), 5: (5, 28), 6: (5, 1), 7: (5, 2), 8: (6, 0), 9: (6, 2)}


# ---- scene generator -----------------------------------------------------------------------------------------------------

def _finish(planes, rng, camera, yaw=None, nodes=None, indices=None, mirror_frac=0.3, emit_frac=0.25):
    """Materials (0 diffuse, 1 mirror), emissions (w != 1 on the emitters) and, unless given, the builder's BVH."""
    from mirror_maze_b200.host import build_bvh

    n = len(planes)
    materials = (rng.random(n) < mirror_frac).astype(np.uint8)
    emissions = np.zeros((n, 4), F32)
    emit = rng.random(n) < emit_frac
    emissions[emit, :3] = rng.uniform(0.2, 1.0, size=(int(emit.sum()), 3))
    emissions[emit, 3] = rng.choice([0.5, 1.5, 2.5, 4.0], size=int(emit.sum()))
    if nodes is None:
        nodes, indices = build_bvh(planes)
    return types.SimpleNamespace(planes=planes, nodes=nodes, indices=indices, materials=materials, emissions=emissions,
                                 camera=tuple(float(c) for c in camera), yaw=yaw)


def _planes(rows):
    from mirror_maze_b200.host import PLANE_DTYPE

    P = np.zeros(len(rows), dtype=PLANE_DTYPE)
    for i, r in enumerate(rows):
        P[i] = r
    return P


def _edge(rng, integer):
    if integer:
        q = np.array(QUADS[int(rng.integers(len(QUADS)))], dtype=F32)
        return rng.permutation(q) * rng.choice([-1.0, 1.0], size=3).astype(F32)
    d = rng.normal(size=3)
    return (d / np.linalg.norm(d) * rng.uniform(1.0, 30.0)).astype(F32)


def tilted(seed, far=False):
    """40-80 rects of random orientation in a cloud around the camera.  far: integer edges and origins at 2^22 + k."""
    rng = np.random.default_rng([11, seed])
    off = np.full(3, 2.0 ** 22, F32) if far else np.zeros(3, F32)
    rows = []
    for _ in range(int(rng.integers(40, 81))):
        v, u = _edge(rng, far or rng.random() < 0.5), _edge(rng, far or rng.random() < 0.5)
        c = rng.uniform(-35.0, 35.0, size=3).astype(F32)
        o = np.round(c - F32(0.5) * (v + u)) if far else c - F32(0.5) * (v + u)
        rows.append((o + off, v, u, rng.uniform(0.2, 0.95, size=3)))
    return _finish(_planes(rows), rng, off + F32([0.5, 0.25, -0.5]), yaw=float(rng.uniform(0, np.pi)))


def _wall_rows(rng, k, n):
    rows = []
    for _ in range(n):
        lo, hi = BANDS[int(rng.integers(k))]
        th, L = rng.uniform(0.0, 2.0 * np.pi), rng.uniform(2.0, 12.0)
        v = np.array([L * np.cos(th), 0.0, L * np.sin(th)], F32)
        c = rng.uniform(-40.0, 40.0, size=2)
        o = np.array([c[0], hi, c[1]], F32) - F32(0.5) * np.array([v[0], 0.0, v[2]], F32)
        rows.append((o, v, (0.0, lo - hi, 0.0), rng.uniform(0.2, 0.95, size=3)))
    return rows


def walls(k, seed):
    """Vertical walls rotated about y by random angles, their y-extents drawn from the first k BANDS."""
    rng = np.random.default_rng([12, k, seed])
    rows = _wall_rows(rng, k, int(rng.integers(24, 41)))
    return _finish(_planes(rows), rng, (0.5, 0.0, 0.5), yaw=float(rng.uniform(0, np.pi)))


def maze_mirrors(mm):
    """The 10x10 maze plus three tilted mirrors in front of the camera at (-5, 0, -45)."""
    base = mm.MazeScene(10, 0)
    extra = _planes([((-7.0, 1.5, -41.0), (3.0, 0.5, 1.0), (0.4, -3.0, 0.3), (0.9, 0.9, 0.9)),
                     ((-3.5, -1.0, -38.0), (2.0, 1.0, -1.5), (0.5, -2.5, 0.5), (0.8, 0.9, 0.8)),
                     ((-6.0, 0.5, -36.0), (1.5, -0.5, 2.5), (-0.3, -2.0, 0.2), (0.9, 0.8, 0.9))])
    from mirror_maze_b200.host import build_bvh
    planes = np.concatenate([base.planes, extra])
    nodes, indices = build_bvh(planes)
    return types.SimpleNamespace(planes=planes, nodes=nodes, indices=indices,
                                 materials=np.concatenate([base.materials, np.ones(3, np.uint8)]),
                                 emissions=np.concatenate([base.emissions, np.zeros((3, 4), F32)]),
                                 camera=(-5.0, 0.0, -45.0), yaw=None)


def _tile_groups(rng, tilt):
    """Four groups of rects in view of a camera at the origin looking down +z: 3 (left wall), 7 (floor), 31 (right wall) and
    126 (back wall: 108 tiles and 18 coplanar overlapping copies, same origin and normal, an edge halved or identical)."""
    def rect(o, v, u):
        v, u = np.array(v, F32), np.array(u, F32)
        if tilt:                                              # a fixed shear: every tile tilted, v and u not perpendicular
            v = v + F32(0.25) * np.array([v[2], v[0] + v[1], v[1]], F32) + F32(0.125) * np.abs(v).sum()
            u = u + F32(0.125) * np.array([u[1], u[2], u[0]], F32)
        return [np.array(o, F32), v, u, rng.uniform(0.2, 0.95, size=3).astype(F32)]

    back = [rect((-36.0 + 6.0 * i, -21.0 + 6.0 * j, 30.0), (6.0, 0.0, 0.0), (0.0, -6.0, 0.0)) for i in range(12) for j in range(9)]
    dups = []
    for idx in rng.choice(len(back), size=18, replace=False):
        o, v, u, _ = back[idx]
        half = rng.random() < 0.5
        dups.append([o, v * F32(0.5) if half else v, u, rng.uniform(0.2, 0.95, size=3).astype(F32)])
    back = back + dups
    back = [back[i] for i in rng.permutation(len(back))]      # copies before and after their originals, at slots < and >= 64
    right = [rect((25.0, 12.0 - 6.0 * j, 5.0 + 5.0 * i), (0.0, 0.0, 5.0), (0.0, -6.0, 0.0)) for i in range(5) for j in range(6)]
    right.append([right[7][0], right[7][1], right[7][2] * F32(0.5), rng.uniform(0.2, 0.95, size=3).astype(F32)])
    floor = [rect((-30.0 + 9.0 * i, -10.0, 5.0 + 3.0 * i), (8.0, 0.0, 0.0), (0.0, 0.0, 20.0)) for i in range(7)]
    left = [rect((-25.0, 10.0, 5.0 + 9.0 * i), (0.0, 0.0, 8.0), (0.0, -20.0, 0.0)) for i in range(3)]
    return [left, floor, right, back]


def _box(rows):
    c = []
    for o, v, u, _ in rows:
        c += [o, o + v, o + u, (o + v) + u]
    c = np.array(c, F32)
    return c.min(axis=0), c.max(axis=0)


def _hand_built(rng, groups, tree):
    """Planes in shuffled order; leaf j holds slots [first_j, first_j + len(groups[j])) in group order, indices[slot] is a
    random plane id.  tree: 'root_leaf' (one leaf) or 'two_levels' (root -> (A, B), A -> (g0, g1), B -> (g2, g3))."""
    from mirror_maze_b200.host import NODE_DTYPE

    slots = [r for g in groups for r in g]
    n = len(slots)
    perm = rng.permutation(n).astype(np.uint32)               # indices[slot] = plane id
    planes = _planes([tuple(slots[s]) for s in np.argsort(perm)])
    firsts = np.cumsum([0] + [len(g) for g in groups])
    if tree == "root_leaf":
        nodes = np.zeros(1, dtype=NODE_DTYPE)
        nodes[0]["aabb_min"], nodes[0]["aabb_max"] = _box(slots)
        nodes[0]["left_first"], nodes[0]["tri_count"] = 0, n
        return planes, nodes, perm
    nodes = np.zeros(7, dtype=NODE_DTYPE)
    members = {3: [0], 4: [1], 5: [2], 6: [3], 1: [0, 1], 2: [2, 3], 0: [0, 1, 2, 3]}
    for i, gs in members.items():
        nodes[i]["aabb_min"], nodes[i]["aabb_max"] = _box([r for g in gs for r in groups[g]])
    for i, lf in ((0, 1), (1, 3), (2, 5)):
        nodes[i]["left_first"], nodes[i]["tri_count"] = lf, 0
    for j in range(4):
        nodes[3 + j]["left_first"], nodes[3 + j]["tri_count"] = firsts[j], len(groups[j])
    return planes, nodes, perm


def wide(tilt, tree, extra=0):
    """Leaves of 3, 7, 31 and 126 rects (tree 'two_levels'), or one root leaf of the 126 (+ extra) back-wall rects."""
    rng = np.random.default_rng([13, int(tilt), len(tree), extra])
    groups = _tile_groups(rng, tilt)
    if tree == "root_leaf":
        groups = [groups[3] + [groups[2][i] for i in range(extra)]]
    planes, nodes, indices = _hand_built(rng, groups, tree)
    return _finish(planes, rng, (0.0, 0.0, 0.0), nodes=nodes, indices=indices)


def scaled(mm, s):
    """The 10x10 maze with every plane coordinate and the camera multiplied by s (float32), BVH rebuilt."""
    from mirror_maze_b200.host import build_bvh

    base = mm.MazeScene(10, 0)
    planes = base.planes.copy()
    for f in ("origin", "v", "u"):
        planes[f] = planes[f] * F32(s)
    nodes, indices = build_bvh(planes)
    return types.SimpleNamespace(planes=planes, nodes=nodes, indices=indices, materials=base.materials,
                                 emissions=base.emissions, camera=tuple(float(F32(c) * F32(s)) for c in (-5.0, 0.0, -45.0)),
                                 yaw=None)


def tiny_coord(mm):
    """The 10x10 maze plus a panel whose box starts at x = 1e-4, inside (0, 2^-10): outside the exact slab quotient's range."""
    from mirror_maze_b200.host import build_bvh

    base = mm.MazeScene(10, 0)
    planes = np.concatenate([base.planes, _planes([((1e-4, 1.0, -30.0), (2.0, 0.0, 0.0), (0.0, -3.0, 0.0), (0.7, 0.2, 0.2))])])
    nodes, indices = build_bvh(planes)
    return types.SimpleNamespace(planes=planes, nodes=nodes, indices=indices,
                                 materials=np.concatenate([base.materials, np.zeros(1, np.uint8)]),
                                 emissions=np.concatenate([base.emissions, F32([[1.0, 0.4, 0.2, 2.5]])]),
                                 camera=(-5.0, 0.0, -45.0), yaw=None)


DEGENERATE_SEED = 0
CAM_Y = 0.75


def degenerate(seed=DEGENERATE_SEED):
    """Rotated walls (2 bands) plus: zero-length edges; a horizontal rect at the camera's y and a vertical one through the
    camera (their planes hold it: a = +-0 for primary rays, 0 / 0 along the plane); rects at 0.05, 0.1 and 0.12 in front of
    it (the a > 0.1 epsilon); walls from y = -0.0 and y = +0.0 up (bit-distinct child bounds) and a wall whose top is the
    camera's y."""
    rng = np.random.default_rng([14, seed])
    cam = F32([0.5, CAM_Y, 0.5])
    rows = _wall_rows(rng, 2, 20)
    rows += [((4.0, 1.0, 8.0), (0.0, 0.0, 0.0), (0.0, -3.0, 0.0), (0.9, 0.2, 0.2)),          # v = 0
             ((-4.0, 1.0, 9.0), (2.0, 0.5, 0.0), (0.0, 0.0, 0.0), (0.2, 0.9, 0.2)),          # u = 0
             ((-9.5, CAM_Y, -9.5), (20.0, 0.0, 0.0), (0.0, 0.0, 20.0), (0.6, 0.6, 0.6)),     # horizontal, through the camera
             ((0.5, 3.0, -5.0), (0.0, 0.0, 12.0), (0.0, -4.0, 0.0), (0.5, 0.5, 0.8)),        # vertical, through the camera
             ((0.3, 0.95, 0.55), (0.4, 0.0, 0.0), (0.0, -0.4, 0.0), (0.9, 0.9, 0.1)),        # a = 0.05 ahead
             ((0.2, 1.0, 0.6), (0.3, 0.05, 0.0), (0.0, -0.5, 0.0), (0.1, 0.9, 0.9)),         # a = 0.1 ahead
             ((0.35, 0.9, 0.62), (0.2, 0.0, 0.02), (0.0, -0.3, 0.0), (0.9, 0.1, 0.9)),       # a = 0.12 ahead
             ((-12.0, -0.0, 14.0), (5.0, 0.0, 3.0), (0.0, 3.0, 0.0), (0.8, 0.7, 0.6)),       # min.y = -0.0
             ((12.0, 0.0, 14.0), (-5.0, 0.0, 3.0), (0.0, 3.0, 0.0), (0.6, 0.7, 0.8)),        # min.y = +0.0
             ((6.0, -4.0, -12.0), (4.0, 0.0, -3.0), (0.0, 4.0 + CAM_Y, 0.0), (0.7, 0.7, 0.7))]   # max.y = the camera's y
    return _finish(_planes(rows), rng, cam, yaw=0.3)


def signed_zero(seed=0):
    """One band of rotated walls plus walls from y = -0.0 and y = +0.0 up and one whose top is the camera's y: few enough
    child y-intervals for the y-table, two of them told apart only by the sign of a zero."""
    rng = np.random.default_rng([15, seed])
    rows = _wall_rows(rng, 1, 16)
    rows += [((-12.0, -0.0, 14.0), (5.0, 0.0, 3.0), (0.0, 3.0, 0.0), (0.8, 0.7, 0.6)),
             ((12.0, 0.0, 14.0), (-5.0, 0.0, 3.0), (0.0, 3.0, 0.0), (0.6, 0.7, 0.8)),
             ((6.0, -4.0, -12.0), (4.0, 0.0, -3.0), (0.0, 4.0 + CAM_Y, 0.0), (0.7, 0.7, 0.7))]
    return _finish(_planes(rows), rng, (0.5, CAM_Y, 0.5), yaw=2.0)


def build_scene(mm, name):
    fam, _, arg = name.partition("_")
    if fam == "tilted":
        return tilted(int(arg))
    if fam == "far":
        return tilted(int(arg), far=True)
    if fam == "walls":
        return walls(*WALLS[int(arg)])
    if name == "maze_mirrors":
        return maze_mirrors(mm)
    if fam == "wide":
        tilt, tree = arg.split("_", 1)
        return wide(tilt == "tilted", tree)
    if fam == "scaled":
        return scaled(mm, {"eighth": 2.0 ** -3, "3.7": 3.7, "2p20": 2.0 ** 20}[arg])
    if name == "tiny_coord":
        return tiny_coord(mm)
    if name == "degenerate":
        return degenerate()
    if name == "signed_zero":
        return signed_zero()
    raise KeyError(name)


# What each scene is built to reach (keys of classify(); a missing key is not part of the scene's purpose).  The upload's
# report must equal classify() on every scene; these pin that each family reaches what it is for.
EXPECT = {
    "tilted_0": dict(axis=False, rect=True, slab=True, y_table=0),
    "tilted_1": dict(axis=False, rect=True, slab=True, y_table=0),
    "far_0": dict(axis=False, rect=True, slab=True, y_table=0),
    "far_1": dict(axis=False, rect=True, slab=True, y_table=0),
    **{f"walls_{n}": dict(axis=False, rect=True, slab=True, n_yiv=n, y_table=n if n <= MAX_Y_INTERVALS else 0) for n in WALLS},
    "maze_mirrors": dict(axis=False, rect=True, slab=True),
    "wide_axis_two_levels": dict(axis=True, rect=True, slab=True, max_leaf=126, depth=3, n_yiv=4, y_table=4),
    "wide_tilted_two_levels": dict(axis=False, rect=True, slab=True, max_leaf=126, depth=3, n_yiv=4, y_table=4),
    "wide_axis_root_leaf": dict(axis=True, rect=True, slab=True, max_leaf=126, depth=1, n_yiv=0, y_table=0),
    "wide_tilted_root_leaf": dict(axis=False, rect=True, slab=True, max_leaf=126, depth=1, n_yiv=0, y_table=0),
    "scaled_eighth": dict(axis=True, rect=True, slab=True, n_yiv=5, y_table=5),
    "scaled_3.7": dict(axis=True, rect=True, slab=True, n_yiv=5, y_table=5),
    "scaled_2p20": dict(axis=False, rect=False, slab=True, n_yiv=5, y_table=5),
    "tiny_coord": dict(slab=False, y_table=0),
    "degenerate": dict(axis=False, rect=True, slab=True),
    "signed_zero": dict(axis=False, rect=True, slab=True, n_yiv=5, y_table=5),
}
NAMES = sorted(EXPECT)


@functools.lru_cache(maxsize=None)
def _scene_cached(name):
    import mirror_maze_b200 as mm
    return build_scene(mm, name)


def scene(mm, name):
    mm.load_library()
    return _scene_cached(name)


# ---- an independent restatement of the upload's classification -------------------------------------------------------------

def _coord_ok(c):
    """scene_prep.cpp coord_ok: 0, or 2^-10 <= |c| <= 2^30 (NaN fails)."""
    a = abs(float(c))
    return a == 0.0 or 2.0 ** -10 <= a <= 2.0 ** 30


def _length(e):
    """sqrt(dot(e, e)) in float32, summed as the upload sums it: (x*x + y*y) + z*z."""
    e = np.asarray(e, F32)
    return np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2], dtype=F32)


def classify(sc):
    """What the upload should report for a scene: fast_slab_ok, fast_rect_ok, axis_rects, bvh_depth, max_leaf, the child
    y-interval count and the y_table a default render uses."""
    from mirror_maze_b200 import host

    nodes = sc.nodes
    stack, depth, max_leaf, slab = [(0, 1)], 0, 0, True
    while stack:
        i, d = stack.pop()
        depth = max(depth, d)
        lf, tc = int(nodes[i]["left_first"]), int(nodes[i]["tri_count"])
        if tc:
            max_leaf = max(max_leaf, tc)
            continue
        for c in (lf, lf + 1):
            stack.append((c, d + 1))
            mn, mx = nodes[c]["aabb_min"], nodes[c]["aabb_max"]
            slab &= all(_coord_ok(x) for x in list(mn) + list(mx)) and bool((mn <= mx).all())
    rect = all(host.rect_edge_thresholds(_length(p[e])) is not None for p in sc.planes for e in ("v", "u"))
    axis = rect and all(host.axis_rect(p) is not None for p in sc.planes)
    n_yiv = y_intervals(nodes)
    return dict(slab=slab, rect=rect, axis=axis, depth=depth, max_leaf=max_leaf, n_yiv=n_yiv,
                y_table=n_yiv if slab and n_yiv <= MAX_Y_INTERVALS else 0)


def dispatch(mm, sc, spp, W=48, H=32, chunk=4, flags=0, time=7):
    u = mm.default_uniform(10, W, H, chunk, time, camera_center=sc.camera, half_theta=sc.yaw)
    ch = mm.gen_chunks(W, H, chunk)
    return u, mm.full_frame_params(u, spp=spp, bounce_limit=8, mirror_limit=15, flags=flags), ch


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_family_reaches_its_classification(mm, name):
    from mirror_maze_b200 import host

    sc = scene(mm, name)
    got = classify(sc)
    for k, v in EXPECT[name].items():
        assert got[k] == v, f"{name}: {k} = {got[k]}, built for {v} ({got})"
    assert len(sc.indices) == len(sc.planes) and sorted(sc.indices.tolist()) == list(range(len(sc.planes)))
    if name.startswith(("tilted", "far")):
        assert 40 <= len(sc.planes) <= 80 and got["n_yiv"] > MAX_Y_INTERVALS
        assert all(host.axis_rect(p) is None for p in sc.planes)
    if name.startswith("wide"):
        assert (sc.indices != np.arange(len(sc.indices))).mean() > 0.9           # slot != plane id
        assert sc.emissions[sc.materials == 0, 3].max() != 1.0


def test_rule_restatements_on_their_edges(mm):
    """The coordinate and edge-length rules at the ends of their ranges, through the upload's own helpers where they exist."""
    from mirror_maze_b200 import host

    assert _coord_ok(0.0) and _coord_ok(-0.0) and _coord_ok(2.0 ** -10) and _coord_ok(-(2.0 ** 30))
    assert not _coord_ok(np.nextafter(F32(2.0 ** -10), F32(0))) and not _coord_ok(np.nextafter(F32(2.0 ** 30), F32(np.inf)))
    assert not _coord_ok(float("nan")) and not _coord_ok(1e-4)
    assert host.rect_edge_thresholds(F32(2.0 ** -20)) is not None and host.rect_edge_thresholds(F32(2.0 ** 23)) is not None
    assert host.rect_edge_thresholds(np.nextafter(F32(2.0 ** 23), F32(np.inf))) is None
    assert host.rect_edge_thresholds(np.nextafter(F32(2.0 ** -20), F32(0))) is None
    for a, b, c in QUADS:                                     # integer edges: the far edge's threshold is exactly L^2
        L = _length((a, b, c))
        assert L == round(float(L)) and host.rect_edge_thresholds(L)[1] == L * L


def test_wall_families_hit_every_interval_count(mm):
    """walls_n has exactly n child y-intervals, and some of them share min.y but not max.y (the y-table tells them apart)."""
    for n in WALLS:
        nodes = scene(mm, f"walls_{n}").nodes
        assert y_intervals(nodes) == n
    iv = _child_intervals(scene(mm, "walls_8").nodes)
    mins = [a for a, _ in iv]
    assert len(set(mins)) < len(iv)


def _child_intervals(nodes):
    out = set()
    for i in range(len(nodes)):
        if nodes[i]["tri_count"] == 0:
            for c in (int(nodes[i]["left_first"]), int(nodes[i]["left_first"]) + 1):
                out.add((F32(nodes[c]["aabb_min"][1]).tobytes(), F32(nodes[c]["aabb_max"][1]).tobytes()))
    return out


def test_degenerate_scenes_have_their_edges(mm):
    sc = scene(mm, "degenerate")
    lens = [(_length(p["v"]), _length(p["u"])) for p in sc.planes]
    assert any(lv == 0 for lv, _ in lens) and any(lu == 0 for _, lu in lens)
    sc = scene(mm, "signed_zero")
    iv = _child_intervals(sc.nodes)
    zero_min = {a for a, _ in iv if np.frombuffer(a, F32)[0] == 0}
    assert len(zero_min) == 2, "+0 and -0 child bounds, told apart by bits"
    assert any(np.frombuffer(b, F32)[0] == F32(CAM_Y) for _, b in iv)              # a bound at the camera's y
    assert classify(sc)["y_table"] > 0


def test_leaf_beyond_the_descriptor_is_built_as_asked(mm):
    sc = wide(False, "root_leaf", extra=1)
    assert classify(sc)["max_leaf"] == MAX_LEAF + 1


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_numpy_transcription(mm, oracle, noise, name):
    """The C++ oracle against oracle/np_oracle.py on every family: per-path arrays, image and counters, bit for bit."""
    from oracle import np_oracle

    sc = scene(mm, name)
    u, p, ch = dispatch(mm, sc, 2, W=32, H=32)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    assert ref[1]["hits"] > 0
    assert_same(ref, np_oracle.render(sc, noise, u, p, ch), name)


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

VARIANTS = ["FLAG_NO_Y_TABLE", "FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_RCP_SLAB", "FLAG_NO_TAIL", "FLAG_POOL_KERNEL",
            "FLAG_REGROUP"]


def check_info(renderer, sc, name):
    info, want = renderer.scene_info(), classify(sc)
    got = dict(slab=info["fast_slab_ok"], rect=info["fast_rect_ok"], axis=info["axis_rects"], depth=info["bvh_depth"],
               max_leaf=info["max_leaf"])
    assert got == {k: int(want[k]) for k in got}, f"{name}: scene_info {info} vs {want}"
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_every_kernel_matches_oracle(mm, oracle, noise, renderer, name):
    sc = scene(mm, name)
    renderer.upload_scene(sc, noise)
    want = check_info(renderer, sc, name)
    u, p, ch = dispatch(mm, sc, 8)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    seg = ref[2]["segments"]
    got = gpu_render(mm, renderer, u, p, ch, True)
    assert renderer.scene_info()["y_table"] == want["y_table"], name
    assert_same(got, ref, name)
    assert_tail(mm, renderer, got[3], p, seg, name)
    if not want["slab"]:
        assert got[1]["literal_rays"] == got[1]["rays"], name
    literal = got[1]["literal_rays"]
    for v in VARIANTS:
        q = with_flags(mm, p, getattr(mm, v))
        r = oracle.render(sc, noise, u, q, ch, debug=True) if v == "FLAG_RCP_SLAB" else ref
        g = gpu_render(mm, renderer, u, q, ch, True)
        what = f"{name} {v}"
        assert_same(g, r, what)
        assert_tail(mm, renderer, g[3], q, r[2]["segments"], what)
        if v == "FLAG_NO_Y_TABLE":
            assert renderer.scene_info()["y_table"] == 0 and g[1]["literal_rays"] == literal, what
    g = gpu_render(mm, renderer, u, with_flags(mm, p, mm.FLAG_COUNTERS), ch, False)
    assert_same(g, (ref[0], ref[1], None), name + " COUNTERS")
    assert_tail(mm, renderer, g[3], p, seg, name + " COUNTERS")


# spp 64: 64-thread blocks; spp 128: 256-thread blocks, two pixels per block
SHAPES = {64: dict(W=32, H=32, chunk=2), 128: dict(W=32, H=16, chunk=2)}


@pytest.mark.gpu
@pytest.mark.parametrize("spp", sorted(SHAPES))
@pytest.mark.parametrize("name", NAMES)
def test_block_shapes_match_oracle(mm, oracle, noise, renderer, name, spp):
    sc = scene(mm, name)
    renderer.upload_scene(sc, noise)
    want = classify(sc)
    u, p, ch = dispatch(mm, sc, spp, **SHAPES[spp])
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    got = gpu_render(mm, renderer, u, p, ch, True)
    assert renderer.scene_info()["y_table"] == want["y_table"], name
    nt = gpu_render(mm, renderer, u, with_flags(mm, p, mm.FLAG_NO_Y_TABLE), ch, True)
    for g, what in ((got, f"{name} spp {spp}"), (nt, f"{name} spp {spp} NO_Y_TABLE")):
        assert_same(g, ref, what)
        assert_tail(mm, renderer, g[3], p, ref[2]["segments"], what)
    assert got[1]["literal_rays"] == nt[1]["literal_rays"]


@pytest.mark.gpu
def test_leaf_of_127_is_refused_and_the_context_still_renders(mm, oracle, noise):
    ok = scene(mm, "wide_tilted_root_leaf")
    u, p, ch = dispatch(mm, ok, 8)
    r = mm.Renderer(0)
    try:
        with pytest.raises(mm.MMError) as e:
            r.upload_scene(wide(False, "root_leaf", extra=1), noise)
        assert e.value.code == ERR_UNSUPPORTED
        r.upload_scene(ok, noise)
        with pytest.raises(mm.MMError) as e:
            r.upload_scene(wide(True, "root_leaf", extra=1), noise)
        assert e.value.code == ERR_UNSUPPORTED
        r.upload_scene(ok, noise)
        assert_same(gpu_render(mm, r, u, p, ch, True), oracle.render(ok, noise, u, p, ch, debug=True), "after a refused upload")
    finally:
        r.close()


@pytest.mark.gpu
def test_one_context_across_interval_counts(mm, oracle, noise):
    """One context takes scenes with 5, 8, 9, 1 and 5 y-intervals, axis-aligned and tilted in turn: every render equals a fresh
    context's and the oracle's bits and reports the new scene's y_table (no stale n_yiv, cfg_smem or axis-aligned rects)."""
    from test_y_table import scene_with_intervals

    seq = [("maze10", lambda: mm.MazeScene(10, 0), 5, True),
           ("walls_8", lambda: scene(mm, "walls_8"), 8, False),
           ("shelves9", lambda: scene_with_intervals(mm, lambda n: mm.MazeScene(n, 0), 9), 0, True),
           ("walls_1", lambda: scene(mm, "walls_1"), 1, False),
           ("maze16", lambda: mm.MazeScene(16, 0), 5, True)]
    r = mm.Renderer(0)
    try:
        for i, (label, make, n_yiv, axis) in enumerate(seq):
            sc = make()
            cam = getattr(sc, "camera", (-5.0, 0.0, -45.0))
            u = mm.default_uniform(10, 48, 32, 4, 3, camera_center=cam, half_theta=getattr(sc, "yaw", None))
            ch = mm.gen_chunks(48, 32, 4)
            p = mm.full_frame_params(u, spp=64 if i % 2 else 8, bounce_limit=8, mirror_limit=15)
            r.upload_scene(sc, noise)
            assert r.scene_info()["axis_rects"] == int(axis), label
            got = gpu_render(mm, r, u, p, ch, True)
            assert r.scene_info()["y_table"] == n_yiv, label
            fresh = mm.Renderer(0)
            try:
                fresh.upload_scene(sc, noise)
                f = gpu_render(mm, fresh, u, p, ch, True)
            finally:
                fresh.close()
            assert_same(got, f[:3], f"{label}: reused context vs fresh context")
            assert got[3] == f[3], label
            assert_same(got, oracle.render(sc, noise, u, p, ch, debug=True), label)
    finally:
        r.close()
