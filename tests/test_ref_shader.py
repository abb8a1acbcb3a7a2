"""The reference's OWN shader source against the oracle.

oracle/_ref/libref_shader.so is reference src/shaders.metal compiled unmodified as C++ (oracle/ref_shader/msl_shim.h
stands in for <metal_stdlib>) and run on the CPU; it is built where /root/reference exists and travels as a binary.
These tests pin oracle/mm_oracle.cpp — the restatement every CUDA parity test is checked against — to it: helper by
helper on random and edge inputs, and image for image on every dispatch shape the unmodified shader can address.
Where the library is absent the committed digests of its images (tests/golden/golden.json: ref_shader_image) are used."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from cases import REF_SHADER_CASES, build_case

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden.json")))


@pytest.fixture(scope="module")
def ref():
    from oracle import oracle as o, ref_shader
    if not ref_shader.available():
        o.build()                       # make -C oracle also builds _ref/libref_shader.so where /root/reference exists
    if not ref_shader.available():
        pytest.skip("oracle/_ref/libref_shader.so not built (needs /root/reference)")
    L = ref_shader.lib()
    L.ref_random.restype = C.c_float
    L.ref_random.argtypes = [C.POINTER(C.c_uint32)]
    L.ref_intersect_aabb.restype = C.c_float
    L.ref_intersect_aabb.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    L.ref_ray_rect.restype = C.c_int
    L.ref_ray_rect.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_float)]
    L.ref_quat_mult.restype = None
    L.ref_quat_mult.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    return ref_shader


def _bits(x):
    return np.float32(x).view(np.uint32)


def test_every_ref_shader_case_is_addressable(mm):
    from oracle import ref_shader
    for name in REF_SHADER_CASES:
        sc, u, p, ch = build_case(mm, name)
        assert ref_shader.addressable(u, p), name
    for name in ("cfg1", "cfg2_small", "bounce0"):          # other limits / shapes are beyond the unmodified shader
        sc, u, p, ch = build_case(mm, name)
        assert not ref_shader.addressable(u, p), name


def test_random_matches_reference_source(ref, oracle):
    O, L = oracle.lib(), ref.lib()
    rng = np.random.default_rng(3)
    for seed in [0, 1, 0xFFFFFFFF, 0x80000000, 291336453, 747796405] + [int(v) for v in rng.integers(0, 2 ** 32, 3000)]:
        a, b = C.c_uint32(seed), C.c_uint32(seed)
        for _ in range(4):
            ra, rb = L.ref_random(C.byref(a)), O.mmo_random(C.byref(b))
            assert _bits(ra) == _bits(rb) and a.value == b.value


SPECIALS = [0.0, -0.0, 1.0, -1.0, 1e-30, -1e-30, 1e-45, 1e30, -1e30, np.inf, -np.inf, np.nan, 0.1, 5.0, -5.0, 50.0]


def _vec3s(rng, n, scale, special_rate):
    v = (rng.standard_normal((n, 3)) * scale).astype(np.float32)
    mask = rng.random((n, 3)) < special_rate
    v[mask] = rng.choice(np.array(SPECIALS, dtype=np.float32), size=int(mask.sum()))
    return v


def test_intersect_aabb_matches_reference_source(ref, oracle):
    """shaders.metal:87-95 on random boxes and rays, a fifth of the components replaced by zeros, denormals, huge values,
    infinities and NaN (0/0, inf - inf, NaN-dropping min/max all occur)."""
    O, L = oracle.lib(), ref.lib()
    rng = np.random.default_rng(11)
    n = 20000
    ori, dirs = _vec3s(rng, n, 30.0, 0.1), _vec3s(rng, n, 1.0, 0.2)
    a, b = _vec3s(rng, n, 40.0, 0.05), _vec3s(rng, n, 40.0, 0.05)
    bmin, bmax = np.fmin(a, b), np.fmax(a, b)
    flat = rng.random(n) < 0.3                                 # zero-thickness boxes, as wall boxes are
    bmax[flat, 0] = bmin[flat, 0]
    ts = np.where(rng.random(n) < 0.5, np.float32(1e30), (rng.random(n) * 80).astype(np.float32)).astype(np.float32)
    for i in range(n):
        args = (ori[i].ctypes.data, dirs[i].ctypes.data, C.c_float(float(ts[i])), bmin[i].ctypes.data, bmax[i].ctypes.data)
        ra, rb = L.ref_intersect_aabb(*args), O.mmo_intersect_aabb(*args)
        assert _bits(ra) == _bits(rb) or (np.isnan(ra) and np.isnan(rb)), (i, ra, rb)


def test_ray_rect_matches_reference_source(ref, oracle, mm):
    """shaders.metal:51-67 on the planes of a maze (axis-aligned, some degenerate) and on random oblique rects."""
    from mirror_maze_b200.host import PLANE_DTYPE
    O, L = oracle.lib(), ref.lib()
    rng = np.random.default_rng(12)
    sc = mm.MazeScene(10, 0)
    obl = np.zeros(64, dtype=PLANE_DTYPE)
    obl["origin"] = rng.standard_normal((64, 3)) * 20
    obl["v"] = rng.standard_normal((64, 3)) * 10
    obl["u"] = rng.standard_normal((64, 3)) * 10
    obl["v"][:4] = 0.0                                          # zero-length edges: NaN normal, never hit
    planes = np.concatenate([sc.planes, obl])
    n = 20000
    ori, dirs = _vec3s(rng, n, 30.0, 0.05), _vec3s(rng, n, 1.0, 0.1)
    which = rng.integers(0, len(planes), n)
    # aim half of the rays at a point on their rect so that hits are common
    for i in range(0, n, 2):
        pl = planes[which[i]]
        target = pl["origin"] + pl["v"] * np.float32(rng.random()) + pl["u"] * np.float32(rng.random())
        d = (target - ori[i]).astype(np.float32)
        if np.isfinite(d).all() and 0 < np.abs(d).max() < 1e15:
            dirs[i] = d / np.float32(np.linalg.norm(d))
    hits = 0
    for i in range(n):
        pl = planes[which[i]:which[i] + 1]
        ta, tb = C.c_float(), C.c_float()
        t0 = C.c_float(1e30 if i % 3 else 25.0)
        ha = L.ref_ray_rect(ori[i].ctypes.data, dirs[i].ctypes.data, t0, pl.ctypes.data, C.byref(ta))
        hb = O.mmo_ray_rect(ori[i].ctypes.data, dirs[i].ctypes.data, t0, pl.ctypes.data, C.byref(tb))
        assert ha == hb and _bits(ta.value) == _bits(tb.value), (i, ha, hb, ta.value, tb.value)
        hits += ha
    assert hits > 2000


def test_quat_mult_matches_reference_source(ref, oracle):
    O, L = oracle.lib(), ref.lib()
    rng = np.random.default_rng(13)
    for _ in range(5000):
        v = rng.standard_normal(3).astype(np.float32)
        q = rng.standard_normal(4).astype(np.float32)
        q /= np.float32(np.linalg.norm(q))
        a, b = np.zeros(3, np.float32), np.zeros(3, np.float32)
        L.ref_quat_mult(v.ctypes.data, q.ctypes.data, a.ctypes.data)
        O.mmo_quat_mult(v.ctypes.data, q.ctypes.data, b.ctypes.data)
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("name", REF_SHADER_CASES)
def test_oracle_image_equals_reference_shader_image(oracle, mm, noise, scenes, name):
    """Whole dispatches: every written pixel of the reference shader's fp32 image, bit for bit.  Where the _ref library
    is absent, the oracle's image stands in for it and the digest of the reference shader's image, committed with the
    fixtures, is the comparison."""
    from oracle import ref_shader
    sc, u, p, ch = build_case(mm, name, scenes)
    got, cnt, _ = oracle.render(sc, noise, u, p, ch)
    want = ref_shader.render(sc, noise, u, p, ch) if ref_shader.available() else got
    assert (want[..., 3] == 1).sum() == cnt["paths"] // p.spp            # every pixel of every chunk was written
    assert got.tobytes() == want.tobytes()
    assert hashlib.sha256(want.tobytes()).hexdigest() == GOLDEN[name]["ref_shader_image"]


@pytest.mark.parametrize("name", REF_SHADER_CASES)
def test_oracle_image_equals_committed_reference_shader_digest(oracle, mm, noise, scenes, name):
    """The same pin without the _ref library: the digest of the reference shader's image, committed with the fixtures."""
    sc, u, p, ch = build_case(mm, name, scenes)
    got, _, _ = oracle.render(sc, noise, u, p, ch)
    assert hashlib.sha256(got.tobytes()).hexdigest() == GOLDEN[name]["ref_shader_image"]


def test_present_blur_matches_reference_fragment_shader(ref):
    """fragment_shader (shaders.metal:214-225), per pixel against the unblurred image, vs the ping-pong blur model that
    the CUDA present pass is tested against (SURVEY 8 f-1)."""
    from oracle import np_oracle
    L = ref.lib()
    L.ref_fragment_blur.restype = None
    L.ref_fragment_blur.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    rng = np.random.default_rng(21)
    for (H, W) in ((1, 1), (2, 3), (5, 7), (33, 65), (120, 160)):
        img = rng.random((H, W, 4), dtype=np.float32)
        out = np.zeros_like(img)
        L.ref_fragment_blur(img.ctypes.data, W, H, out.ctypes.data)
        assert out.tobytes() == np_oracle.present_blur(img).tobytes()


def test_seed_saturation_happens_in_these_cases(oracle):
    """The float -> uint conversion of the seed (shaders.metal:298) saturates for threads whose fp32 sum reaches 2^32;
    C++ leaves that cast undefined and x86 would wrap, so the shim's saturating conversion is exercised, not assumed."""
    O = oracle.lib()
    n = np.float32(128.0) / np.float32(255.0)
    sat = 0
    for ty in range(0, 768):
        for tx in (0, 511, 1023):
            s = (np.float32(n + n) + np.float32((tx * 15823) & 0xFFFFFFFF)) + np.float32((ty * 9737333) & 0xFFFFFFFF)
            if s >= np.float32(4294967296.0):
                sat += 1
                assert O.mmo_seed(C.c_float(float(n)), C.c_float(float(n)), tx, ty, 0) == 0xFFFFFFFF
    assert sat > 0


def test_random_dispatches_equal_reference_shader(ref, oracle, mm, noise):
    """Seeded random mazes, poses, times, chunk subsets and dispatch shapes (chunk 2/4/8, spp 8..64) among those the
    unmodified shader can address: oracle image vs reference-shader image, bit for bit."""
    rng = np.random.default_rng(77)
    done = 0
    for _ in range(16):
        maze = int(rng.choice([10, 16, 32]))
        chunk = int(rng.choice([2, 4, 8]))
        spp = int(rng.choice([s for s in (8, 16, 32, 64) if chunk * chunk * s <= 1024]))
        gx, gy = int(rng.choice([2, 4, 8])), int(rng.integers(1, 7))
        W, H = 2 * chunk * chunk * gx, int(rng.choice([32, 64, 96]))
        sc = mm.MazeScene(maze, 0)
        half = 5.0 * maze
        cell = rng.integers(0, maze, size=2)
        center = (-half + 10.0 * cell[0] + float(rng.uniform(0.5, 9.5)), float(rng.uniform(-7.5, 1.9)),
                  -half + 10.0 * cell[1] + float(rng.uniform(0.5, 9.5)))
        u = mm.default_uniform(maze, W, H, chunk, time=int(rng.integers(0, 100000)), camera_center=center,
                               half_theta=float(rng.uniform(0.0, np.pi)))
        allc = mm.gen_chunks(W, H, chunk)
        ch = allc[rng.permutation(len(allc))[: gx * gy]].copy()
        if len(ch) < gx * gy:
            continue
        p = mm.full_frame_params(u, spp=spp, bounce_limit=5, mirror_limit=15)
        p.grid_x, p.grid_y = gx, gy
        got, _, _ = oracle.render(sc, noise, u, p, ch)
        assert got.tobytes() == ref.render(sc, noise, u, p, ch).tobytes(), (maze, chunk, spp, gx, gy, center)
        done += 1
    assert done >= 10
