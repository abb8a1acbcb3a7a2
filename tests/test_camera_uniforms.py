"""The path start against the oracle for any camera and noise texel: pitch, roll, focal length, viewport, view size, texel bytes.

Every kernel begins a path in trace_device.cuh's start_at: the thread's pixel, the camera ray (shaders.metal:281-284, with
quat_mult / quat_dot), the noise texel (sample_noise_xy) and the seed (:298).  It reads every field of the 56-byte uniform and
texel (0,0) of the noise texture.  The other parity tests build their cameras with default_uniform, so rotation.x and
rotation.z are +0, the focal length is 1, the viewport is (2 W/H, 2), the view size is integral and texel (0,0) is the committed
(128, 128, 128, 255).  The classes here reach the rest:

- rotation: identity and its negation, pure pitch (exactly +-90 degrees with components RN(sqrt(1/2))), pure roll (90, and 180
  with w = +0 and -0), seeded unit quaternions with four non-zero components, a yaw with the signs of its zero components flipped,
  non-unit k * q and the zero quaternion;
- viewport and focal length: viewports unrelated to W / H, zero, negative, very wide and very narrow; focal lengths 0, -0, -1, 1e6;
- view size and centre: fractional view sizes, centres above the walls and below the floor looking in, a centre on a wall
  coordinate under a pitched camera, centre components at axis_safe's 2^-40 and 2^30 edges and their neighbours;
- non-finite: NaN in each of centre, rotation, viewport and focal length, and +-inf focal length (every path ends as a miss);
- noise texel (0,0): four distinct channels, bytes c whose c / 255 differs from c * RN(1/255), channel pairs whose fp32 sum
  R/255 + G/255 sits below, on or above 0.5, 1.0, 1.5 and 2.0 (where the seed's roundings tie), and textures of other sizes
  whose other texels are random (the output depends on texel (0,0) only).

Half the camera cases run at large `time` values, where the fraction of the seed sum decides its rounding.  Without a GPU, the
C++ oracle is compared with oracle/np_oracle.py on every class (and with the reference's own shader where its library is built),
and a numpy restatement of the path start counts that every claimed class is reached.  With a GPU, every class runs through every
kernel path, block shape, render_views and the 1024-thread shapes, each compared bit for bit with the oracle."""
import functools
import math

import numpy as np
import pytest

from test_general_scenes import scene as general_scene
from test_high_spp import assert_tail as assert_high_spp_tail
from test_ray_probe import axis_safe
from test_tail_and_shapes import COUNTER_KEYS, assert_same, assert_tail, gpu_render, with_flags

F = np.float32
U = np.uint32
NONE = 0xFFFFFFFF
SQRT_HALF = F(math.sqrt(0.5))                # RN(sqrt(1/2)): the components of a 90-degree turn


def up(x):
    return F(np.nextafter(F(x), F(np.inf)))


def down(x):
    return F(np.nextafter(F(x), F(-np.inf)))


def neg0():
    return F(-0.0)


# ---- quaternions -----------------------------------------------------------------------------------------------------------------

def axis_quat(axis, degrees):
    """Unit quaternion of a turn by `degrees` about axis 'x', 'y' or 'z', rounded to float32 per component."""
    h = math.radians(degrees) / 2.0
    q = [0.0, 0.0, 0.0, math.cos(h)]
    q["xyz".index(axis)] = math.sin(h)
    return tuple(F(c) for c in q)


def quat_mul(a, b):
    """Hamilton product in float64, rounded to float32 (used only to build test cameras)."""
    ax, ay, az, aw = (float(c) for c in a)
    bx, by, bz, bw = (float(c) for c in b)
    return (F(aw * bx + ax * bw + ay * bz - az * by), F(aw * by - ax * bz + ay * bw + az * bx),
            F(aw * bz + ax * by - ay * bx + az * bw), F(aw * bw - ax * bx - ay * by - az * bz))


def random_quats(n, seed=20261022):
    """Seeded unit quaternions (normalised in float64, rounded to float32) with all four components non-zero."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        q = rng.normal(size=4)
        q = q / np.linalg.norm(q)
        if np.abs(q).min() > 0.05:
            out.append(tuple(F(c) for c in q))
    return out


RANDOM_Q = random_quats(2)
YAW = axis_quat("y", 80.0)                    # (0, s, 0, c): the form default_uniform's yaw takes


# ---- camera classes --------------------------------------------------------------------------------------------------------------
# Each case overrides fields of the scene's base uniform: rot (x, y, z, w), vp(W, H) -> viewport, focal, center(base) -> centre,
# size {spp tier: (W, H)}, time.  Cases without a size render the tier's frame (FRAMES).

LARGE_TIMES = (8388609, 16777219, 2147483651, 4294967295)


def _cases():
    c = {}
    c["rot_identity"] = dict(cls="rotation", rot=(F(0), F(0), F(0), F(1)))
    c["rot_neg_identity"] = dict(cls="rotation", rot=(neg0(), neg0(), neg0(), F(-1)))
    c["rot_pitch_30"] = dict(cls="rotation", rot=axis_quat("x", 30.0))
    c["rot_pitch_up_90"] = dict(cls="rotation", rot=(SQRT_HALF, F(0), F(0), SQRT_HALF))
    c["rot_pitch_down_90"] = dict(cls="rotation", rot=(-SQRT_HALF, F(0), F(0), SQRT_HALF))
    c["rot_roll_90"] = dict(cls="rotation", rot=(F(0), F(0), SQRT_HALF, SQRT_HALF))
    c["rot_roll_180_pos_w"] = dict(cls="rotation", rot=(F(0), F(0), F(1), F(0)))
    c["rot_roll_180_neg_w"] = dict(cls="rotation", rot=(neg0(), neg0(), F(1), neg0()))
    for i, q in enumerate(RANDOM_Q):
        c[f"rot_random_{i}"] = dict(cls="rotation", rot=q)
    for name, (sx, sz) in {"mp": (neg0(), F(0)), "pm": (F(0), neg0()), "mm": (neg0(), neg0())}.items():
        c[f"rot_signed_zero_{name}"] = dict(cls="rotation", rot=(sx, YAW[1], sz, YAW[3]))
    for name, k in (("half", 0.5), ("two", 2.0), ("one_ulp2", 1.0 + 2.0 ** -22)):
        c[f"rot_scaled_{name}"] = dict(cls="rotation", rot=tuple(F(F(k) * q) for q in RANDOM_Q[0]))
    c["rot_zero"] = dict(cls="rotation", rot=(F(0), F(0), F(0), F(0)))
    c["vp_square"] = dict(cls="viewport", vp=lambda W, H: (2.0, 2.0))
    c["vp_swapped"] = dict(cls="viewport", vp=lambda W, H: (2.0, float(F(2.0) * (F(W) / F(H)))))
    c["vp_zero"] = dict(cls="viewport", vp=lambda W, H: (0.0, 0.0))
    c["vp_neg_x"] = dict(cls="viewport", vp=lambda W, H: (-float(F(2.0) * (F(W) / F(H))), 2.0))
    c["vp_neg_y"] = dict(cls="viewport", vp=lambda W, H: (float(F(2.0) * (F(W) / F(H))), -2.0))
    c["vp_neg_both"] = dict(cls="viewport", vp=lambda W, H: (-3.0, -1.25))
    c["vp_wide"] = dict(cls="viewport", vp=lambda W, H: (201.5, 2.0))
    c["vp_narrow"] = dict(cls="viewport", vp=lambda W, H: (1.0e-4, 7.5e-5))
    c["focal_zero"] = dict(cls="focal", focal=0.0)
    c["focal_neg_zero"] = dict(cls="focal", focal=-0.0)
    c["focal_neg_one"] = dict(cls="focal", focal=-1.0)
    c["focal_1e6"] = dict(cls="focal", focal=1.0e6)
    c["size_frac_a"] = dict(cls="view_size", size={1: (60.5, 44.25), 16: (60.5, 44.25), 64: (20.5, 12.25), 256: (9.75, 6.5), "cpu": (30.5, 18.25)})
    c["size_frac_b"] = dict(cls="view_size", size={1: (47.75, 31.5), 16: (47.75, 31.5), 64: (17.25, 10.75), 256: (8.5, 5.25), "cpu": (25.75, 17.5)},
                            vp=lambda W, H: (2.5, 1.5))
    c["centre_above"] = dict(cls="centre", center=lambda b: (b[0], b[1] + 12.0, b[2]), rot=quat_mul(YAW, axis_quat("x", -60.0)))
    c["centre_below"] = dict(cls="centre", center=lambda b: (b[0], b[1] - 30.0, b[2]), rot=quat_mul(YAW, axis_quat("x", 55.0)))
    c["centre_on_wall"] = dict(cls="centre", center=lambda b: (b[0] - 5.0, b[1], b[2] + 5.0), rot=quat_mul(YAW, axis_quat("x", -25.0)))
    for name, x in (("below", down(2.0 ** -40)), ("at", F(2.0 ** -40)), ("above", up(2.0 ** -40))):
        c[f"edge_tiny_x_{name}"] = dict(cls="edge", center=lambda b, x=x: (float(x), b[1], b[2]))
    for name, z in (("below", down(2.0 ** 30)), ("at", F(2.0 ** 30)), ("above", up(2.0 ** 30))):
        c[f"edge_huge_z_{name}"] = dict(cls="edge", center=lambda b, z=z: (b[0], b[1], -float(z)))
    nan = float("nan")
    c["nan_centre"] = dict(cls="nonfinite", center=lambda b: (nan, b[1], b[2]))
    c["nan_rotation"] = dict(cls="nonfinite", rot=(F(0), YAW[1], F(0), F(nan)))
    c["nan_viewport"] = dict(cls="nonfinite", vp=lambda W, H: (2.0, nan))
    c["nan_focal"] = dict(cls="nonfinite", focal=nan)
    c["inf_focal"] = dict(cls="nonfinite", focal=float("inf"))
    c["neg_inf_focal"] = dict(cls="nonfinite", focal=float("-inf"))
    for i, name in enumerate(c):
        c[name]["time"] = 7 if i % 2 == 0 else LARGE_TIMES[(i // 2) % len(LARGE_TIMES)]
    return c


CAMERAS = _cases()
CAMERA_NAMES = list(CAMERAS)
CLASSES = sorted({c["cls"] for c in CAMERAS.values()})

# spp tier -> (chunk, W, H): 64-thread blocks at spp 1, 16 and 64 (64, 4 and 1 pixels a block), 256-thread blocks at spp 256 (one
# pixel); HIGH_SPP below runs the 1024-thread blocks.  "cpu" is the frame of the tests without a GPU (spp 4).
FRAMES = {1: (4, 48, 32), 16: (4, 48, 32), 64: (2, 16, 12), 256: (1, 8, 6), "cpu": (4, 24, 16)}


def base_of(mm, scene_name):
    """(scene, base centre, base yaw) of a scene the GPU cases run on."""
    if scene_name.startswith("maze"):
        n = int(scene_name[4:])
        u = mm.default_uniform(n, 48, 32, 4)
        c = u.cam.camera_center
        return mm.MazeScene(n, 0), (c.x, c.y, c.z), 0.7
    sc = general_scene(mm, scene_name)
    return sc, sc.camera, sc.yaw


@functools.lru_cache(maxsize=None)
def _maze(n):
    import mirror_maze_b200 as mm
    return base_of(mm, f"maze{n}")


def scene_base(mm, scene_name):
    mm.load_library()
    if scene_name.startswith("maze"):
        return _maze(int(scene_name[4:]))
    return base_of(mm, scene_name)


def camera_uniform(mm, name, base, tier, chunk=None, W=None, H=None):
    """The uniform of camera case `name` over a scene base (scene, centre, yaw) at spp tier `tier`."""
    spec = CAMERAS[name]
    c, W0, H0 = FRAMES[tier]
    chunk = chunk or c
    if W is None:
        W, H = spec.get("size", {}).get(tier, (W0, H0))
    u = mm.default_uniform(10, W, H, chunk, spec["time"], camera_center=base[1], half_theta=base[2])
    if "rot" in spec:
        u.cam.rotation = mm.Float4(*[float(v) for v in spec["rot"]])
    if "vp" in spec:
        u.cam.viewport = mm.Float2(*spec["vp"](F(W), F(H)))
    if "focal" in spec:
        u.cam.focal_length = spec["focal"]
    if "center" in spec:
        u.cam.camera_center = mm.Float3(*spec["center"](base[1]))
    return u


def camera_dispatch(mm, name, base, tier, spp=None, bounce=6, flags=0):
    u = camera_uniform(mm, name, base, tier)
    ch = mm.gen_chunks(u.view_width, u.view_height, u.chunk_width)
    p = mm.full_frame_params(u, spp=spp or (4 if tier == "cpu" else tier), bounce_limit=bounce, mirror_limit=15, flags=flags)
    return u, p, ch


# ---- noise textures --------------------------------------------------------------------------------------------------------------

RECIP = F(1.0) / F(255.0)
RECIP_BYTES = [c for c in range(256) if F(c) / F(255.0) != F(c) * RECIP]   # the bytes where the divide and RN(1/255) * c differ


def unit(c):
    return F(c) / F(255.0)


def pair_sum(r, g):
    return unit(r) + unit(g)


def _noise_cases():
    """name -> (class, texel (0,0) as 4 bytes, texture size (w, h))."""
    out = {}
    for i, t in enumerate([(200, 30, 90, 250), (10, 240, 130, 0), (77, 180, 255, 1), (255, 0, 128, 64)]):
        out[f"channels_{i}"] = ("channels", t, None)
    # R + G = 255 with c * RN(1/255) summing above 1.0 (the divide gives exactly 1.0), and pairs of other such bytes
    tie_pairs = [(r, 255 - r) for r in RECIP_BYTES if F(r) * RECIP + F(255 - r) * RECIP != F(1.0)]
    for i, (r, g) in enumerate([tie_pairs[0], tie_pairs[len(tie_pairs) // 2], tie_pairs[-1]]):
        out[f"recip_tie_{i}"] = ("recip", (r, g, 255 - r, 17), None)
    for i, (r, g) in enumerate([(RECIP_BYTES[3], RECIP_BYTES[40]), (RECIP_BYTES[77], RECIP_BYTES[101]), (RECIP_BYTES[125], RECIP_BYTES[0])]):
        out[f"recip_other_{i}"] = ("recip", (r, g, 9, 200), None)
    # R + G just below, on and just above 0.5, 1.0, 1.5 and 2.0 (0.5 and 1.5 are not sums of two bytes / 255)
    sums = {"0.5_below": [(127, 0), (60, 67)], "0.5_above": [(128, 0), (1, 127)],
            "1.0_below": [(254, 0), (127, 127), (100, 154)], "1.0_on": [(255, 0), (128, 127), (3, 252)],
            "1.0_above": [(1, 255), (128, 128), (200, 56)], "1.5_below": [(255, 127), (191, 191)], "1.5_above": [(255, 128), (192, 191)],
            "2.0_below": [(254, 255), (255, 254)], "2.0_on": [(255, 255)]}
    for k, pairs in sums.items():
        for i, (r, g) in enumerate(pairs):
            out[f"sum_{k}_{i}"] = ("sums", (r, g, 255 - g, 255), None)
    for w, h in ((1, 1), (1, 7), (3, 5), (512, 1), (1024, 1024)):
        out[f"size_{w}x{h}"] = ("size", None, (w, h))
    return out


NOISE = _noise_cases()
NOISE_NAMES = list(NOISE)


@functools.lru_cache(maxsize=None)
def _texture(name, committed_bytes):
    cls, texel, size = NOISE[name]
    committed = np.frombuffer(committed_bytes, np.uint8).reshape(512, 512, 4)
    if cls == "size":
        w, h = size
        rng = np.random.default_rng([w, h])
        t = rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8)
        t[0, 0] = committed[0, 0]
    else:
        t = committed.copy()
        t[0, 0] = texel
    t.setflags(write=False)
    return t


def texture(noise, name):
    return _texture(name, noise.tobytes())


# ---- the path start, restated -----------------------------------------------------------------------------------------------------

def path_start(u, p, chunks, noise, divide=True, ny_channel=1):
    """np_oracle._render up to the jitter (shaders.metal:261-303), vectorised over every path of the dispatch: returns the ray
    before rotation, after rotation and after the jitter, the seed, the texel coordinates and the texid.  divide = False and
    ny_channel restate two wrong readings of the texel (c * RN(1/255), another channel for ny) to count where they would differ."""
    from oracle.np_oracle import _f2u_sat, _normalize, _random, _dot, _cross

    W, H = F(u.view_width), F(u.view_height)
    chunk = int(u.chunk_width)
    ppc, spp = chunk * chunk, int(p.spp)
    T = ppc * spp
    dimx = min(32, T)
    dimy = T // dimx
    first, step, count = p.group_first, (p.group_step or 1), p.group_count
    if count == 0:
        first, step, count = 0, 1, p.grid_x * p.grid_y
    k = np.repeat(np.arange(count, dtype=np.int64), T)
    flat = np.tile(np.arange(T, dtype=np.int64), count)
    g = first + k * step
    tgx, tgy = g % p.grid_x, g // p.grid_x
    gx, gy = flat % dimx, flat // dimx
    ch = np.asarray(chunks)[g]
    pn = flat // spp
    px = ch["x"].astype(np.int64) + pn // chunk
    py = ch["y"].astype(np.int64) + pn % chunk
    texx, texy = (tgx * dimx + gx).astype(U), (tgy * dimy + gy).astype(U)
    n = len(flat)
    cam = u.cam
    with np.errstate(all="ignore"):
        center = [F(cam.camera_center.x), F(cam.camera_center.y), F(cam.camera_center.z)]
        vpx, vpy, focal = F(cam.viewport.x), F(cam.viewport.y), F(cam.focal_length)
        pnx, pny = px.astype(U).astype(F) / W, py.astype(U).astype(F) / H
        corner = [center[0] - vpx / F(2.0), center[1] - vpy / F(2.0), center[2] - (-focal)]
        pre = [(corner[0] + pnx * vpx) - center[0], (corner[1] + pny * vpy) - center[1],
               np.full(n, (corner[2] + F(0.0)) - center[2], dtype=F)]
        rd = _normalize(pre)
        q = [F(cam.rotation.x), F(cam.rotation.y), F(cam.rotation.z), F(cam.rotation.w)]

        def quat_dot(q1, q2):
            s = q1[3] * q2[3] - _dot(q1[:3], q2[:3])
            c = _cross(q1[:3], q2[:3])
            return [(c[i] + q1[3] * q2[i]) + q2[3] * q1[i] for i in range(3)] + [s]

        r = quat_dot(quat_dot([-q[0], -q[1], -q[2], q[3]], rd + [np.zeros(n, F)]), q)
        rot = [np.asarray(r[i], dtype=F) * np.ones(n, F) for i in range(3)]
        nh, nw = noise.shape[:2]
        uu, vv = gx.astype(F), gy.astype(F)
        ix = np.clip(np.floor((uu - np.floor(uu)) * F(nw)).astype(np.int64), 0, nw - 1)
        iy = np.clip(np.floor((vv - np.floor(vv)) * F(nh)).astype(np.int64), 0, nh - 1)
        tex = noise[iy, ix].astype(F)
        nx = tex[:, 0] / F(255.0) if divide else tex[:, 0] * RECIP
        ny = tex[:, ny_channel] / F(255.0) if divide else tex[:, ny_channel] * RECIP
        seed_f = (((nx + ny) + (texx * U(15823)).astype(F)) + (texy * U(9737333)).astype(F)) + F(u.time)
        seed = _f2u_sat(seed_f)
        st, r1 = _random(seed)
        st, r2 = _random(st)
        d = [rot[0] + ((r1 - F(0.5)) * F(2.0)) * F(0.001), rot[1] + ((r2 - F(0.5)) * F(2.0)) * F(0.001), rot[2] + F(0.0) * F(0.001)]
    return dict(pre=np.stack(pre, 1).astype(F), rot=np.stack(rot, 1), dir=np.stack(d, 1).astype(F),
                ori=np.tile(np.array(center, F), (n, 1)), seed=seed, ix=ix, iy=iy, texx=texx, texy=texy)


def literal_lanes(ps):
    """Primary rays the kernel traces with the literal-divide slab form (axis_safe fails on some axis)."""
    with np.errstate(invalid="ignore"):
        return ~axis_safe(ps["ori"], ps["dir"]).all(axis=1)


# ---- without a GPU -----------------------------------------------------------------------------------------------------------------

def test_camera_cases_are_what_they_claim(mm):
    """The rotation, viewport, focal and centre cases carry the values their names claim, bit for bit where it matters."""
    assert CLASSES == ["centre", "edge", "focal", "nonfinite", "rotation", "view_size", "viewport"]
    b = scene_base(mm, "maze10")
    got = {n: camera_uniform(mm, n, b, 16) for n in CAMERA_NAMES}

    def rot(n):
        r = got[n].cam.rotation
        return np.array([r.x, r.y, r.z, r.w], F)

    def sign_bits(v):
        return tuple(int(x) for x in np.signbit(v))

    assert rot("rot_identity").tobytes() == np.array([0, 0, 0, 1], F).tobytes()
    assert sign_bits(rot("rot_neg_identity")) == (1, 1, 1, 1) and (rot("rot_neg_identity")[:3] == 0).all()
    assert rot("rot_pitch_up_90").tolist() == [SQRT_HALF, 0, 0, SQRT_HALF] and SQRT_HALF == F(0.70710677)
    assert rot("rot_pitch_down_90")[0] == -SQRT_HALF
    assert sign_bits(rot("rot_roll_180_pos_w"))[3] == 0 and sign_bits(rot("rot_roll_180_neg_w"))[3] == 1
    assert rot("rot_roll_180_neg_w")[3] == 0
    for n in ("rot_random_0", "rot_random_1", "centre_above", "centre_below", "centre_on_wall"):
        assert (rot(n) != 0).all(), n
    for n, bits in (("mp", (1, 0)), ("pm", (0, 1)), ("mm", (1, 1))):
        r = rot(f"rot_signed_zero_{n}")
        assert r[0] == 0 and r[2] == 0 and (sign_bits(r)[0], sign_bits(r)[2]) == bits and r[1] != 0 and r[3] != 0
    norms = {n: float(np.linalg.norm(rot(n).astype(np.float64))) for n in ("rot_scaled_half", "rot_scaled_two", "rot_scaled_one_ulp2")}
    assert abs(norms["rot_scaled_half"] - 0.5) < 1e-6 and abs(norms["rot_scaled_two"] - 2.0) < 1e-6
    assert 1.0 < norms["rot_scaled_one_ulp2"] < 1.0 + 1e-6 and (rot("rot_scaled_one_ulp2") != rot("rot_random_0")).all()
    assert (rot("rot_zero") == 0).all()
    default_vp = (F(2.0) * (F(48) / F(32)), F(2.0))
    for n in ("vp_square", "vp_swapped", "vp_zero", "vp_neg_x", "vp_neg_y", "vp_neg_both", "vp_wide", "vp_narrow", "size_frac_b"):
        v = got[n].cam.viewport
        assert (F(v.x), F(v.y)) != default_vp, n
    assert got["vp_zero"].cam.viewport.x == 0 and got["vp_wide"].cam.viewport.x > 200 and got["vp_narrow"].cam.viewport.x < 2e-4
    assert min(got[n].cam.viewport.x for n in ("vp_neg_x", "vp_neg_both")) < 0 and got["vp_neg_y"].cam.viewport.y < 0
    assert [got[n].cam.focal_length for n in ("focal_zero", "focal_neg_one", "focal_1e6")] == [0.0, -1.0, 1e6]
    assert math.copysign(1.0, got["focal_neg_zero"].cam.focal_length) == -1.0
    for n in ("size_frac_a", "size_frac_b"):
        for tier in (1, 16, 64, 256, "cpu"):
            W, H = CAMERAS[n]["size"][tier]
            assert W != int(W) and H != int(H)
    c = got["centre_on_wall"].cam.camera_center
    assert c.x % 10 == 0 and c.z % 10 == 0
    assert got["centre_above"].cam.camera_center.y > float(mm.MazeScene(10, 0).nodes[0]["aabb_max"][1])
    assert got["centre_below"].cam.camera_center.y < float(mm.MazeScene(10, 0).nodes[0]["aabb_min"][1])
    xs = [F(got[f"edge_tiny_x_{k}"].cam.camera_center.x) for k in ("below", "at", "above")]
    assert xs == [down(2.0 ** -40), F(2.0 ** -40), up(2.0 ** -40)]
    zs = [F(-got[f"edge_huge_z_{k}"].cam.camera_center.z) for k in ("below", "at", "above")]
    assert zs == [down(2.0 ** 30), F(2.0 ** 30), up(2.0 ** 30)]
    assert sum(CAMERAS[n]["time"] >= 1 << 23 for n in CAMERA_NAMES) >= len(CAMERA_NAMES) // 2 - 1


def test_path_start_reaches_every_camera_class(mm, noise):
    """Over the camera cases on the 10x10 maze at the CPU frame (chunk 4, spp 4), the restated path start reaches: rotated
    directions with a component exactly +0 and exactly -0; warps (32 consecutive paths) that mix axis_safe and literal primary
    rays; primary rays whose largest component is y, with both signs; pre-rotation dir.z exactly 0 at focal length 0; the
    centre's axis_safe edges on both sides; and NaN on every path of the non-finite cases (and only there)."""
    b = scene_base(mm, "maze10")
    pos0 = neg0_ = mixed = y_up = y_down = 0
    for n in CAMERA_NAMES:
        u, p, ch = camera_dispatch(mm, n, b, "cpu")
        ps = path_start(u, p, ch, noise)
        rot, d = ps["rot"], ps["dir"]
        pos0 += int(((rot == 0) & ~np.signbit(rot)).sum())
        neg0_ += int(((rot == 0) & np.signbit(rot)).sum())
        lit = literal_lanes(ps)
        w = lit[: len(lit) // 32 * 32].reshape(-1, 32)
        mixed += int((w.any(axis=1) & ~w.all(axis=1)).sum())
        with np.errstate(invalid="ignore"):
            ydom = (np.abs(d[:, 1]) > np.abs(d[:, 0])) & (np.abs(d[:, 1]) > np.abs(d[:, 2]))
        y_up += int((ydom & (d[:, 1] > 0)).sum())
        y_down += int((ydom & (d[:, 1] < 0)).sum())
        spec = CAMERAS[n]
        if spec["cls"] == "nonfinite":
            assert np.isnan(d).any(axis=1).all(), n
        else:
            assert not np.isnan(d).any(axis=1).all(), n
        if n in ("focal_zero", "focal_neg_zero"):
            assert (ps["pre"][:, 2] == 0).all() and not np.signbit(ps["pre"][:, 2]).any(), n
        if n == "edge_tiny_x_below":
            assert lit.all(), n                                   # |x| < 2^-40: every primary ray is literal
        if n in ("edge_tiny_x_at", "edge_tiny_x_above", "edge_huge_z_below", "edge_huge_z_at"):
            assert not lit.all(), n
        if n == "edge_huge_z_above":
            assert lit.all(), n
    assert pos0 > 0 and neg0_ > 0, (pos0, neg0_)
    assert mixed > 0
    assert y_up > 0 and y_down > 0, (y_up, y_down)


def test_texture_cases_are_what_they_claim(noise):
    """Channels distinct; the reciprocal bytes and tie pairs; the pair sums on their sides of 0.5, 1.0, 1.5 and 2.0; the size
    class's other texels random and texel (0,0) the committed one."""
    assert len(RECIP_BYTES) == 126 and 128 not in RECIP_BYTES
    assert tuple(noise[0, 0]) == (128, 128, 128, 255)
    for name, (cls, texel, size) in NOISE.items():
        t = texture(noise, name)
        r, g = int(t[0, 0, 0]), int(t[0, 0, 1])
        if cls == "channels":
            assert len(set(texel)) == 4
        elif cls == "recip":
            assert r in RECIP_BYTES and (g in RECIP_BYTES or "tie" in name)
            if "tie" in name:
                assert r + g == 255 and pair_sum(r, g) == F(1.0) and F(r) * RECIP + F(g) * RECIP > F(1.0)
        elif cls == "sums":
            target = F(name.split("_")[1])
            side = name.split("_")[2]
            s = pair_sum(r, g)
            assert {"below": s < target, "on": s == target, "above": s > target}[side], (name, s)
            assert abs(float(s) - float(target)) < 0.005
        else:
            w, h = size
            assert t.shape == (h, w, 4) and tuple(t[0, 0]) == (128, 128, 128, 255)
            if w * h > 1:
                assert (t.reshape(-1, 4)[1:] != t[0, 0]).any(axis=1).mean() > 0.9
    assert len(NOISE) >= 30


NOISE_TIMES = (0, 16777220)        # time 2^24 + 4: s + time rounds to even at the ties of R/255 + G/255 = 1.0


def noise_dispatch(mm, time, W=24, H=16, spp=4):
    u = mm.default_uniform(10, W, H, 4, time)
    return u, mm.full_frame_params(u, spp=spp, bounce_limit=5), mm.gen_chunks(W, H, 4)


def test_path_start_reaches_every_noise_class(mm, noise):
    """Per texture, at the CPU frame and both NOISE_TIMES: only texel (0,0) is sampled; every channel texel's seeds change when ny
    is read from another channel; every reciprocal tie texel's seeds change under c * RN(1/255); the pair sums straddle the seed's
    rounding boundaries (some seed changes against the texel one step down) for a third of them at least; the size class gives the
    committed seeds."""
    committed = {t: path_start(*noise_dispatch(mm, t), noise)["seed"] for t in NOISE_TIMES}
    reached = {"channels": 0, "recip": 0, "sums": 0, "size": 0}
    for name, (cls, texel, size) in NOISE.items():
        tex = texture(noise, name)
        for t in NOISE_TIMES:
            args = noise_dispatch(mm, t)
            ps = path_start(*args, tex)
            assert (ps["ix"] == 0).all() and (ps["iy"] == 0).all()
            if cls == "channels":
                other = [path_start(*args, tex, ny_channel=c)["seed"] for c in (0, 2, 3)]
                reached[cls] += all((o != ps["seed"]).any() for o in other)
            elif cls == "recip":
                reached[cls] += bool((path_start(*args, tex, divide=False)["seed"] != ps["seed"]).any())
            elif cls == "sums":
                r, g = int(tex[0, 0, 0]), int(tex[0, 0, 1])
                nb = tex.copy()
                nb[0, 0, :2] = (r - 1, g) if r > 0 else (r, g - 1)        # one step down
                reached[cls] += bool((path_start(*args, nb)["seed"] != ps["seed"]).any())
            else:
                reached[cls] += bool((ps["seed"] == committed[t]).all())
    n = {c: sum(1 for v in NOISE.values() if v[0] == c) * len(NOISE_TIMES) for c in reached}
    assert reached["channels"] == n["channels"] and reached["size"] == n["size"], reached
    ties = sum(k.startswith("recip_tie") for k in NOISE)
    assert reached["recip"] >= ties * len(NOISE_TIMES) and reached["sums"] >= n["sums"] // 3, reached


def np_render(mm, sc, noise, u, p, ch):
    from oracle import np_oracle

    img, cnt, dbg = np_oracle.render(sc, noise, u, p, ch)
    if p.flags & mm.FLAG_SCREEN_RGBA8:
        img = np_oracle.quant8(img)
    return img, cnt, {k: np.ascontiguousarray(v, dtype=U if k != "radiance" else F) for k, v in dbg.items()}


CPU_SCENES = ["maze10", "tilted_0"]


@pytest.mark.parametrize("name", CAMERA_NAMES)
@pytest.mark.parametrize("scene_name", CPU_SCENES)
def test_oracle_matches_numpy_transcription_on_camera(mm, oracle, noise, scene_name, name):
    """The C++ oracle against oracle/np_oracle.py, two independent transcriptions, on every camera case: per-path arrays, image and
    counters, bit for bit."""
    b = scene_base(mm, scene_name)
    u, p, ch = camera_dispatch(mm, name, b, "cpu")
    ref = oracle.render(b[0], noise, u, p, ch, debug=True)
    assert_same(ref, np_render(mm, b[0], noise, u, p, ch), f"{scene_name} {name}")
    if CAMERAS[name]["cls"] == "nonfinite":
        assert (ref[2]["first_hit"] == NONE).all() and (ref[2]["segments"] == 1).all(), name


@pytest.mark.parametrize("name", NOISE_NAMES)
def test_oracle_matches_numpy_transcription_on_noise(mm, oracle, noise, scenes, name):
    """The same on every texture, at both NOISE_TIMES; and against the committed texture: a texture whose restated seeds equal
    the committed texture's renders the committed image (the size class always does)."""
    sc = scenes(10)
    tex = texture(noise, name)
    for t in NOISE_TIMES:
        u, p, ch = noise_dispatch(mm, t)
        ref = oracle.render(sc, tex, u, p, ch, debug=True)
        assert_same(ref, np_render(mm, sc, tex, u, p, ch), f"{name} time {t}")
        same_seeds = (path_start(u, p, ch, tex)["seed"] == path_start(u, p, ch, noise)["seed"]).all()
        base = oracle.render(sc, noise, u, p, ch)[0]
        if same_seeds:
            assert ref[0].tobytes() == base.tobytes(), name
        if NOISE[name][0] == "size":
            assert same_seeds, name


def test_every_texel_class_but_size_changes_the_image(mm, oracle, noise, scenes):
    """Every noise class except the size class changes the oracle image against the committed texture (at the CPU frame, at
    one of NOISE_TIMES) for most of its textures; the size class leaves it unchanged."""
    sc = scenes(10)
    changed = {}
    for t in NOISE_TIMES:
        u, p, ch = noise_dispatch(mm, t)
        base = oracle.render(sc, noise, u, p, ch)[0]
        for name, (cls, _, _) in NOISE.items():
            img = oracle.render(sc, texture(noise, name), u, p, ch)[0]
            changed[name] = changed.get(name, False) or img.tobytes() != base.tobytes()
    for cls in ("channels", "recip", "sums", "size"):
        names = [n for n in NOISE if NOISE[n][0] == cls]
        k = sum(changed[n] for n in names)
        if cls == "size":
            assert k == 0
        else:
            assert k >= (len(names) + 1) // 2, (cls, [n for n in names if not changed[n]])


REF_SHADER_CAMERAS = ["rot_neg_identity", "rot_pitch_down_90", "rot_roll_180_neg_w", "rot_random_0", "rot_signed_zero_mp",
                      "rot_scaled_two", "rot_zero", "vp_swapped", "vp_neg_both", "vp_narrow", "focal_zero", "focal_neg_one",
                      "size_frac_b", "centre_above", "edge_tiny_x_below", "nan_focal"]


def test_oracle_equals_reference_shader_on_camera_and_noise(mm, oracle, noise, scenes):
    """Where the reference's own shader is built (oracle/_ref/libref_shader.so): the oracle's image against it on dispatches it
    can address (limits 5 / 15, spp 8, grid_x = (W / 2) / chunk^2), for camera cases and for one texture of each noise class."""
    from oracle import ref_shader

    if not ref_shader.available():
        pytest.skip("oracle/_ref/libref_shader.so not built (needs the reference's source)")
    b = scene_base(mm, "maze10")
    jobs = [(n, None) for n in REF_SHADER_CAMERAS] + [("rot_random_1", k) for k in ("channels_0", "recip_tie_0", "sum_1.0_on_1",
                                                                                     "sum_0.5_above_1", "size_3x5")]
    for cam, tex_name in jobs:
        spec_size = CAMERAS[cam].get("size", {}).get(16)
        W, H = spec_size if spec_size else (64.0, 32.0)
        u = camera_uniform(mm, cam, b, 16, chunk=4, W=W, H=H)
        tex = noise if tex_name is None else texture(noise, tex_name)
        p = mm.full_frame_params(u, spp=8, bounce_limit=5, mirror_limit=15)
        allc = mm.gen_chunks(u.view_width, u.view_height, 4)
        gx = int((F(u.view_width) / F(2.0)) / F(16))
        gy = len(allc) // gx
        p.grid_x, p.grid_y = gx, gy
        ch = allc[np.random.default_rng(5).permutation(len(allc))[: gx * gy]].copy()
        assert ref_shader.addressable(u, p), cam
        got = oracle.render(b[0], tex, u, p, ch)[0]
        assert got.tobytes() == ref_shader.render(b[0], tex, u, p, ch).tobytes(), (cam, tex_name)


# ---- on the GPU ----------------------------------------------------------------------------------------------------------------------

GPU_SCENES = ["maze10", "maze16", "tilted_0"]
VARIANTS = [0, "FLAG_NO_Y_TABLE", "FLAG_NO_TAIL", "FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_RCP_SLAB", "FLAG_COUNTERS",
            "FLAG_SCREEN_RGBA8", "FLAG_REGROUP", "FLAG_POOL_KERNEL"]


def rgba8_ref(ref):
    from oracle import np_oracle

    return np_oracle.quant8(ref[0]), ref[1], ref[2]


def check_plain_counters(mm, cnt, ref_cnt, flags, what):
    """A render without per-path arrays runs the kernels callers run: under FLAG_COUNTERS the counting instantiation, which
    must give every counter of the reference; otherwise the plain one, which counts paths, rays and hits only.  (The debug
    kernels count everything, so callers pass FLAG_COUNTERS for them.)"""
    if flags & mm.FLAG_COUNTERS:
        for k in COUNTER_KEYS:
            assert cnt[k] == ref_cnt[k], f"counter {k}: {cnt[k]} != {ref_cnt[k]}: {what}"
    else:
        assert cnt["inner_visits"] == 0 and cnt["rect_tests"] == 0, f"a counting kernel ran: {cnt}: {what}"


def check_variant(mm, renderer, u, q, ch, ref, what, tail=assert_tail):
    """Renders with the per-path arrays (the debug kernels) and without them (the kernels callers and bench.py run); image,
    counters and tail against ref in both, the per-path arrays in the first."""
    for debug in (True, False):
        w = f"{what} debug {debug}"
        g = gpu_render(mm, renderer, u, q, ch, debug)
        assert_same(g, ref if debug else (ref[0], ref[1], None), w)
        if not debug:
            check_plain_counters(mm, g[1], ref[1], q.flags, w)
        if tail is assert_tail:
            assert_tail(mm, renderer, g[3], q, ref[2]["segments"], w)
        else:
            tail(mm, g[3], q, ref[2]["segments"], w)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CAMERA_NAMES)
@pytest.mark.parametrize("scene_name", GPU_SCENES)
def test_camera_through_every_kernel_matches_oracle(mm, oracle, noise, renderer, scene_name, name):
    """One camera case on one scene: at spp 16 every kernel path (y-table, no y-table, no tail, literal, general rects, RCP slab
    against the oracle in RCP mode, counters, RGBA8 screen, regroup, pool); at spp 1, 64 and 256 (every block shape) the default
    kernel, no y-table and (spp <= 64) the pool.  Each runs with and without per-path arrays.  Each oracle render finishes before
    its uniform goes to the GPU."""
    b = scene_base(mm, scene_name)
    sc = b[0]
    u, p, ch = camera_dispatch(mm, name, b, 16)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    rcp = oracle.render(sc, noise, u, with_flags(mm, p, mm.FLAG_RCP_SLAB), ch, debug=True)
    tiers = {}
    for spp in (1, 64, 256):
        tu, tp, tch = camera_dispatch(mm, name, b, spp)
        tiers[spp] = (tu, tp, tch, oracle.render(sc, noise, tu, tp, tch, debug=True))
    if CAMERAS[name]["cls"] == "nonfinite":
        for r in [ref] + [t[3] for t in tiers.values()]:
            assert (r[2]["first_hit"] == NONE).all() and (r[2]["segments"] == 1).all(), name
    renderer.upload_scene(sc, noise)
    for v in VARIANTS:
        flag = getattr(mm, v) if v else 0
        q = with_flags(mm, p, flag)
        want = rcp if flag == mm.FLAG_RCP_SLAB else rgba8_ref(ref) if flag == mm.FLAG_SCREEN_RGBA8 else ref
        check_variant(mm, renderer, u, q, ch, want, f"{scene_name} {name} spp 16 {v or 'default'}")
    for spp, (tu, tp, tch, tref) in tiers.items():
        for v in ["default", "FLAG_NO_Y_TABLE"] + (["FLAG_POOL_KERNEL"] if spp <= 64 else []):
            q = with_flags(mm, tp, 0 if v == "default" else getattr(mm, v))
            check_variant(mm, renderer, tu, q, tch, tref, f"{scene_name} {name} spp {spp} {v}")


# One view of every camera class in one launch, on a fractional frame (the view_size class is the launch's own W x H)
VIEW_CAMERAS = ["rot_random_1", "vp_swapped", "focal_zero", "size_frac_b", "centre_above", "centre_below", "edge_tiny_x_below",
                "nan_rotation"]
VIEW_FRAME = CAMERAS["size_frac_b"]["size"][16]


def split_views(dbg, n_views):
    n = len(dbg["segments"]) // n_views
    return [{k: dbg[k][v * n:(v + 1) * n] for k in dbg} for v in range(n_views)]


def check_views(mm, r, us, p, lists, refs, what):
    """render_views with per-path arrays, with FLAG_COUNTERS and without: every view's image (and arrays) against its reference,
    the launch's counters against the sum of the views'."""
    W, H = int(us[0].view_width), int(us[0].view_height)
    for debug, flags in ((True, 0), (False, mm.FLAG_COUNTERS), (False, 0)):
        q = with_flags(mm, p, flags)
        w = f"{what} debug {debug} flags {flags}"
        outs = [np.zeros((H, W, 4), F) for _ in us]
        _, cnt, dbg = r.render_views(us, q, lists, outs=outs, debug=debug)
        per_view = split_views(dbg, len(us)) if debug else [None] * len(us)
        for v, ref in enumerate(refs):
            assert_same((outs[v], ref[1], per_view[v]), ref if debug else (ref[0], ref[1], None), f"{w} view {v}")
        summed = {k: sum(rf[1][k] for rf in refs) for k in COUNTER_KEYS if k != "max_stack"}
        summed["max_stack"] = max(rf[1]["max_stack"] for rf in refs)
        for k in ("paths", "rays", "hits"):
            assert cnt[k] == summed[k], f"counter {k}: {w}"
        check_plain_counters(mm, cnt, summed, flags | (mm.FLAG_COUNTERS if debug else 0), w)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", GPU_SCENES)
def test_views_of_every_camera_class_in_one_launch(mm, oracle, noise, scene_name):
    """One render_views launch of eight views, one of every camera class (two of the centre class), on a shared fractional frame
    and chunk width with their own times: with and without per-path arrays and counters, every view equals the oracle, and each
    equals a lone mm_render of it on one other context."""
    b = scene_base(mm, scene_name)
    sc = b[0]
    assert {CAMERAS[n]["cls"] for n in VIEW_CAMERAS} == set(CLASSES)
    us = [camera_uniform(mm, n, b, 16, W=VIEW_FRAME[0], H=VIEW_FRAME[1]) for n in VIEW_CAMERAS]
    p = mm.full_frame_params(us[0], spp=16, bounce_limit=6, mirror_limit=15)
    base = mm.gen_chunks(us[0].view_width, us[0].view_height, 4)
    lists = [base[np.random.default_rng(40 + v).permutation(len(base))].copy() for v in range(len(us))]
    refs = [oracle.render(sc, noise, us[v], p, lists[v], debug=True) for v in range(len(us))]
    r = mm.Renderer(0)
    try:
        r.upload_scene(sc, noise)
        check_views(mm, r, us, p, lists, refs, scene_name)
    finally:
        r.close()
    lone = mm.Renderer(0)
    try:
        lone.upload_scene(sc, noise)
        for v, name in enumerate(VIEW_CAMERAS):
            assert_same(lone.render(us[v], p, lists[v], debug=True), refs[v], f"{scene_name} lone {name}")
    finally:
        lone.close()


HIGH_SPP_CAMERAS = ["rot_random_0", "rot_pitch_up_90", "vp_neg_both", "focal_neg_one", "centre_below"]
HIGH_SPP = {512: (4, 3), 1024: (3, 2)}        # chunk 1: the reference's one-pixel threadgroups


@pytest.mark.gpu
@pytest.mark.parametrize("spp", sorted(HIGH_SPP))
@pytest.mark.parametrize("name", HIGH_SPP_CAMERAS)
def test_camera_at_1024_thread_blocks_matches_transcription(mm, noise, renderer, name, spp):
    """spp 512 and 1024 at chunk 1 on the 32x32 maze, against oracle/np_oracle.py (the C++ oracle stops at spp 256): default
    kernel, no y-table, the literal form and counters, with and without per-path arrays, every observable and the tail."""
    b = scene_base(mm, "maze32")
    sc = b[0]
    W, H = HIGH_SPP[spp]
    u = camera_uniform(mm, name, b, 256, chunk=1, W=W, H=H)
    ch = mm.gen_chunks(W, H, 1)
    p = mm.full_frame_params(u, spp=spp, bounce_limit=8, mirror_limit=15)
    ref = np_render(mm, sc, noise, u, p, ch)
    renderer.upload_scene(sc, noise)
    for v in (0, mm.FLAG_NO_Y_TABLE, mm.FLAG_FORCE_LITERAL, mm.FLAG_COUNTERS):
        check_variant(mm, renderer, u, with_flags(mm, p, v), ch, ref, f"{name} spp {spp} flags {v}", tail=assert_high_spp_tail)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NOISE_NAMES)
def test_texture_through_the_kernels_matches_oracle(mm, oracle, noise, name):
    """One upload per texture: the default kernel and no y-table at both NOISE_TIMES, and both times as two views of one
    render_views launch, each with and without per-path arrays, against the oracle on the same texture (48 x 32, spp 16: texid_y
    reaches 3 with texid_x = 0)."""
    sc = mm.MazeScene(10, 0)
    tex = texture(noise, name)
    cases = [noise_dispatch(mm, t, W=48, H=32, spp=16) for t in NOISE_TIMES]
    refs = [oracle.render(sc, tex, u, p, ch, debug=True) for u, p, ch in cases]
    r = mm.Renderer(0)
    try:
        r.upload_scene(sc, tex)
        for (u, p, ch), ref in zip(cases, refs):
            for v in (0, mm.FLAG_NO_Y_TABLE):
                check_variant(mm, r, u, with_flags(mm, p, v), ch, ref, f"{name} time {u.time} flags {v}")
        check_views(mm, r, [c[0] for c in cases], cases[0][1], [cases[0][2]] * len(cases), refs, name)
    finally:
        r.close()
