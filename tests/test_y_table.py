"""The y-table traversal (trace_ytab_kernel, trace_tail_kernel<..., true>; DESIGN.md §3-4): a ray's y slab quotients of the
scene's few distinct child y-intervals are computed once per traversal call, and every interior visit reads them from a
per-lane shared-memory table.  Frames, counters and per-path observables are the same bits as trace_kernel's
(MM_FLAG_NO_Y_TABLE) and the oracle's, on every parity case, block shape, tail setting, rect form and delivery route, and
for scenes at the table's cap of 8 intervals and one past it."""
import os
import types

import numpy as np
import pytest

from cases import CASES, build_case
from test_tail_and_shapes import assert_same, assert_tail, gpu_render, with_flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_Y_INTERVALS = 8                  # render_kernel.cuh: kMaxYIntervals


def y_intervals(nodes):
    """The distinct (min.y, max.y) bit patterns of the children of reachable interior nodes (scene_prep.cpp, PairRecY)."""
    reach, stack = set(), [0]
    while stack:
        i = stack.pop()
        reach.add(i)
        if nodes[i]["tri_count"] == 0:
            stack += [int(nodes[i]["left_first"]), int(nodes[i]["left_first"]) + 1]
    seen = set()
    for i in sorted(reach):
        if nodes[i]["tri_count"] == 0:
            for c in (int(nodes[i]["left_first"]), int(nodes[i]["left_first"]) + 1):
                seen.add(np.array([nodes[c]["aabb_min"][1], nodes[c]["aabb_max"][1]], np.float32).tobytes())
    return len(seen)


def shelf_scene(mm, scenes, n_shelves):
    """The 10x10 maze plus n_shelves small horizontal mirrors at distinct heights, each in its own cell: every shelf adds
    child y-intervals to the BVH."""
    from mirror_maze_b200.host import PLANE_DTYPE, build_bvh

    base = scenes(10)
    extra = np.zeros(n_shelves, dtype=PLANE_DTYPE)
    for i in range(n_shelves):
        x, z = -20.0 + 10.0 * (i % 5), -20.0 + 10.0 * (i // 5)
        extra[i] = ((x + 1.0, -7.0 + 0.75 * i, z + 1.0), (3.0, 0.0, 0.0), (0.0, 0.0, 3.0), (0.8, 0.8, 0.8))
    planes = np.concatenate([base.planes, extra])
    nodes, indices = build_bvh(planes)
    return types.SimpleNamespace(planes=planes, nodes=nodes, indices=indices,
                                 materials=np.concatenate([base.materials, np.ones(n_shelves, np.uint8)]),
                                 emissions=np.concatenate([base.emissions, np.zeros((n_shelves, 4), np.float32)]))


def scene_with_intervals(mm, scenes, want):
    for k in range(0, 20):
        sc = shelf_scene(mm, scenes, k)
        if y_intervals(sc.nodes) == want:
            return sc
    raise AssertionError(f"no shelf scene with {want} y-intervals")


# ---- without a GPU --------------------------------------------------------------------------------------------------------

def test_ytab_instruction_mix_shows_no_contraction():
    """The y-table kernel holds the exact traversal in 3 instantiations: the mixed-literal one (6 quotient pairs a visit, as in
    trace_kernel) and the y-table one for axis-aligned and general rects (4 pairs a visit, plus the table's 8 pairs).  Two
    unrolled visits each: (12 + 2 x (8 + 8)) pairs of add, mul, fma, fma, fma = FADD2 : FMUL2 : FFMA2 = 44 : 44 : 132.  A fused
    or dropped instruction changes the counts (see test_abi.py's check of trace_kernel)."""
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
    kernels = {n: c for n, c in counts.items() if "trace_ytab_kernel" in n}
    assert len(kernels) == 6
    for n, c in kernels.items():
        assert tuple(c) == (44, 44, 132), (n, c)


@pytest.mark.parametrize("maze", [10, 32, 64])
def test_maze_scenes_have_five_y_intervals(mm, scenes, maze):
    """Walls, light panels, outer walls, floor and roof: every maze's BVH children span 5 distinct y-intervals."""
    assert y_intervals(scenes(maze).nodes) == 5


def test_shelf_scenes_reach_the_cap_and_pass_it(mm, scenes):
    assert y_intervals(scene_with_intervals(mm, scenes, MAX_Y_INTERVALS).nodes) == MAX_Y_INTERVALS
    assert y_intervals(scene_with_intervals(mm, scenes, MAX_Y_INTERVALS + 1).nodes) == MAX_Y_INTERVALS + 1


# ---- on the GPU -----------------------------------------------------------------------------------------------------------

def render_both(mm, renderer, u, p, ch, debug=True):
    """(y-table render, trace_kernel render) of one dispatch; checks which kernel each ran."""
    yt = gpu_render(mm, renderer, u, p, ch, debug)
    n_yiv = renderer.scene_info()["y_table"]
    nt = gpu_render(mm, renderer, u, with_flags(mm, p, p.flags | mm.FLAG_NO_Y_TABLE), ch, debug)
    assert renderer.scene_info()["y_table"] == 0
    return yt, nt, n_yiv


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_every_case_with_and_without_the_table(mm, oracle, noise, scenes, renderer, name):
    sc, u, p, ch = build_case(mm, name, scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    yt, nt, n_yiv = render_both(mm, renderer, u, p, ch)
    assert n_yiv == 5
    assert_same(yt, ref, name + " y-table")
    assert_same(nt, ref, name + " NO_Y_TABLE")
    assert yt[1]["literal_rays"] == nt[1]["literal_rays"]
    assert_tail(mm, renderer, yt[3], p, ref[2]["segments"], name + " y-table")
    assert_tail(mm, renderer, nt[3], p, ref[2]["segments"], name + " NO_Y_TABLE")


# spp 64 (64-thread blocks), 128 and 256 (256-thread blocks); the tail on and off; both rect forms; counters-only variant
VARIANTS = [(64, 0), (128, 0), (256, 0), (16, "FLAG_NO_TAIL"), (16, "FLAG_GENERAL_RECTS"), (16, "FLAG_COUNTERS"),
            (128, "FLAG_GENERAL_RECTS"), (16, "FLAG_SCREEN_RGBA8")]


@pytest.mark.gpu
@pytest.mark.parametrize("spp,flag", VARIANTS)
def test_block_shapes_and_flags(mm, oracle, noise, scenes, renderer, spp, flag):
    sc = scenes(32)
    renderer.upload_scene(sc, noise)
    u = mm.default_uniform(32, 96, 64, 2)
    ch = mm.gen_chunks(96, 64, 2)
    p = mm.full_frame_params(u, spp=spp, bounce_limit=8, mirror_limit=15, flags=getattr(mm, flag) if flag else 0)
    debug = flag not in ("FLAG_COUNTERS", "FLAG_SCREEN_RGBA8")
    yt, nt, n_yiv = render_both(mm, renderer, u, p, ch, debug)
    assert n_yiv == 5
    what = f"spp {spp} {flag}"
    if flag == "FLAG_SCREEN_RGBA8":                          # no oracle for quantised stores: the two kernels agree
        assert yt[0].tobytes() == nt[0].tobytes() and yt[1] == nt[1] and yt[3] == nt[3]
        return
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    assert_same(yt, ref if debug else ref[:2] + (None,), what + " y-table")
    assert_same(nt, ref if debug else ref[:2] + (None,), what + " NO_Y_TABLE")
    if flag == "FLAG_COUNTERS":
        assert yt[1] == nt[1]
    assert_tail(mm, renderer, yt[3], p, ref[2]["segments"], what)


@pytest.mark.gpu
def test_literal_lanes_inside_y_table_warps(mm, oracle, noise, scenes, renderer):
    """tiny_origin: every primary ray takes the literal traversal over the 192-B records, later segments the y-table one."""
    sc, u, p, ch = build_case(mm, "tiny_origin", scenes)
    renderer.upload_scene(sc, noise)
    yt, nt, n_yiv = render_both(mm, renderer, u, p, ch)
    assert n_yiv == 5
    assert yt[1]["paths"] <= yt[1]["literal_rays"] < yt[1]["rays"]
    assert_same(yt, oracle.render(sc, noise, u, p, ch, debug=True), "tiny_origin")


@pytest.mark.gpu
def test_y_table_delivery_routes(mm, noise, scenes, renderer):
    """Tiles (mm_render_device + scatter), a zero-copy host frame, and peer frames (mm_render_peers_device) from the y-table
    kernels equal trace_kernel's frame."""
    import torch

    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    full = renderer.render(u, with_flags(mm, p, mm.FLAG_NO_Y_TABLE), ch)[0]
    H, W = int(u.view_height), int(u.view_width)
    hf = mm.HostFrame(H, W)
    renderer.render(u, p, ch, out=hf.array)
    assert renderer.scene_info()["y_table"] == 5 and renderer.last_tail()[0] > 0
    assert hf.array.tobytes() == full.tobytes()
    hf.close()

    dev = torch.device("cuda", 0)
    renderer.set_chunks(ch)
    ppc = u.chunk_width ** 2
    tiles = torch.zeros((p.grid_x * p.grid_y, ppc, 4), dtype=torch.float32, device=dev)
    image = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    renderer.render_device(u, p, tiles_ptr=tiles.data_ptr())
    renderer.scatter_tiles_device(u, p, tiles.data_ptr(), image.data_ptr())
    renderer.sync()
    assert image.cpu().numpy().tobytes() == full.tobytes()

    frames = [torch.zeros((H, W, 4), dtype=torch.float32, device=dev) for _ in range(2)]
    renderer.render_peers_device(u, p, [f.data_ptr() for f in frames])
    renderer.sync()
    assert renderer.scene_info()["y_table"] == 5
    for f in frames:
        assert f.cpu().numpy().tobytes() == full.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [MAX_Y_INTERVALS, MAX_Y_INTERVALS + 1])
def test_scene_at_and_past_the_cap(mm, oracle, noise, scenes, n):
    sc = scene_with_intervals(mm, scenes, n)
    r = mm.Renderer(0)
    try:
        r.upload_scene(sc, noise)
        u = mm.default_uniform(10, 96, 64, 4)
        ch = mm.gen_chunks(96, 64, 4)
        p = mm.full_frame_params(u, spp=16, bounce_limit=8, mirror_limit=15)
        ref = oracle.render(sc, noise, u, p, ch, debug=True)
        yt, nt, n_yiv = render_both(mm, r, u, p, ch)
        assert n_yiv == (n if n <= MAX_Y_INTERVALS else 0)
        assert_same(yt, ref, f"{n} intervals")
        assert_same(nt, ref, f"{n} intervals NO_Y_TABLE")
        assert_tail(mm, r, yt[3], p, ref[2]["segments"], f"{n} intervals")
    finally:
        r.close()
