"""The straggler tail's trigger, pinned exactly, and dispatch shapes that no case of tests/cases.py reaches.

The tail (render_kernel.cu: trace_kernel queues the paths of sparse warps past bounce_limit, trace_tail_kernel finishes
them) is bit-identical to the one-kernel render whichever paths it queues, so parity alone cannot tell a right trigger
from a wrong one.  tail_model() predicts from the oracle's per-path segment counts exactly how many paths the trigger
queues and how many pixels it defers, and every GPU render here checks mm_last_tail against it.

Every comparison is bit for bit against oracle.render(..., debug=True): the first-hit, segment, mirror-hit and radiance
arrays, the image and the oracle's seven counters.  GPU renders go into a zeroed mapped pinned frame (zero-copy stores),
so the image holds exactly the pixels the dispatch wrote, like the oracle's.  Tests marked gpu need a B200; the others
(the trigger model and the oracle companions) run anywhere."""
import os

import numpy as np
import pytest

from cases import build_case

COUNTER_KEYS = ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits", "max_stack")   # the oracle's
TAIL_K_DEFAULT = 8                    # api.cu build_launch: kTailK
TAIL_PATH_BYTES = 80                  # sizeof(TailPath): five float4
TAIL_BUDGET = 1 << 30                 # api.cu build_launch: kTailBudget, queue + deferred-pixel slots


# ---- the trigger model ---------------------------------------------------------------------------------------------------

def tail_queued(segments, bounce_limit, k):
    """Boolean mask of the paths trace_kernel queues, from each path's segment count (render_kernel.cu, DESIGN §4).

    Warps are 32 consecutive path indices of the launch.  A lane is live at segment boundary s when its path runs more
    than s segments.  A warp queues all its live lanes at the first s >= bounce_limit where 1 <= live <= k, once.  live(s)
    never grows with s, so that boundary is s* = max(bounce_limit, the (k+1)-th largest segment count of the warp), and the
    queued lanes are those with segments > s*."""
    seg = np.asarray(segments, dtype=np.int64)
    n = len(seg)
    if k <= 0 or n == 0:
        return np.zeros(n, dtype=bool)
    w = np.zeros(-(-n // 32) * 32, dtype=np.int64)           # lanes without a path: 0 segments, never live
    w[:n] = seg
    w = w.reshape(-1, 32)
    kth = -np.sort(-w, axis=1)[:, k] if k < 32 else np.zeros(len(w), dtype=np.int64)
    s = np.maximum(int(bounce_limit), kth)
    return (w > s[:, None]).reshape(-1)[:n]


def tail_model(segments, bounce_limit, k, spp):
    """(queued paths, deferred pixels) with a queue that holds them all.  The queue head is the sum of the warps' live
    counts whatever the capacity; a deferred pixel is a pixel (path >> log2 spp) with a queued path."""
    q = np.nonzero(tail_queued(segments, bounce_limit, k))[0]
    return len(q), len(np.unique(q >> (int(spp).bit_length() - 1)))


def tail_capacity(total_paths, spp, cap_env=None):
    """Queue entries build_launch provides: an eighth of the launch's paths plus 1024, within kTailBudget, and MM_TAIL_CAP."""
    cap = min(total_paths // 8 + 1024, TAIL_BUDGET // (TAIL_PATH_BYTES + (4 + 3 * spp) * 4))
    return cap if cap_env is None else min(cap, cap_env)


def _trigger_by_simulation(segments, bounce_limit, k):
    """The trigger as trace_kernel's bounce loop runs it, boundary by boundary: the independent check of tail_queued."""
    seg = list(segments)
    out = [False] * len(seg)
    for w0 in range(0, len(seg), 32):
        lanes = range(w0, min(w0 + 32, len(seg)))
        s = 0
        while True:
            live = [i for i in lanes if seg[i] > s]
            if not live:
                break
            if k > 0 and len(live) <= k and s >= bounce_limit:
                for i in live:
                    out[i] = True
                break
            s += 1
    return np.array(out, dtype=bool)


# ---- shapes, renders, comparisons ----------------------------------------------------------------------------------------

# Dispatch shapes no case of tests/cases.py reaches.  32x32 and 64x64 mazes where the tail should engage (a 16x16 maze
# sends only 0.1-0.2 % of its paths past bounce_limit).
SHAPES = {
    # spp 128: two pixels per 256-thread block, so the block epilogue's pslot holds two pixels; 16-octet serial sum
    "spp128_chunk1": dict(maze=32, W=24, H=16, chunk=1, spp=128, bounce=8, mirror=15),                       # T = 128
    "spp128_chunk2": dict(maze=32, W=32, H=24, chunk=2, spp=128, bounce=8, mirror=15),                       # T = 512
    # T < 32 and not a power of two: virtual groups straddle warps, dim_x = T
    "t9_chunk3_spp1": dict(maze=32, W=192, H=108, chunk=3, spp=1, bounce=8, mirror=15),
    "t18_chunk3_spp2_ragged": dict(maze=64, W=151, H=92, chunk=3, spp=2, bounce=8, mirror=15, time=5),
    "t25_chunk5_spp1": dict(maze=32, W=200, H=100, chunk=5, spp=1, bounce=8, mirror=15, center=(-15.0, 0.0, 5.0), half_theta=0.9),
    # very large groups: dim_y = 2048, so texid_y * 9737333 wraps in u32 (shaders.metal:298)
    "chunk64_spp16": dict(maze=32, W=128, H=64, chunk=64, spp=16, bounce=8, mirror=15),                      # T = 65536
    "chunk32_spp256": dict(maze=64, W=32, H=32, chunk=32, spp=256, bounce=8, mirror=15),                     # T = 2^18
    # mirror_limit 0 and 1 on the mirror-heavy pose of the mirror_limit2 case
    "mirror_limit0": dict(maze=32, W=96, H=64, chunk=4, spp=8, bounce=8, mirror=0, center=(-5.0, 0.0, 35.0), half_theta=2.4),
    "mirror_limit1": dict(maze=32, W=96, H=64, chunk=4, spp=8, bounce=8, mirror=1, center=(-5.0, 0.0, 35.0), half_theta=2.4),
    # both limits at their 4096 maximum: about 580 segments a path, n | mirror_hits << 16 in the queued state
    "limits4096": dict(maze=16, W=32, H=32, chunk=4, spp=8, bounce=4096, mirror=4096),
}

# the 640x360 16-spp frame of a 32x32 maze: a queue longer than trace_tail_kernel's grid stride at K = 8 and 32
STRIDE_FRAME = dict(maze=32, W=640, H=360, chunk=4, spp=16, bounce=8, mirror=15)


def build_shape(mm, scenes, c):
    sc = scenes(c["maze"])
    u = mm.default_uniform(c["maze"], c["W"], c["H"], c["chunk"], c.get("time", 0), camera_center=c.get("center"),
                           half_theta=c.get("half_theta"))
    ch = mm.gen_chunks(c["W"], c["H"], c["chunk"])
    p = mm.full_frame_params(u, spp=c["spp"], bounce_limit=c["bounce"], mirror_limit=c["mirror"], flags=c.get("flags", 0))
    if "part" in c:
        p.group_first, p.group_step, p.group_count = c["part"]
    return sc, u, p, ch


def with_flags(mm, p, flags):
    q = mm.Params.from_buffer_copy(bytes(p))
    q.flags = flags
    return q


def gpu_render(mm, renderer, u, p, ch, debug):
    """renderer.render into a zeroed mapped pinned frame; returns (image, counters, debug arrays, last_tail())."""
    hf = mm.HostFrame(int(u.view_height), int(u.view_width))
    try:
        img, cnt, dbg = renderer.render(u, p, ch, out=hf.array, debug=debug)
        return img.copy(), cnt, dbg, renderer.last_tail()
    finally:
        hf.close()


def assert_same(got, ref, what):
    img, cnt, dbg = got[:3]
    rimg, rcnt, rdbg = ref
    if dbg is not None:
        for k in ("first_hit", "segments", "mirror_hits", "radiance"):
            assert dbg[k].tobytes() == rdbg[k].tobytes(), f"{k} differs: {what}"
        keys = COUNTER_KEYS
    else:                                                    # the plain kernel variants count rays, hits and paths only
        keys = COUNTER_KEYS if got[1].get("inner_visits") else ("paths", "rays", "hits")
    assert img.tobytes() == rimg.tobytes(), f"image not bit-identical: {what}"
    for k in keys:
        assert cnt[k] == rcnt[k], f"counter {k}: {cnt[k]} != {rcnt[k]}: {what}"


def pool_engages(mm, renderer, p):
    """configure_pool's test for the maze scenes: the pool kernel runs instead of trace_kernel (and has no tail)."""
    info = renderer.scene_info()
    return bool(p.flags & mm.FLAG_POOL_KERNEL) and not (p.flags & (mm.FLAG_FORCE_LITERAL | mm.FLAG_RCP_SLAB)) \
        and p.spp <= 64 and bool(info["fast_slab_ok"]) and bool(info["fast_rect_ok"])


def assert_tail(mm, renderer, got_tail, p, segments, what, k=TAIL_K_DEFAULT, cap_env=None):
    """mm_last_tail against the model of the oracle's segments of the same dispatch."""
    if p.flags & (mm.FLAG_NO_TAIL | mm.FLAG_REGROUP) or pool_engages(mm, renderer, p):
        assert got_tail == (0, 0), f"tail ran under flags {p.flags}: {got_tail}: {what}"
        return
    cap = tail_capacity(len(segments), p.spp, cap_env)
    queued, pixels = tail_model(segments, p.bounce_limit, k if cap else 0, p.spp)
    if queued <= cap:
        assert got_tail == (queued, pixels), f"last_tail {got_tail} != model {(queued, pixels)} (K {k}, cap {cap}): {what}"
    else:                                                    # which warps win the queue is a race; how many entries it holds is not
        assert got_tail[0] == cap and got_tail[1] <= min(pixels, cap), \
            f"last_tail {got_tail} vs model {(queued, pixels)} with capacity {cap} (K {k}): {what}"


# ---- 1. the trigger model ------------------------------------------------------------------------------------------------

def test_tail_model_on_hand_built_warps():
    seg = np.full(40, 8)                                     # warp 0: 32 lanes, warp 1: a partial last warp of 8 lanes
    seg[[3, 17, 30]] = [9, 10, 12]                           # warp 0: 3 lanes past bounce_limit 8
    seg[[33, 39]] = 9                                        # warp 1: 2 lanes past it
    assert tail_queued(seg, 8, 8).nonzero()[0].tolist() == [3, 17, 30, 33, 39]
    assert tail_model(seg, 8, 8, 4) == (5, 5)                # at 4 spp: pixels 0, 4, 7, 8 and 9
    assert tail_model(seg, 8, 8, 16) == (5, 3)               # at 16 spp: pixels 0, 1 and 2
    # K = 2: warp 0 has 3 live lanes at s = 8 and queues the 2 left at s = 9; warp 1 queues its 2 at s = 8
    assert tail_queued(seg, 8, 2).nonzero()[0].tolist() == [17, 30, 33, 39]
    # K = 1: warp 0 queues its last lane at s = 10; warp 1 goes from 2 live lanes to none and never queues
    assert tail_queued(seg, 8, 1).nonzero()[0].tolist() == [30]
    # bounce_limit above the warp's longest path: nothing is live there
    assert tail_model(seg, 12, 32, 1) == (0, 0)
    # a warp whose live lanes never drop to K: two lanes run to the end together, K = 1 never fires
    two = np.full(32, 4)
    two[[5, 6]] = 20
    assert tail_model(two, 4, 1, 1) == (0, 0)
    assert tail_model(two, 4, 2, 1) == (2, 2)
    # s = bounce_limit itself counts: live = 2 <= K at s = 4 queues both with 16 segments to go
    assert tail_queued(two, 4, 2).nonzero()[0].tolist() == [5, 6]
    # bounce_limit 0: no path runs a segment, so nothing is live at any boundary
    assert tail_model(np.zeros(70, dtype=np.uint32), 0, 8, 2) == (0, 0)
    # K = 0 disables the trigger; K = 32 queues every path past bounce_limit
    rng = np.random.default_rng(3)
    r = rng.integers(0, 14, size=1000)
    assert tail_model(r, 8, 0, 8) == (0, 0)
    assert tail_queued(r, 8, 32).tolist() == (r > 8).tolist()


@pytest.mark.parametrize("k", [1, 2, 5, 8, 16, 31, 32])
def test_tail_model_equals_boundary_by_boundary_simulation(k):
    """The closed form of tail_queued against the bounce loop run boundary by boundary, on random segment counts with long
    tails and partial last warps."""
    rng = np.random.default_rng(100 + k)
    for bl in (1, 3, 8):
        n = int(rng.integers(1, 700))
        seg = bl + rng.geometric(0.55, size=n) - 1           # most paths end at bounce_limit, some after mirror hits
        seg = np.where(rng.random(n) < 0.2, rng.integers(1, bl + 1, size=n), seg)   # paths that miss before it
        assert tail_queued(seg, bl, k).tolist() == _trigger_by_simulation(seg, bl, k).tolist(), (k, bl, n)


def test_tail_model_reference_counts(mm, oracle, noise, scenes):
    """The model on the oracle's segments of cfg2_small: 20 595 paths / 11 784 pixels at K = 8; 29 958 / 12 005 at K = 32,
    where it is every path with more than bounce_limit segments (9.03 % of 331 776)."""
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    seg = oracle.render(sc, noise, u, p, ch, debug=True)[2]["segments"]
    assert len(seg) == 331776
    assert tail_model(seg, p.bounce_limit, 8, p.spp) == (20595, 11784)
    assert tail_model(seg, p.bounce_limit, 32, p.spp) == (29958, 12005) == (int((seg > 8).sum()), 12005)


# ---- GPU: the trigger against mm_last_tail -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 8, 16, 31, 32])
def test_tail_trigger_matches_model(mm, oracle, noise, scenes, renderer, monkeypatch, k):
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    monkeypatch.setenv("MM_TAIL_K", str(k))
    for debug in (True, False):
        got = gpu_render(mm, renderer, u, p, ch, debug)
        what = f"cfg2_small K {k} debug {debug}"
        assert_same(got, ref if debug else (ref[0], ref[1], None), what)
        assert_tail(mm, renderer, got[3], p, ref[2]["segments"], what, k=k)
    assert got[3][0] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 500, 5000, 20595, 20596])
def test_tail_capped_queue_matches_model(mm, oracle, noise, scenes, renderer, monkeypatch, cap):
    """MM_TAIL_CAP below, at and above the 20 595 paths the default trigger queues in cfg2_small."""
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    monkeypatch.setenv("MM_TAIL_CAP", str(cap))
    got = gpu_render(mm, renderer, u, p, ch, True)
    assert_same(got, ref, f"cap {cap}")
    assert_tail(mm, renderer, got[3], p, ref[2]["segments"], f"cap {cap}", cap_env=cap)
    assert got[3][0] == min(cap, 20595)


# ---- GPU: the tail under stress ------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 32])
def test_tail_queue_longer_than_grid_stride(mm, oracle, noise, scenes, renderer, monkeypatch, k):
    """With debug arrays on, a queue longer than trace_tail_kernel's grid (n_sms x 4 blocks of 256 threads), so its
    grid-stride loop runs at least twice and the segment count pseg + seg is summed across iterations."""
    import torch

    stride = torch.cuda.get_device_properties(0).multi_processor_count * 1024
    sc, u, p, ch = build_shape(mm, scenes, STRIDE_FRAME)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    monkeypatch.setenv("MM_TAIL_K", str(k))
    got = gpu_render(mm, renderer, u, p, ch, True)
    what = f"640x360 K {k}"
    assert_same(got, ref, what)
    assert_tail(mm, renderer, got[3], p, ref[2]["segments"], what, k=k)
    queued = got[3][0]
    print(f"K {k}: queued {queued}, stride {stride}, ratio {queued / stride:.2f}")
    assert queued > stride, f"{queued} queued paths fit one grid stride of {stride}"
    one = gpu_render(mm, renderer, u, with_flags(mm, p, mm.FLAG_NO_TAIL), ch, True)
    assert_same(one, ref, what + " NO_TAIL")
    assert one[3] == (0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("flag", ["FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_RCP_SLAB", "FLAG_COUNTERS", "FLAG_SCREEN_RGBA8"])
def test_tail_under_every_arithmetic_and_output_variant(mm, oracle, noise, scenes, renderer, flag):
    """The trigger does not depend on these flags: the same model of the oracle's segments (in RCP mode for RCP_SLAB)."""
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    p = with_flags(mm, p, getattr(mm, flag))
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    for debug in (True, False):
        got = gpu_render(mm, renderer, u, p, ch, debug)
        assert_same(got, ref if debug else (ref[0], ref[1], None), f"{flag} debug {debug}")
        assert_tail(mm, renderer, got[3], p, ref[2]["segments"], f"{flag} debug {debug}")
        assert got[3][0] > 0
    one = gpu_render(mm, renderer, u, with_flags(mm, p, p.flags | mm.FLAG_NO_TAIL), ch, False)
    assert one[0].tobytes() == got[0].tobytes() and one[3] == (0, 0)


@pytest.mark.gpu
def test_tail_in_partial_dispatches(mm, oracle, noise, scenes):
    """Three interleaved ranks on one context, each into the frame (debug arrays on) and into tiles and a device frame at
    once: each rank's last_tail matches the model of the oracle's render of that same partial dispatch (launch-local path
    indices), the deferred pixels land at their tile index (h[3]) and the scattered tiles rebuild the frame."""
    import torch

    c = dict(maze=32, W=200, H=108, chunk=4, spp=16, bounce=8, mirror=15, time=3)
    sc, u, p, ch = build_shape(mm, scenes, c)
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    H, W = c["H"], c["W"]
    n_groups = p.grid_x * p.grid_y
    world = 3
    full_ref = np.zeros((H, W, 4), dtype=np.float32)
    dev = torch.device("cuda", 0)
    image = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    scattered = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    ppc = c["chunk"] ** 2
    for rank in range(world):
        q = mm.Params.from_buffer_copy(bytes(p))
        q.group_first, q.group_step, q.group_count = mm.tile_partition(n_groups, rank, world)
        what = f"rank {rank} of {world}"
        ref = oracle.render(sc, noise, u, q, ch, debug=True)
        oracle.render(sc, noise, u, q, ch, out=full_ref)
        got = gpu_render(mm, r, u, q, ch, True)
        assert_same(got, ref, what)
        assert_tail(mm, r, got[3], q, ref[2]["segments"], what)
        assert got[3][0] > 0
        r.set_chunks(ch)
        tiles = torch.zeros((q.group_count, ppc, 4), dtype=torch.float32, device=dev)
        r.render_device(u, q, image_ptr=image.data_ptr(), tiles_ptr=tiles.data_ptr())
        assert_tail(mm, r, r.last_tail(), q, ref[2]["segments"], what + " render_device")
        r.scatter_tiles_device(u, q, tiles.data_ptr(), scattered.data_ptr())
        r.sync()
        torch.cuda.synchronize()
    assert image.cpu().numpy().tobytes() == full_ref.tobytes()
    assert scattered.cpu().numpy().tobytes() == full_ref.tobytes()
    r.close()


@pytest.mark.gpu
def test_tail_buffers_reused_across_spp(mm, oracle, noise, scenes):
    """One context: 16 spp large, then 256 spp small (larger deferred-pixel slots, shorter queue: the buffers are reused),
    128 spp, 16 spp again, and last a frame that needs a longer queue and more slot bytes than any before (regrowth)."""
    seq = [dict(maze=32, W=320, H=180, chunk=4, spp=16, bounce=8, mirror=15),
           dict(maze=32, W=24, H=16, chunk=1, spp=256, bounce=8, mirror=15, center=(-5.0, 0.0, 35.0), half_theta=2.4),
           dict(maze=32, W=32, H=32, chunk=2, spp=128, bounce=8, mirror=15),
           dict(maze=32, W=192, H=108, chunk=4, spp=16, bounce=8, mirror=15, time=7),
           dict(maze=64, W=384, H=216, chunk=4, spp=16, bounce=8, mirror=15)]
    r = mm.Renderer(0)
    for i, c in enumerate(seq):
        sc, u, p, ch = build_shape(mm, scenes, c)
        r.upload_scene(sc, noise)
        ref = oracle.render(sc, noise, u, p, ch, debug=True)
        for debug in (True, False):
            got = gpu_render(mm, r, u, p, ch, debug)
            what = f"render {i} of the sequence, {c}, debug {debug}"
            assert_same(got, ref if debug else (ref[0], ref[1], None), what)
            assert_tail(mm, r, got[3], p, ref[2]["segments"], what)
            assert got[3][0] > 0, what
    r.close()


@pytest.mark.gpu
def test_regroup_and_pool_kernels_have_no_tail(mm, oracle, noise, scenes, renderer):
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    for flags in (mm.FLAG_REGROUP, mm.FLAG_POOL_KERNEL):
        q = with_flags(mm, p, flags)
        assert flags == mm.FLAG_REGROUP or pool_engages(mm, renderer, q)
        for debug in (True, False):
            got = gpu_render(mm, renderer, u, q, ch, debug)
            assert_same(got, ref if debug else (ref[0], ref[1], None), f"flags {flags}")
            assert got[3] == (0, 0)


# ---- 3. dispatch shapes no case reaches ----------------------------------------------------------------------------------

VARIANTS = ["default", "FLAG_NO_TAIL", "FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_REGROUP", "FLAG_POOL_KERNEL"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_shape_every_kernel_matches_oracle(mm, oracle, noise, scenes, renderer, name):
    sc, u, p, ch = build_shape(mm, scenes, SHAPES[name])
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    engaged = False
    for v in VARIANTS:
        q = with_flags(mm, p, 0 if v == "default" else getattr(mm, v))
        for debug in (True, False):
            got = gpu_render(mm, renderer, u, q, ch, debug)
            what = f"{name} {v} debug {debug}"
            assert_same(got, ref if debug else (ref[0], ref[1], None), what)
            assert_tail(mm, renderer, got[3], q, ref[2]["segments"], what)
            engaged |= got[3][0] > 0
    past = int((ref[2]["segments"] > p.bounce_limit).sum())
    assert engaged or past < 32, f"{name}: {past} paths past bounce_limit, none queued"


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_shape_oracle_matches_numpy_transcription(mm, oracle, noise, scenes, name):
    """The new shapes in the C++ oracle against oracle/np_oracle.py, the independent transcription (the small ones)."""
    from oracle import np_oracle

    sc, u, p, ch = build_shape(mm, scenes, SHAPES[name])
    n_paths = (p.group_count or p.grid_x * p.grid_y) * u.chunk_width ** 2 * p.spp
    if n_paths * min(p.bounce_limit + p.mirror_limit, 40) > 4_000_000:
        pytest.skip(f"{n_paths} paths: too slow for the numpy transcription")
    assert_same(oracle.render(sc, noise, u, p, ch, debug=True), np_oracle.render(sc, noise, u, p, ch), name)


# ---- 4. seeded random dispatches -----------------------------------------------------------------------------------------

SHAPES_SEED = int(os.environ.get("MM_SHAPES_SEED", "20261020"))
SHAPES_DRAWS = int(os.environ.get("MM_SHAPES_DRAWS", "40"))
MAX_PATHS = 300_000
DRAW_FLAGS = ["FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_RCP_SLAB", "FLAG_COUNTERS", "FLAG_SCREEN_RGBA8", "FLAG_NO_TAIL",
              "FLAG_REGROUP", "FLAG_POOL_KERNEL"]


def draw_dispatch(i):
    """Draw i of the legal dispatch space: a dict of plain values (printed in every assertion message)."""
    rng = np.random.default_rng([SHAPES_SEED, i])
    maze = 256 if rng.random() < 0.08 else int(rng.integers(2, 65))
    while True:
        chunk = int(rng.choice([int(rng.integers(1, 9)), int(rng.integers(1, 65))]))
        spp = 1 << int(rng.integers(0, 9))
        T = chunk * chunk * spp
        if (T <= 32 or T % 32 == 0) and T <= MAX_PATHS:
            break
    max_groups = MAX_PATHS // T
    gx = int(rng.integers(1, min(max_groups, 48) + 1))
    gy = int(rng.integers(1, max(1, min(max_groups // gx, 48)) + 1))
    W = gx * chunk + (int(rng.integers(0, chunk)) if rng.random() < 0.5 else 0)     # frames that are not chunk multiples
    H = gy * chunk + (int(rng.integers(0, chunk)) if rng.random() < 0.5 else 0)
    half = 5.0 * maze
    where = rng.integers(0, 4)
    if where == 0:                                           # inside, in a cell
        cx, cz = -half + 10.0 * rng.integers(0, maze) + 5.0, -half + 10.0 * rng.integers(0, maze) + 5.0
    elif where == 1:                                         # inside, anywhere
        cx, cz = rng.uniform(-half, half), rng.uniform(-half, half)
    elif where == 2:                                         # on a wall plane coordinate
        cx, cz = -half + 10.0 * rng.integers(0, maze + 1), rng.uniform(-half, half)
    else:                                                    # outside the box
        cx, cz = rng.uniform(-3 * half - 50, 3 * half + 50), -half - rng.uniform(1.0, 200.0)
    cy = float(rng.uniform(-7.0, 1.5))
    time = int(rng.integers(0, 1000)) if rng.random() < 0.6 else int(rng.integers(0, 1 << 26))
    n_groups = gx * gy
    if rng.random() < 0.5:
        world = int(rng.integers(1, 6))
        part = tuple(int(v) for v in (lambda r: (r, world, (n_groups - r + world - 1) // world))(int(rng.integers(0, min(world, n_groups)))))
    else:
        step = int(rng.integers(1, 5))
        first = int(rng.integers(0, n_groups))
        part = (first, step, int(rng.integers(1, (n_groups - 1 - first) // step + 2)))
    flags = [f for f in DRAW_FLAGS if rng.random() < 0.25]
    return dict(maze=maze, W=W, H=H, chunk=chunk, spp=spp, bounce=int(rng.integers(0, 25)), mirror=int(rng.integers(0, 17)),
                time=time, center=(float(cx), cy, float(cz)), half_theta=float(rng.uniform(0.0, np.pi)), part=part,
                flag_names=flags, tail_k=int(rng.integers(0, 33)))


def build_draw(mm, scenes, c):
    sc, u, p, ch = build_shape(mm, scenes, c)
    p.flags = sum(getattr(mm, f) for f in c["flag_names"])
    return sc, u, p, ch


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(SHAPES_DRAWS))
def test_random_dispatch_matches_oracle(mm, oracle, noise, scenes, renderer, monkeypatch, i):
    c = draw_dispatch(i)
    sc, u, p, ch = build_draw(mm, scenes, c)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    monkeypatch.setenv("MM_TAIL_K", str(c["tail_k"]))
    for debug in (True, False):
        got = gpu_render(mm, renderer, u, p, ch, debug)
        what = f"draw {i}: {c}, debug {debug}"
        assert_same(got, ref if debug else (ref[0], ref[1], None), what)
        assert_tail(mm, renderer, got[3], p, ref[2]["segments"], what, k=c["tail_k"])


@pytest.mark.parametrize("i", range(SHAPES_DRAWS))
def test_random_dispatch_oracle_accepts_and_matches_numpy(mm, oracle, noise, scenes, i):
    """Every draw is a dispatch the C++ oracle renders; the small ones equal oracle/np_oracle.py bit for bit."""
    from oracle import np_oracle

    c = draw_dispatch(i)
    sc, u, p, ch = build_draw(mm, scenes, c)
    n_paths = p.group_count * u.chunk_width ** 2 * p.spp
    assert 0 < n_paths <= MAX_PATHS, c
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    assert ref[1]["paths"] == n_paths, c
    if n_paths < 20_000:
        img, cnt, dbg = np_oracle.render(sc, noise, u, p, ch)
        if p.flags & mm.FLAG_SCREEN_RGBA8:                   # the transcription leaves the screen's quantisation to its caller
            img = np_oracle.quant8(img)
        assert_same(ref, (img, cnt, dbg), f"draw {i}: {c}")
