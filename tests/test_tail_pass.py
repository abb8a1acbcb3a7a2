"""The straggler tail (render_kernel.cu: trace_kernel queues the paths of warps past bounce_limit segments with few live lanes,
trace_tail_kernel finishes them): frames, counters and per-path observables are the same bits with the tail, without it
(MM_FLAG_NO_TAIL) and in the oracle, including when the queue overflows and through every pixel delivery route."""
import numpy as np
import pytest

from cases import build_case

pytestmark = pytest.mark.gpu
COUNTER_KEYS = ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits", "max_stack")   # the oracle's
# cases with many paths past bounce_limit (mirror hits), several spp / block shapes, and mirror_limit 15 and 2
TAIL_CASES = ["cfg2_small", "maze64", "cfg3_small", "yaw", "mirror_limit2", "chunk1_spp256", "chunk3_spp32", "chunk16_spp1",
              "chunk2_spp4", "tiny_origin"]


def with_flags(mm, p, flags):
    q = mm.Params.from_buffer_copy(bytes(p))
    q.flags = flags
    return q


def assert_identical(a, b):
    img, cnt, dbg = a
    rimg, rcnt, rdbg = b
    assert img.tobytes() == rimg.tobytes(), "image not bit-identical"
    for k in ("first_hit", "segments", "mirror_hits", "radiance"):
        assert dbg[k].tobytes() == rdbg[k].tobytes(), k
    for k in COUNTER_KEYS:
        assert cnt[k] == rcnt[k], k


@pytest.mark.parametrize("name", TAIL_CASES)
def test_tail_equals_single_kernel_and_oracle(mm, oracle, noise, scenes, renderer, name):
    sc, u, p, ch = build_case(mm, name, scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    tail = renderer.render(u, p, ch, debug=True)
    queued, pixels = renderer.last_tail()
    one = renderer.render(u, with_flags(mm, p, mm.FLAG_NO_TAIL), ch, debug=True)
    assert renderer.last_tail() == (0, 0)
    assert_identical(tail, ref)
    assert_identical(one, ref)
    assert tail[1]["literal_rays"] == one[1]["literal_rays"]
    past = int((ref[2]["segments"] > p.bounce_limit).sum())
    if past >= 64:
        assert queued > 0, f"{past} paths ran past bounce_limit, none was queued"
        assert 0 < pixels <= queued


def test_tail_counters_only_and_rgba8(mm, oracle, noise, scenes, renderer):
    """The counters-only and the plain kernel variants, and quantised pixel stores from both kernels."""
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    for flags in (mm.FLAG_COUNTERS, 0, mm.FLAG_SCREEN_RGBA8):
        a = renderer.render(u, with_flags(mm, p, flags), ch)
        assert renderer.last_tail()[0] > 0
        b = renderer.render(u, with_flags(mm, p, flags | mm.FLAG_NO_TAIL), ch)
        assert a[0].tobytes() == b[0].tobytes()
        assert a[1] == b[1]


@pytest.mark.parametrize("cap", [0, 1, 37, 500])
def test_tail_queue_overflow(mm, oracle, noise, scenes, renderer, monkeypatch, cap):
    """A queue smaller than the demand: the warps that find it full keep their paths (some warps partly spilled)."""
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)
    monkeypatch.setenv("MM_TAIL_CAP", str(cap))
    got = renderer.render(u, p, ch, debug=True)
    queued, pixels = renderer.last_tail()
    monkeypatch.delenv("MM_TAIL_CAP")
    assert queued == cap and pixels <= cap
    assert_identical(got, ref)


def test_tail_tiles_and_zero_copy_host_frame(mm, noise, scenes, renderer):
    """Deferred pixels reach the tile array (mm_render_device) and a mapped pinned host frame (zero-copy stores)."""
    import torch

    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    full = renderer.render(u, with_flags(mm, p, mm.FLAG_NO_TAIL), ch)[0]
    H, W = int(u.view_height), int(u.view_width)
    hf = mm.HostFrame(H, W)
    renderer.render(u, p, ch, out=hf.array)
    assert renderer.last_tail()[0] > 0
    assert hf.array.tobytes() == full.tobytes()
    hf.close()

    dev = torch.device("cuda", 0)
    renderer.set_chunks(ch)
    ppc = u.chunk_width ** 2
    n_groups = p.grid_x * p.grid_y
    tiles = torch.zeros((n_groups, ppc, 4), dtype=torch.float32, device=dev)
    image = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    renderer.render_device(u, p, tiles_ptr=tiles.data_ptr())
    renderer.scatter_tiles_device(u, p, tiles.data_ptr(), image.data_ptr())
    renderer.sync()
    assert renderer.last_tail()[0] > 0
    assert image.cpu().numpy().tobytes() == full.tobytes()


def test_tail_two_gpu_fused_frame(mm, noise, scenes, renderer):
    """mm_multi with NVLink peer stores: deferred pixels are stored into every device's frame before the frame completes."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sc, u, p, ch = build_case(mm, "cfg2_small", scenes)
    renderer.upload_scene(sc, noise)
    full = renderer.render(u, with_flags(mm, p, mm.FLAG_NO_TAIL), ch)[0]
    m = mm.MultiRenderer([0, 1], "peer")
    m.upload_scene(sc, noise)
    out = np.zeros_like(full)
    m.render(u, p, ch, out)
    m.close()
    assert out.tobytes() == full.tobytes()
