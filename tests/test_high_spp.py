"""spp 512 and 1024: the 1024-thread block shape (two pixels or one a block), including the reference's chunk-width-1
dispatch at 1024 samples per pixel (32 x 32 threads for one pixel).

The C++ oracle (oracle/mm_oracle.cpp) accepts spp up to 256, the range its comparison with the reference's own shader covers.
The new sample counts are checked against oracle/np_oracle.py, the independent numpy transcription, which has no spp limit.
It is pinned to the C++ oracle path by path here: a dispatch of chunk c at spp s runs the same paths as one of chunk 2c at
spp s/4 (T, the group dims and so every seed are the same), with each pixel's quarter of the samples moved onto it by a
shifted chunk list, and the per-pixel reduction is restated on its own.

Every GPU comparison is bit for bit against the reference render: image, counters and the four per-path arrays, with GPU
renders into a zeroed mapped pinned frame so that the image holds exactly the pixels the dispatch wrote.  Every GPU render
also checks mm_last_tail against the straggler-tail model of the reference's segment counts.  Above spp 256 MM_FLAG_REGROUP
and MM_FLAG_POOL_KERNEL fall back to the default kernel, so the tail runs under them too.  Tests marked gpu need a B200; the
others (the transcription against the oracle, the refusals, the new kernels' instruction mix) run anywhere."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_general_scenes import dispatch as general_dispatch, scene as general_scene
from test_tail_and_shapes import COUNTER_KEYS, assert_same, build_shape, gpu_render, tail_capacity, tail_model, with_flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_UNSUPPORTED = -5
TAIL_K_DEFAULT = 8                    # api.cu build_launch: kTailK
DBG_KEYS = ("first_hit", "segments", "mirror_hits", "radiance")

# 32x32 maze, 8 bounces: enough paths past bounce_limit for the tail to engage at both sample counts
S512 = dict(maze=32, W=24, H=16, chunk=1, spp=512, bounce=8, mirror=15, time=5)                  # 196 608 paths, 2 pixels a block
S1024 = dict(maze=32, W=16, H=12, chunk=1, spp=1024, bounce=8, mirror=15, time=9)                # 196 608 paths, 1 pixel a block
S1024_C4 = dict(maze=32, W=18, H=13, chunk=4, spp=1024, bounce=8, mirror=15, time=2,              # T = 16 384, ragged frame
                center=(-5.0, 0.0, 35.0), half_theta=2.4)


def expected_tail(mm, p, segments, k=TAIL_K_DEFAULT, cap_env=None):
    """(queued, deferred) the tail model predicts, or None when the queue overflows (then only its length is known).  Above
    spp 256 no flag but MM_FLAG_NO_TAIL turns the tail off: MM_FLAG_REGROUP and MM_FLAG_POOL_KERNEL run the default kernel."""
    if p.flags & mm.FLAG_NO_TAIL:
        return (0, 0)
    cap = tail_capacity(len(segments), p.spp, cap_env)
    queued, pixels = tail_model(segments, p.bounce_limit, k if cap else 0, p.spp)
    return (queued, pixels) if queued <= cap else None


def assert_tail(mm, got_tail, p, segments, what, k=TAIL_K_DEFAULT, cap_env=None):
    want = expected_tail(mm, p, segments, k, cap_env)
    if want is not None:
        assert got_tail == want, f"last_tail {got_tail} != model {want} (K {k}): {what}"
    else:                                                    # which warps win the queue is a race; how many entries it holds is not
        cap = tail_capacity(len(segments), p.spp, cap_env)
        queued, pixels = tail_model(segments, p.bounce_limit, k, p.spp)
        assert got_tail[0] == cap and got_tail[1] <= min(pixels, cap), \
            f"last_tail {got_tail} vs model {(queued, pixels)} with capacity {cap} (K {k}): {what}"


def check(mm, renderer, u, p, ch, ref, what, k=TAIL_K_DEFAULT, cap_env=None, debug_modes=(True, False)):
    """Renders with and without debug arrays into a zeroed mapped frame; image, counters, arrays and tail against ref."""
    tails = []
    for debug in debug_modes:
        got = gpu_render(mm, renderer, u, p, ch, debug)
        w = f"{what} debug {debug}"
        assert_same(got, ref if debug else (ref[0], ref[1], None), w)
        assert_tail(mm, got[3], p, ref[2]["segments"], w, k=k, cap_env=cap_env)
        tails.append(got[3])
    return tails


def n_paths_of(u, p):
    return (p.group_count or p.grid_x * p.grid_y) * u.chunk_width ** 2 * p.spp


_REF_CACHE = {}


def reference(mm, sc, noise, u, p, ch):
    """(image, counters, per-path arrays) of a dispatch from oracle/np_oracle.py, with the RGBA8 screen's quantisation applied.
    Of the flags only MM_FLAG_RCP_SLAB and MM_FLAG_SCREEN_RGBA8 change results; renders are cached on everything else."""
    from oracle import np_oracle

    q = mm.Params.from_buffer_copy(bytes(p))
    q.flags = p.flags & (mm.FLAG_RCP_SLAB | mm.FLAG_SCREEN_RGBA8)
    key = (id(sc), bytes(u), bytes(q), np.ascontiguousarray(ch).tobytes())
    if key not in _REF_CACHE:
        img, cnt, dbg = np_oracle.render(sc, noise, u, q, ch)
        if q.flags & mm.FLAG_SCREEN_RGBA8:                   # the transcription leaves the screen's quantisation to its caller
            img = np_oracle.quant8(img)
        _REF_CACHE[key] = (img, cnt, {k: np.ascontiguousarray(v) for k, v in dbg.items()})
    return _REF_CACHE[key]


def stitched_oracle_paths(mm, oracle, sc, noise, u, p, ch):
    """The per-path arrays of a dispatch of chunk c at spp s (512 or 1024) from the C++ oracle, which stops at spp 256.  A
    dispatch of chunk 2c at spp s/4 has the same T, group dims, texids and seeds, so path (group, flat) is the same path
    wherever its pixel is; its pixel is the chunk origin plus (j // 2c, j % 2c) for j = flat // (s/4), where the target's is
    the origin plus (i // c, i % c) for i = flat // s.  One render per j, with the chunk list shifted by the difference, gives
    every path of sub-range j on its own pixel.  The chunk origins must be at least 2c - 1."""
    c, s = int(u.chunk_width), int(p.spp)
    c2, s2, T = 2 * c, s // 4, c * c * s
    u2 = mm.Uniform.from_buffer_copy(bytes(u))
    u2.chunk_width = c2
    p2 = mm.Params.from_buffer_copy(bytes(p))
    p2.spp = s2
    sub = (np.arange(n_paths_of(u, p)) % T) // s2
    out = None
    for j in range(c2 * c2):
        i = j // 4
        ch2 = ch.copy()
        ch2["x"] = ch["x"].astype(np.int64) + (i // c - j // c2)
        ch2["y"] = ch["y"].astype(np.int64) + (i % c - j % c2)
        dbg = oracle.render(sc, noise, u2, p2, ch2, debug=True)[2]
        if out is None:
            out = {k: np.empty_like(v) for k, v in dbg.items()}
        for k in dbg:
            out[k][sub == j] = dbg[k][sub == j]
    return out


def restated_image(u, p, ch, radiance, rgba8):
    """The reference's per-pixel reduction (shaders.metal:344-366) restated from per-path radiance, pixel by pixel: tone-map,
    pairwise sums at strides 1, 2, 4 within each group of 8, the octets summed serially, divided by spp; stored at the
    pixel's position when inside the frame."""
    from oracle import np_oracle

    F = np.float32
    c, s = int(u.chunk_width), int(p.spp)
    W, H = int(u.view_width), int(u.view_height)
    count = p.group_count or p.grid_x * p.grid_y
    first, step = (p.group_first, p.group_step or 1) if p.group_count else (0, 1)
    tone = np.sqrt(np.fmax(np.asarray(radiance, F).reshape(count, c * c, s, 3), F(0.0)))
    img = np.zeros((H, W, 4), F)
    for k in range(count):
        g = first + k * step
        for pn in range(c * c):
            x, y = int(ch[g]["x"]) + pn // c, int(ch[g]["y"]) + pn % c
            if x >= W or y >= H:
                continue
            v = tone[k, pn].copy()
            for stride in (1, 2, 4):
                v[::2 * stride] = v[::2 * stride] + v[stride::2 * stride]
            acc = v[0].copy()
            for o in range(8, s, 8):
                acc = acc + v[o]
            img[y, x, :3] = acc / F(s)
            img[y, x, 3] = F(1.0)
    return np_oracle.quant8(img) if rgba8 else img


# ---- without a GPU -------------------------------------------------------------------------------------------------------------

NP_CASES = {
    # chunk 1 (the reference's one-pixel-per-threadgroup shape), 2 and 4; partial group ranges; frames that are not chunk
    # multiples; the RGBA8 screen.  Every case stays under 20 k paths.
    "spp1024_chunk1": dict(maze=32, W=5, H=3, chunk=1, spp=1024, bounce=8, mirror=15, time=3),
    "spp512_chunk1_part": dict(maze=32, W=9, H=5, chunk=1, spp=512, bounce=8, mirror=15, time=11, part=(3, 4, 10)),
    "spp512_chunk2_ragged": dict(maze=16, W=9, H=7, chunk=2, spp=512, bounce=6, mirror=15, time=4, part=(1, 3, 4)),
    "spp1024_chunk2_rgba8": dict(maze=32, W=5, H=4, chunk=2, spp=1024, bounce=8, mirror=15, flags=512, part=(0, 1, 4)),
    "spp512_chunk4_rgba8_ragged": dict(maze=32, W=11, H=9, chunk=4, spp=512, bounce=8, mirror=15, time=700, flags=512,
                                       center=(-5.0, 0.0, 35.0), half_theta=2.4, part=(1, 2, 2)),
    "spp1024_chunk4_part": dict(maze=10, W=8, H=9, chunk=4, spp=1024, bounce=5, mirror=15, part=(3, 1, 1)),
}


@pytest.mark.parametrize("name", sorted(NP_CASES))
def test_transcription_image_is_the_reduction_of_its_paths(mm, noise, scenes, name):
    """np_oracle's image at spp 512 and 1024 equals the reference's reduction restated from its own per-path radiance, and
    its counters count every path."""
    sc, u, p, ch = build_shape(mm, scenes, NP_CASES[name])
    n = n_paths_of(u, p)
    assert n <= 20_000, n
    img, cnt, dbg = reference(mm, sc, noise, u, p, ch)
    assert cnt["paths"] == n and len(dbg["radiance"]) == n
    want = restated_image(u, p, ch, dbg["radiance"], bool(p.flags & mm.FLAG_SCREEN_RGBA8))
    assert img.tobytes() == want.tobytes(), name
    assert np.count_nonzero(img[..., 3]) > 0


STITCH_CASES = {
    "spp1024_chunk1": dict(maze=32, W=7, H=3, chunk=1, spp=1024, bounce=8, mirror=15, time=3),
    "spp512_chunk1_part": dict(maze=32, W=9, H=5, chunk=1, spp=512, bounce=8, mirror=15, time=11, part=(3, 4, 10)),
    "spp1024_chunk2_part": dict(maze=16, W=9, H=7, chunk=2, spp=1024, bounce=6, mirror=15, time=4, part=(1, 3, 4)),
    "spp512_chunk2_rcp": dict(maze=32, W=6, H=6, chunk=2, spp=512, bounce=8, mirror=15, time=700, flags=64,
                              center=(-5.0, 0.0, 35.0), half_theta=2.4),
}


@pytest.mark.parametrize("name", sorted(STITCH_CASES))
def test_transcription_equals_the_oracle_path_by_path(mm, oracle, noise, scenes, name):
    """First hit, segments, mirror hits and radiance of every path at spp 512 and 1024: np_oracle against the C++ oracle's
    same paths, rendered at spp 128 / 256 (stitched_oracle_paths), with the RCP_SLAB arithmetic in one case."""
    sc, u, p, ch = build_shape(mm, scenes, STITCH_CASES[name])
    c = u.chunk_width
    ch = ch.copy()
    ch["x"] += 2 * c                                         # room for the shifted chunk lists (the pixels move, the paths do not care)
    ch["y"] += 2 * c
    got = stitched_oracle_paths(mm, oracle, sc, noise, u, p, ch)
    ref = reference(mm, sc, noise, u, p, ch)[2]
    for k in DBG_KEYS:
        assert got[k].tobytes() == np.ascontiguousarray(ref[k], dtype=got[k].dtype).tobytes(), (name, k)


def test_stitching_reproduces_the_oracle_where_it_reaches(mm, oracle, noise, scenes):
    """The stitch itself, at spp 256 from spp 64, where the C++ oracle renders both: same per-path arrays as its direct render."""
    sc, u, p, ch = build_shape(mm, scenes, dict(maze=32, W=6, H=4, chunk=1, spp=256, bounce=8, mirror=15, time=2))
    ch = ch.copy()
    ch["x"] += 2
    ch["y"] += 2
    got = stitched_oracle_paths(mm, oracle, sc, noise, u, p, ch)
    ref = oracle.render(sc, noise, u, p, ch, debug=True)[2]
    for k in DBG_KEYS:
        assert got[k].tobytes() == ref[k].tobytes(), k


REFUSED = [("spp2048", 2048, 1), ("spp3", 3, 1), ("chunk33_spp1024", 1024, 33)]


def refused_dispatch(mm, spp, chunk):
    u = mm.default_uniform(10, 66, 66, chunk)
    ch = mm.gen_chunks(66, 66, chunk)
    return u, mm.full_frame_params(u, spp=spp, bounce_limit=4, mirror_limit=15), ch


@pytest.mark.parametrize("name,spp,chunk", REFUSED)
def test_oracle_refuses_outside_the_limits(mm, oracle, noise, scenes, name, spp, chunk):
    """spp 2048 (a pixel would span blocks), spp 3 (not a power of two), chunk 33 at spp 1024 (T above 2^20)."""
    u, p, ch = refused_dispatch(mm, spp, chunk)
    with pytest.raises(RuntimeError, match=str(ERR_UNSUPPORTED)):
        oracle.render(scenes(10), noise, u, p, ch)


def test_largest_group_is_two_to_the_twenty():
    """chunk 32 at spp 1024 is T = 2^20, the largest virtual group (rendered on the GPU below); chunk 33 is past it."""
    assert 32 * 32 * 1024 == 1 << 20 and 33 * 33 * 1024 > 1 << 20


def _sass_counts():
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


def test_1024_thread_kernels_keep_the_packed_fp32_mix():
    """The 1024-thread kernels run the same traversal as their 64- and 256-thread siblings: FADD2 : FMUL2 : FFMA2 =
    60 : 60 : 108 for trace_kernel<CNT, DBG, 1024> and views_wide_kernel, 44 : 44 : 132 for trace_ytab_wide_kernel and
    views_ytab_wide_kernel, for each of the three CNT / DBG variants kernel_ptr selects."""
    counts = _sass_counts()
    want = {"12trace_kernel": (60, 60, 108), "17views_wide_kernel": (60, 60, 108),
            "22trace_ytab_wide_kernel": (44, 44, 132), "22views_ytab_wide_kernel": (44, 44, 132)}
    for kernel, mix in want.items():
        huge = {n: tuple(c) for n, c in counts.items() if kernel in n and (kernel != "12trace_kernel" or "Li1024E" in n)}
        assert sorted(n.split(kernel)[1][:9] for n in huge) == ["ILb0ELb0E", "ILb1ELb0E", "ILb1ELb1E"], huge
        assert all(c == mix for c in huge.values()), huge
    assert not any("trace_kernel_rg" in n and "Li1024E" in n for n in counts)   # regroup falls back above spp 256


# ---- on the GPU: refusals, shape and sizes ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name,spp,chunk", REFUSED)
def test_library_refuses_outside_the_limits(mm, noise, scenes, renderer, name, spp, chunk):
    renderer.upload_scene(scenes(10), noise)
    u, p, ch = refused_dispatch(mm, spp, chunk)
    with pytest.raises(mm.MMError) as e:
        renderer.render(u, p, ch)
    assert e.value.code == ERR_UNSUPPORTED


@pytest.mark.gpu
def test_scene_info_reports_the_1024_thread_block(mm, oracle, noise, scenes, renderer):
    """One 1024-thread block an SM at spp 512 and 1024, with and without the y-table; spp 256 keeps its 256 x 4."""
    sc = scenes(32)
    renderer.upload_scene(sc, noise)
    for spp, bt, per_sm in ((256, 256, 4), (512, 1024, 1), (1024, 1024, 1)):
        for flags in (0, mm.FLAG_NO_Y_TABLE):
            u = mm.default_uniform(32, 4, 2, 1, 1)
            p = mm.full_frame_params(u, spp=spp, bounce_limit=8, mirror_limit=15, flags=flags)
            ch = mm.gen_chunks(4, 2, 1)
            got = gpu_render(mm, renderer, u, p, ch, False)
            info = renderer.scene_info()
            assert (info["block_threads"], info["blocks_per_sm"]) == (bt, per_sm), (spp, flags, info)
            assert bool(info["y_table"]) == (flags == 0), (spp, flags, info)
            assert info["smem_bytes"] == 12 * bt + (bt // 32) * info["y_table"] * 256, (spp, flags, info)
            ref = oracle.render(sc, noise, u, p, ch) if spp <= 256 else reference(mm, sc, noise, u, p, ch)
            assert_same(got, (*ref[:2], None), f"spp {spp} flags {flags}")


@pytest.mark.gpu
def test_largest_group_chunk32_spp1024(mm, oracle, noise, scenes, renderer):
    """T = 2^20: one virtual group of 32 x 32768 threads, 1024 blocks of one pixel each, on a ragged 40 x 33 frame."""
    c = dict(maze=16, W=40, H=33, chunk=32, spp=1024, bounce=4, mirror=15, time=1, part=(0, 1, 1))
    sc, u, p, ch = build_shape(mm, scenes, c)
    renderer.upload_scene(sc, noise)
    ref = reference(mm, sc, noise, u, p, ch)
    check(mm, renderer, u, p, ch, ref, "chunk 32 spp 1024", debug_modes=(True,))


# ---- on the GPU: every flag ------------------------------------------------------------------------------------------------

FLAGS = ["default", "COUNTERS", "FORCE_LITERAL", "RCP_SLAB", "GENERAL_RECTS", "NO_Y_TABLE", "NO_TAIL", "SCREEN_RGBA8",
         "NO_ZERO_COPY", "POOL_KERNEL", "REGROUP"]


@pytest.mark.gpu
@pytest.mark.parametrize("flag", FLAGS)
def test_every_flag_matches_reference(mm, oracle, noise, scenes, renderer, flag):
    """Each flag at spp 512 and 1024, chunk 1.  POOL_KERNEL and REGROUP run the default kernel, tail on."""
    for shape in (S512, S1024):
        sc, u, p, ch = build_shape(mm, scenes, shape)
        renderer.upload_scene(sc, noise)
        p = with_flags(mm, p, 0 if flag == "default" else getattr(mm, "FLAG_" + flag))
        ref = reference(mm, sc, noise, u, p, ch)
        tails = check(mm, renderer, u, p, ch, ref, f"{flag} spp {p.spp}")
        assert renderer.scene_info()["block_threads"] == 1024
        if flag != "NO_TAIL":
            assert tails[0][0] > 0, f"{flag} spp {p.spp}: no path queued"


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 8, 32])
def test_tail_k_matches_model(mm, oracle, noise, scenes, renderer, monkeypatch, k):
    for shape in (S512, S1024, S1024_C4):
        sc, u, p, ch = build_shape(mm, scenes, shape)
        renderer.upload_scene(sc, noise)
        ref = reference(mm, sc, noise, u, p, ch)
        monkeypatch.setenv("MM_TAIL_K", str(k))
        check(mm, renderer, u, p, ch, ref, f"K {k} spp {p.spp} chunk {u.chunk_width}", k=k)


@pytest.mark.gpu
def test_tail_cap_cuts_the_queue_mid_launch(mm, oracle, noise, scenes, renderer, monkeypatch):
    """MM_TAIL_CAP at 1, a third and all but one of what the trigger queues, and exactly that: paths past the cap trace on in
    their warps with their pixel's other samples still deferred, and the image stays the reference render."""
    for shape in (S512, S1024):
        sc, u, p, ch = build_shape(mm, scenes, shape)
        renderer.upload_scene(sc, noise)
        ref = reference(mm, sc, noise, u, p, ch)
        queued, _ = tail_model(ref[2]["segments"], p.bounce_limit, TAIL_K_DEFAULT, p.spp)
        assert queued > 3, (shape, queued)
        for cap in (1, queued // 3, queued - 1, queued):
            monkeypatch.setenv("MM_TAIL_CAP", str(cap))
            tails = check(mm, renderer, u, p, ch, ref, f"cap {cap} of {queued}, spp {p.spp}", cap_env=cap)
            assert tails[0][0] == cap


# ---- on the GPU: every output route ----------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_host_frames_zero_copy_and_staged(mm, oracle, noise, scenes, renderer):
    """The mapped pinned frame (zero-copy stores), the same with NO_ZERO_COPY (DMA copy) and a pageable frame (staged copy)."""
    for shape in (S512, S1024_C4):
        sc, u, p, ch = build_shape(mm, scenes, shape)
        renderer.upload_scene(sc, noise)
        ref = reference(mm, sc, noise, u, p, ch)[0]
        H, W = int(u.view_height), int(u.view_width)
        for flags in (0, mm.FLAG_NO_ZERO_COPY):
            hf = mm.HostFrame(H, W)
            try:
                renderer.render(u, with_flags(mm, p, flags), ch, out=hf.array)
                assert hf.array.tobytes() == ref.tobytes(), (shape, flags)
            finally:
                hf.close()
        pageable = np.zeros((H, W, 4), np.float32)
        renderer.render(u, p, ch, out=pageable)
        assert pageable.tobytes() == ref.tobytes(), shape


@pytest.mark.gpu
def test_device_frame_tiles_and_peer_frames_in_partial_dispatches(mm, oracle, noise, scenes):
    """Three interleaved ranks at spp 1024 (chunk 1 and chunk 2): each rank into a device frame and tiles at once, tiles
    scattered with mm_scatter_tiles_device, and through mm_render_peers_device into two frames; each rank's tail against the
    model of the reference render of that rank."""
    import torch

    dev = torch.device("cuda", 0)
    for c in (dict(S1024, W=17, H=11), dict(maze=32, W=13, H=10, chunk=2, spp=1024, bounce=8, mirror=15, time=6)):
        sc, u, p, ch = build_shape(mm, scenes, c)
        r = mm.Renderer(0)
        r.upload_scene(sc, noise)
        H, W, ppc = c["H"], c["W"], c["chunk"] ** 2
        n_groups = p.grid_x * p.grid_y
        full_ref = np.zeros((H, W, 4), dtype=np.float32)
        image, scattered = (torch.zeros((H, W, 4), dtype=torch.float32, device=dev) for _ in range(2))
        peers = [torch.zeros((H, W, 4), dtype=torch.float32, device=dev) for _ in range(2)]
        r.set_chunks(ch)
        for rank in range(3):
            q = mm.Params.from_buffer_copy(bytes(p))
            q.group_first, q.group_step, q.group_count = mm.tile_partition(n_groups, rank, 3)
            ref = reference(mm, sc, noise, u, q, ch)
            written = ref[0][..., 3] != 0
            full_ref[written] = ref[0][written]
            what = f"{c} rank {rank}"
            tiles = torch.zeros((q.group_count, ppc, 4), dtype=torch.float32, device=dev)
            r.render_device(u, q, image_ptr=image.data_ptr(), tiles_ptr=tiles.data_ptr())
            assert_tail(mm, r.last_tail(), q, ref[2]["segments"], what + " render_device")
            r.scatter_tiles_device(u, q, tiles.data_ptr(), scattered.data_ptr())
            r.render_peers_device(u, q, [f.data_ptr() for f in peers])
            assert_tail(mm, r.last_tail(), q, ref[2]["segments"], what + " render_peers_device")
            r.sync()
        torch.cuda.synchronize()
        for name, t in (("image", image), ("scattered tiles", scattered), ("peer 0", peers[0]), ("peer 1", peers[1])):
            assert t.cpu().numpy().tobytes() == full_ref.tobytes(), f"{c}: {name}"
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_views", [2, 3])
def test_render_views_equal_reference_and_single_renders(mm, oracle, noise, scenes, n_views):
    """K distinct poses at spp 1024, chunk 1, in one launch: each view against the reference render (image and per-path arrays) and
    against mm_render of that view alone (image, counters summed, debug arrays, tail summed where no queue fills)."""
    from test_views import fresh, poses, shuffled, singles, split_debug, summed

    sc = scenes(32)
    W, H = 10, 6
    us = poses(mm, n_views, 32, W, H, seed=50 + n_views, chunk=1)
    p = mm.full_frame_params(us[0], spp=1024, bounce_limit=8, flags=mm.FLAG_COUNTERS)
    lists = [shuffled(mm.gen_chunks(W, H, 1), 70 + v) for v in range(n_views)]
    frames, cnts, dbgs, tails = singles(mm, sc, noise, us, p, lists, debug=True)
    models = []
    r = fresh(mm, sc, noise)
    outs = [mm.HostFrame(H, W) for _ in range(n_views)]
    _, cnt, dbg = r.render_views(us, p, lists, outs=outs, debug=True)
    per_view = split_debug(dbg, n_views)
    for v in range(n_views):
        ref, _, rdbg = reference(mm, sc, noise, us[v], p, lists[v])
        assert outs[v].array.tobytes() == ref.tobytes() == frames[v].tobytes(), v
        for k in DBG_KEYS:
            assert per_view[v][k].tobytes() == dbgs[v][k].tobytes(), (v, k)
            assert per_view[v][k].tobytes() == np.ascontiguousarray(rdbg[k], dtype=per_view[v][k].dtype).tobytes(), (v, k)
        assert_tail(mm, tails[v], p, rdbg["segments"], f"view {v} alone")
        models.append(tail_model(rdbg["segments"], p.bounce_limit, TAIL_K_DEFAULT, p.spp))
    assert cnt == summed(cnts)
    # One pixel a block: no warp or block spans two views, so the batch queues what the views queue alone.  The batch's queue
    # holds an eighth of all views' paths (plus 1024); past that, which warps win its entries is a race.
    queued, pixels = (sum(m[0] for m in models), sum(m[1] for m in models))
    cap = tail_capacity(n_views * len(rdbg["segments"]), p.spp)
    got = r.last_tail()
    assert got == (queued, pixels) if queued <= cap else (got[0] == cap and got[1] <= pixels), (got, queued, pixels, cap)
    for o in outs:
        o.close()
    r.close()


# ---- on the GPU: other scenes, context reuse, random draws ---------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name,spp", [("walls_9", 512), ("tilted_0", 512), ("walls_8", 1024)])
def test_general_scenes(mm, oracle, noise, renderer, name, spp):
    """9 y-intervals (no y-table), a tilted cloud, and 8 y-intervals at spp 1024: the largest y-table, 32 warps x 8 x 256 B
    beside the 12 KB of reduction scratch."""
    sc = general_scene(mm, name)
    renderer.upload_scene(sc, noise)
    u, p, ch = general_dispatch(mm, sc, spp, W=12, H=7, chunk=2)
    ref = reference(mm, sc, noise, u, p, ch)
    check(mm, renderer, u, p, ch, ref, f"{name} spp {spp}")
    info = renderer.scene_info()
    assert info["block_threads"] == 1024
    assert info["smem_bytes"] == 12 * 1024 + 32 * info["y_table"] * 256
    if name == "walls_8":
        assert info["y_table"] == 8 and info["smem_bytes"] == 77824


@pytest.mark.gpu
def test_one_context_alternates_block_shapes_and_tail_buffers(mm, oracle, noise, scenes):
    """spp 16 (64-thread blocks, a large frame) -> 1024 (1024-thread blocks, 12 304-B deferred-pixel slots: the slot buffer
    regrows) -> 64 -> 1024 again (buffers reused) on one context."""
    seq = [dict(maze=32, W=320, H=180, chunk=4, spp=16, bounce=8, mirror=15),
           S1024,
           dict(maze=32, W=160, H=96, chunk=4, spp=64, bounce=8, mirror=15, time=3),
           dict(S1024, time=21)]
    r = mm.Renderer(0)
    for i, c in enumerate(seq):
        sc, u, p, ch = build_shape(mm, scenes, c)
        r.upload_scene(sc, noise)
        ref = oracle.render(sc, noise, u, p, ch, debug=True) if c["spp"] <= 256 else reference(mm, sc, noise, u, p, ch)
        tails = check(mm, r, u, p, ch, ref, f"render {i} of the sequence, {c}")
        assert tails[0][0] > 0, c
        assert r.scene_info()["block_threads"] == (1024 if c["spp"] > 256 else 64)
    r.close()


DRAW_SEED = int(os.environ.get("MM_HIGH_SPP_SEED", "20261022"))
DRAWS = int(os.environ.get("MM_HIGH_SPP_DRAWS", "16"))
MAX_PATHS = 200_000
DRAW_FLAGS = ["FLAG_FORCE_LITERAL", "FLAG_GENERAL_RECTS", "FLAG_RCP_SLAB", "FLAG_COUNTERS", "FLAG_SCREEN_RGBA8", "FLAG_NO_TAIL",
              "FLAG_NO_Y_TABLE", "FLAG_REGROUP", "FLAG_POOL_KERNEL"]


def draw_dispatch(i):
    """Draw i of the new dispatch space: spp 512 or 1024, chunk 1..16, group range, flags, pose, time, MM_TAIL_K."""
    rng = np.random.default_rng([DRAW_SEED, i])
    maze = int(rng.choice([10, 16, 32, 64]))
    spp = int(rng.choice([512, 1024]))
    chunk = int(rng.choice([1, 1, 1, 2, 2, 3, 4, 8, 16]))
    T = chunk * chunk * spp
    max_groups = max(1, MAX_PATHS // T)
    gx = int(rng.integers(1, min(max_groups, 24) + 1))
    gy = int(rng.integers(1, max(1, min(max_groups // gx, 24)) + 1))
    W = gx * chunk + (int(rng.integers(0, chunk)) if rng.random() < 0.5 else 0)
    H = gy * chunk + (int(rng.integers(0, chunk)) if rng.random() < 0.5 else 0)
    half = 5.0 * maze
    cx, cz = (-half + 10.0 * int(rng.integers(0, maze)) + 5.0, -half + 10.0 * int(rng.integers(0, maze)) + 5.0) if rng.random() < 0.7 \
        else (float(rng.uniform(-half, half)), float(rng.uniform(-half, half)))
    time = int(rng.integers(0, 1000)) if rng.random() < 0.6 else int(rng.integers(0, 1 << 26))
    n_groups = gx * gy
    if rng.random() < 0.5:
        world = int(rng.integers(1, 5))
        r = int(rng.integers(0, min(world, n_groups)))
        part = (r, world, (n_groups - r + world - 1) // world)
    else:
        step = int(rng.integers(1, 4))
        first = int(rng.integers(0, n_groups))
        part = (first, step, int(rng.integers(1, (n_groups - 1 - first) // step + 2)))
    flags = [f for f in DRAW_FLAGS if rng.random() < 0.2]
    return dict(maze=maze, W=W, H=H, chunk=chunk, spp=spp, bounce=int(rng.integers(1, 13)), mirror=int(rng.integers(0, 16)),
                time=time, center=(cx, float(rng.uniform(-7.0, 1.5)), cz), half_theta=float(rng.uniform(0.0, np.pi)), part=part,
                flag_names=flags, tail_k=int(rng.integers(0, 33)))


def build_draw(mm, scenes, c):
    sc, u, p, ch = build_shape(mm, scenes, c)
    p.flags = sum(getattr(mm, f) for f in c["flag_names"])
    return sc, u, p, ch


def test_draws_are_legal_and_cover_the_space(mm, scenes):
    draws = [draw_dispatch(i) for i in range(DRAWS)]
    for c in draws:
        T = c["chunk"] ** 2 * c["spp"]
        assert (T <= 32 or T % 32 == 0) and T <= 1 << 20 and c["part"][2] * T <= max(MAX_PATHS, T), c
    assert {c["spp"] for c in draws} == {512, 1024} and 1 in {c["chunk"] for c in draws}


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(DRAWS))
def test_random_dispatch_matches_reference(mm, oracle, noise, scenes, renderer, monkeypatch, i):
    c = draw_dispatch(i)
    sc, u, p, ch = build_draw(mm, scenes, c)
    renderer.upload_scene(sc, noise)
    ref = reference(mm, sc, noise, u, p, ch)
    monkeypatch.setenv("MM_TAIL_K", str(c["tail_k"]))
    check(mm, renderer, u, p, ch, ref, f"draw {i}: {c}", k=c["tail_k"])
    assert ref[1]["paths"] == n_paths_of(u, p)
    assert set(ref[1]) >= set(COUNTER_KEYS)
