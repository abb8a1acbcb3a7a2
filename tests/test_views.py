"""Several camera views in one launch (mm_render_views / mm_present_views): every view equals what mm_render / mm_present give
for that view alone, bit for bit; the view screens are the context's own and persist like mm_render's screen."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from cases import build_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32
DBG_KEYS = ("first_hit", "segments", "mirror_hits", "radiance")


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


def test_views_kernels_keep_the_packed_fp32_mix():
    """The multi-view kernels run the same traversal instantiations as the single-view ones: views_kernel FADD2 : FMUL2 : FFMA2 =
    60 : 60 : 108 like trace_kernel, views_ytab_kernel 44 : 44 : 132 like trace_ytab_kernel, and every views_tail_kernel the mix of
    the trace_tail_kernel with the same template arguments.  A contracted, dropped or extra packed instruction changes the counts."""
    counts = _sass_counts()
    plain = {n: tuple(c) for n, c in counts.items() if "12views_kernel" in n}
    ytab = {n: tuple(c) for n, c in counts.items() if "17views_ytab_kernel" in n}
    tails = {n: tuple(c) for n, c in counts.items() if "17views_tail_kernel" in n}
    assert len(plain) == 6 and len(ytab) == 6 and len(tails) == 6
    assert all(c == (60, 60, 108) for c in plain.values()), plain
    assert all(c == (44, 44, 132) for c in ytab.values()), ytab
    single_tails = {n.split("trace_tail_kernel")[1].split("EEEv")[0]: tuple(c) for n, c in counts.items() if "trace_tail_kernel" in n}
    for n, c in tails.items():
        assert c == single_tails[n.split("views_tail_kernel")[1].split("EEEv")[0]], (n, c)
    assert any("blur_views_kernel" in n for n in counts)


def test_views_entry_points_fail_cleanly_without_a_gpu(mm):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = mm.load_library()
    u, p = mm.default_uniform(10, 32, 32), mm.Params(spp=1, bounce_limit=1, mirror_limit=15, grid_x=8, grid_y=8)
    ch = mm.gen_chunks(32, 32, 4)
    assert lib.mm_render_views(None, C.byref(u), 1, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == -1
    assert lib.mm_render_views_async(None, C.byref(u), 1, C.byref(p), ch.ctypes.data, len(ch), None, None) == -1
    assert lib.mm_render_views(None, None, 0, None, None, 0, None, None, None) == -1
    assert lib.mm_present_views(None, 0, None) == -1
    assert lib.mm_present_views(None, 1, None) == -1
    with pytest.raises(mm.MMError):
        mm.Renderer(0)


# ---- on the GPU -------------------------------------------------------------------------------------------------------------

def poses(mm, n, maze, W, H, seed, chunk=4):
    """n views at seeded cell centres with seeded yaws and times."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        i, j = (int(x) for x in rng.integers(-(maze // 2), maze // 2, size=2))
        out.append(mm.default_uniform(maze, W, H, chunk, int(rng.integers(0, 1000)), camera_center=(10.0 * i + 5.0, 0.0, 10.0 * j + 5.0),
                                      half_theta=float(rng.uniform(0.0, math.pi))))
    return out


def shuffled(chunks, seed):
    return chunks[np.random.default_rng(seed).permutation(len(chunks))].copy()


def copy_params(mm, p, **kw):
    q = mm.Params.from_buffer_copy(bytes(p))
    for k, v in kw.items():
        setattr(q, k, v)
    return q


def summed(cnts):
    out = {k: sum(c[k] for c in cnts) for k in cnts[0]}
    out["max_stack"] = max(c["max_stack"] for c in cnts)
    return out


def fresh(mm, sc, noise):
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    return r


def singles(mm, sc, noise, us, p, chunk_lists, debug=False):
    """Every view rendered alone by mm_render, each on a fresh context (a zero screen): (frames, counters, debug dicts, tails)."""
    frames, cnts, dbgs, tails = [], [], [], []
    for u, ch in zip(us, chunk_lists):
        r = fresh(mm, sc, noise)
        img, cnt, dbg = r.render(u, p, ch, debug=debug)
        frames.append(img); cnts.append(cnt); dbgs.append(dbg); tails.append(r.last_tail())
        r.close()
    return frames, cnts, dbgs, tails


def split_debug(dbg, n):
    return [{k: np.split(dbg[k], n)[v] for k in DBG_KEYS} for v in range(n)]


@pytest.mark.gpu
def test_one_view_equals_mm_render_on_the_full_frame(mm, noise, scenes):
    """K = 1 on the 1080p x 16 spp x 8 bounces 32x32 frame: frame, counters, the four debug arrays and the straggler tail."""
    sc = scenes(32)
    u = mm.default_uniform(32, 1920, 1080, 4)
    p = mm.full_frame_params(u, spp=16, bounce_limit=8, flags=mm.FLAG_COUNTERS)
    ch = mm.gen_chunks(1920, 1080, 4)
    r = fresh(mm, sc, noise)
    img, cnt, dbg = r.render(u, p, ch, debug=True)
    tail = r.last_tail()
    out = np.empty_like(img)
    _, vcnt, vdbg = r.render_views([u], p, [ch], outs=[out], debug=True)
    assert tail[0] > 0
    assert r.last_tail() == tail
    assert out.tobytes() == img.tobytes()
    assert vcnt == cnt
    for k in DBG_KEYS:
        assert vdbg[k].tobytes() == dbg[k].tobytes(), k
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_views", [2, 3, 8])
def test_distinct_poses_equal_the_oracle_view_by_view(mm, oracle, noise, scenes, n_views):
    sc = scenes(16)
    us = poses(mm, n_views, 16, 128, 96, seed=n_views)
    p = mm.full_frame_params(us[0], spp=8, bounce_limit=8, flags=mm.FLAG_COUNTERS)
    base = mm.gen_chunks(128, 96, 4)
    lists = [shuffled(base, 100 + v) for v in range(n_views)]
    r = fresh(mm, sc, noise)
    outs = [np.empty((96, 128, 4), F) for _ in range(n_views)]
    _, cnt, dbg = r.render_views(us, p, lists, outs=outs, debug=True)
    per_view = split_debug(dbg, n_views)
    for v in range(n_views):
        ref, _, rdbg = oracle.render(sc, noise, us[v], p, lists[v], debug=True)
        assert outs[v].tobytes() == ref.tobytes(), v
        for k in DBG_KEYS:
            assert per_view[v][k].tobytes() == np.ascontiguousarray(rdbg[k], dtype=per_view[v][k].dtype).tobytes(), (v, k)
    _, cnts, _, _ = singles(mm, sc, noise, us, p, lists)
    assert cnt == summed(cnts)
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rgba8", [False, True])
def test_flythrough_with_present_views_equals_oracle_and_separate_renderers(mm, oracle, noise, scenes, rgba8):
    """3 views x 4 frames, a ChunkBag per view, 1/8 of the screen per frame, then present_views: against the oracle + the blur model
    and against three separate Renderers running render + present / present_rgba8."""
    from oracle import np_oracle

    sc = scenes(16)
    W, H, n = 128, 96, 3
    us = poses(mm, n, 16, W, H, seed=7)
    flags = mm.FLAG_SCREEN_RGBA8 if rgba8 else 0
    p = mm.Params(spp=8, bounce_limit=8, mirror_limit=15, grid_x=16, grid_y=6, flags=flags)   # 96 of 768 chunks
    bags = [mm.ChunkBag(W, H, 4, seed=20 + v) for v in range(n)]
    r = fresh(mm, sc, noise)
    seps = [fresh(mm, sc, noise) for _ in range(n)]
    hfs = [mm.HostFrame(H, W) for _ in range(n)]
    model = [np.zeros((H, W, 4), F) for _ in range(n)]
    nbytes = H * W * (4 if rgba8 else 16)
    for f in range(4):
        for u in us:
            u.time = 10 * f + 1
        lists = [b.next(96) for b in bags]
        r.render_views(us, p, lists)
        r.present_views(hfs, rgba8=rgba8)
        r.wait_present()
        for v in range(n):
            seps[v].render(us[v], p, lists[v])
            sep = np.empty((H, W, 4), F)
            sep8 = np.empty((H, W, 4), np.uint8)
            if rgba8:
                seps[v].present_rgba8(sep, sep8)
            else:
                seps[v].present(sep)
            oracle.render(sc, noise, us[v], p, lists[v], out=model[v])
            model[v] = np_oracle.present_blur(model[v], rgba8=rgba8)
            got = hfs[v].array.reshape(-1).view(np.uint8)[:nbytes]
            if rgba8:
                texels = np.rint(model[v] * F(255.0)).astype(np.uint8)
                assert got.tobytes() == texels.tobytes() == sep8.tobytes(), (f, v)
                assert sep.tobytes() == model[v].tobytes(), (f, v)
            else:
                assert got.tobytes() == model[v].tobytes() == sep.tobytes(), (f, v)
    for x in seps + [r]:
        x.close()
    for h in hfs:
        h.close()


FLAG_CASES = ["COUNTERS", "FORCE_LITERAL", "RCP_SLAB", "GENERAL_RECTS", "NO_Y_TABLE", "NO_TAIL", "NO_ZERO_COPY", "SCREEN_RGBA8"]


@pytest.mark.gpu
@pytest.mark.parametrize("flag", FLAG_CASES)
def test_each_flag_gives_the_single_view_bits(mm, oracle, noise, scenes, flag):
    sc = scenes(16)
    us = poses(mm, 3, 16, 128, 96, seed=31)
    p = mm.full_frame_params(us[0], spp=8, bounce_limit=8, flags=getattr(mm, "FLAG_" + flag) | mm.FLAG_COUNTERS)
    lists = [shuffled(mm.gen_chunks(128, 96, 4), 40 + v) for v in range(3)]
    frames, cnts, dbgs, tails = singles(mm, sc, noise, us, p, lists, debug=True)
    r = fresh(mm, sc, noise)
    hfs = [mm.HostFrame(96, 128) for _ in range(3)]
    _, cnt, dbg = r.render_views(us, p, lists, outs=hfs, debug=True)
    per_view = split_debug(dbg, 3)
    for v in range(3):
        assert hfs[v].array.tobytes() == frames[v].tobytes(), v
        for k in DBG_KEYS:
            assert per_view[v][k].tobytes() == dbgs[v][k].tobytes(), (v, k)
        if flag == "RCP_SLAB":
            assert frames[v].tobytes() == oracle.render(sc, noise, us[v], p, lists[v])[0].tobytes(), v
    assert cnt == summed(cnts)
    if flag == "NO_TAIL":
        assert r.last_tail() == (0, 0)
    for h in hfs:
        h.close()
    r.close()


@pytest.mark.gpu
def test_pool_and_regroup_flags_are_unsupported(mm, noise, scenes):
    sc = scenes(10)
    us = poses(mm, 2, 10, 32, 32, seed=1)
    ch = mm.gen_chunks(32, 32, 4)
    r = fresh(mm, sc, noise)
    for flag in (mm.FLAG_POOL_KERNEL, mm.FLAG_REGROUP):
        p = mm.full_frame_params(us[0], spp=8, bounce_limit=4, flags=flag)
        with pytest.raises(mm.MMError) as e:
            r.render_views(us, p, [ch, ch])
        assert e.value.code == -5
    r.close()


@pytest.mark.gpu
def test_tail_of_the_batch_is_the_sum_when_no_warp_spans_two_views(mm, noise, scenes):
    """T = 16 px x 16 spp = 256 paths per group: every view's paths fill whole blocks, so each warp's and block's queueing is what
    the single-view render does and, as long as no queue fills, mm_last_tail of the batch is the sum.  The views share the start
    pose at different times and yaws (a pose facing many mirrors can queue more than the eighth of its paths a single-view
    queue holds, and the batch's larger queue would then take what the single one leaves in its warps)."""
    sc = scenes(32)
    us = [mm.default_uniform(32, 256, 128, 4, time=7 * v + 1, half_theta=0.9 + 0.2 * v) for v in range(4)]
    p = mm.full_frame_params(us[0], spp=16, bounce_limit=8)
    lists = [shuffled(mm.gen_chunks(256, 128, 4), 60 + v) for v in range(4)]
    frames, cnts, _, tails = singles(mm, sc, noise, us, p, lists)
    view_paths = len(lists[0]) * 16 * 16
    assert all(0 < t[0] < view_paths // 8 + 1024 for t in tails), tails   # no single-view queue filled
    r = fresh(mm, sc, noise)
    outs = [np.empty((128, 256, 4), F) for _ in range(4)]
    _, cnt, _ = r.render_views(us, p, lists, outs=outs)
    queued, pixels = r.last_tail()
    assert (queued, pixels) == (sum(t[0] for t in tails), sum(t[1] for t in tails))
    assert queued < 4 * view_paths // 8 + 1024               # nor did the batch's
    assert all(o.tobytes() == f.tobytes() for o, f in zip(outs, frames))
    assert cnt == summed(cnts)
    r.close()


@pytest.mark.gpu
def test_warps_that_straddle_views(mm, noise, scenes):
    """spp 1, chunk 1 and a 7 x 5 grid: 35 paths per view, so warps and blocks hold paths of two or three views."""
    sc = scenes(10)
    us = poses(mm, 5, 10, 24, 16, seed=9, chunk=1)
    p = mm.Params(spp=1, bounce_limit=8, mirror_limit=15, grid_x=7, grid_y=5, flags=mm.FLAG_COUNTERS)
    base = mm.gen_chunks(24, 16, 1)
    lists = [shuffled(base, 80 + v)[:35] for v in range(5)]
    frames, cnts, dbgs, _ = singles(mm, sc, noise, us, p, lists, debug=True)
    r = fresh(mm, sc, noise)
    outs = [np.empty((16, 24, 4), F) for _ in range(5)]
    _, cnt, dbg = r.render_views(us, p, lists, outs=outs, debug=True)
    for v, d in enumerate(split_debug(dbg, 5)):
        assert outs[v].tobytes() == frames[v].tobytes(), v
        for k in DBG_KEYS:
            assert d[k].tobytes() == dbgs[v][k].tobytes(), (v, k)
    assert cnt == summed(cnts)
    r.close()


@pytest.mark.gpu
def test_outputs_partial_chunks_and_screen_lifetime(mm, noise, scenes):
    sc, u0, p, ch = build_case(mm, "yaw", scenes)
    H, W = int(u0.view_height), int(u0.view_width)
    us = poses(mm, 3, 16, W, H, seed=3)
    half = copy_params(mm, p, grid_x=16, grid_y=6)                    # 96 of 768 chunks
    lists = [shuffled(ch, 90 + v)[:96] for v in range(3)]
    frames, _, _, _ = singles(mm, sc, noise, us, half, lists)
    r = fresh(mm, sc, noise)
    # views mixing a pinned HostFrame (zero-copy), a pageable array and None; partial lists touch only their chunks
    hf, pageable = mm.HostFrame(H, W), np.full((H, W, 4), 7.0, F)
    r.render_views(us, half, lists, outs=[hf, pageable, None])
    assert hf.array.tobytes() == frames[0].tobytes()
    assert pageable.tobytes() == frames[1].tobytes()          # the whole view screen: zero outside the chunks rendered
    got = [mm.HostFrame(H, W) for _ in range(3)]
    r.present_views(None)                                      # blur only
    r.wait_present()
    from oracle import np_oracle
    r.present_views(got)
    r.wait_present()
    for v in range(3):
        assert got[v].array.tobytes() == np_oracle.present_blur(np_oracle.present_blur(frames[v])).tobytes(), v
    # mm_render / mm_present on the same context leave the view screens alone, and the reverse holds too
    single = np.empty((H, W, 4), F)
    r.render(u0, p, ch, out=single)
    ref_single = single.copy()
    blurred = np.empty((H, W, 4), F)
    r.present(blurred)
    assert blurred.tobytes() == np_oracle.present_blur(ref_single).tobytes()
    r.render_views(us, half, lists)                            # accumulates on the twice-blurred view screens
    r.present_views(got)
    r.wait_present()
    for v in range(3):
        want = np_oracle.present_blur(np_oracle.present_blur(frames[v]))
        fresh_px = frames[v][..., 3] != 0                      # the rendered chunks' pixels (alpha 1), re-rendered alike
        want[fresh_px] = frames[v][fresh_px]
        assert got[v].array.tobytes() == np_oracle.present_blur(want).tobytes(), v
    again = np.empty((H, W, 4), F)
    r.present(again)
    assert again.tobytes() == np_oracle.present_blur(np_oracle.present_blur(ref_single)).tobytes()
    # a changed K, or a changed view size, restarts the view screens at zero
    two = [np.empty((H, W, 4), F) for _ in range(2)]
    r.render_views(us[:2], half, lists[:2], outs=two)
    assert two[0].tobytes() == frames[0].tobytes() and two[1].tobytes() == frames[1].tobytes()
    small = [mm.default_uniform(16, 64, 48, 4, 5) for _ in range(2)]
    sp = mm.Params(spp=8, bounce_limit=8, mirror_limit=15, grid_x=4, grid_y=4)
    sl = [mm.gen_chunks(64, 48, 4)[:16], mm.gen_chunks(64, 48, 4)[16:32]]
    sf, _, _, _ = singles(mm, sc, noise, small, sp, sl)
    so = [np.empty((48, 64, 4), F) for _ in range(2)]
    r.render_views(small, sp, sl, outs=so)
    assert so[0].tobytes() == sf[0].tobytes() and so[1].tobytes() == sf[1].tobytes()
    for h in [hf] + got:
        h.close()
    r.close()


@pytest.mark.gpu
def test_group_range_selects_the_same_groups_in_every_view(mm, noise, scenes):
    sc = scenes(16)
    us = poses(mm, 3, 16, 128, 96, seed=13)
    p = mm.full_frame_params(us[0], spp=8, bounce_limit=8, flags=mm.FLAG_COUNTERS)
    lists = [shuffled(mm.gen_chunks(128, 96, 4), 70 + v) for v in range(3)]
    for first, step, count in ((5, 3, 200), (0, 1, 1), (767, 1, 1), (1, 2, 383)):
        q = copy_params(mm, p, group_first=first, group_step=step, group_count=count)
        frames, cnts, dbgs, _ = singles(mm, sc, noise, us, q, lists, debug=True)
        r = fresh(mm, sc, noise)
        outs = [np.empty((96, 128, 4), F) for _ in range(3)]
        _, cnt, dbg = r.render_views(us, q, lists, outs=outs, debug=True)
        for v, d in enumerate(split_debug(dbg, 3)):
            assert outs[v].tobytes() == frames[v].tobytes(), (first, step, count, v)
            for k in DBG_KEYS:
                assert d[k].tobytes() == dbgs[v][k].tobytes(), (first, step, count, v, k)
        assert cnt == summed(cnts)
        r.close()


@pytest.mark.gpu
def test_malformed_calls_are_errors(mm, noise, scenes):
    sc = scenes(10)
    r = fresh(mm, sc, noise)
    lib, ctx = mm.load_library(), r._ctx
    us = poses(mm, 2, 10, 32, 32, seed=2)
    p = mm.full_frame_params(us[0], spp=4, bounce_limit=4)
    ch = np.concatenate([mm.gen_chunks(32, 32, 4)] * 2)
    U = (mm.Uniform * 65)(*([us[0]] * 65))
    assert lib.mm_present_views(ctx, 0, None) == -1                                       # nothing rendered yet
    assert lib.mm_render_views(ctx, U, 0, C.byref(p), ch.ctypes.data, 0, None, None, None) == -1
    assert lib.mm_render_views(ctx, U, 65, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == -1
    assert lib.mm_render_views(ctx, None, 2, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == -1
    assert lib.mm_render_views(ctx, U, 2, None, ch.ctypes.data, len(ch), None, None, None) == -1
    assert lib.mm_render_views(ctx, U, 2, C.byref(p), None, len(ch), None, None, None) == -1
    assert lib.mm_render_views(ctx, U, 2, C.byref(p), ch.ctypes.data, len(ch) - 1, None, None, None) == -1
    other = (mm.Uniform * 2)(us[0], mm.default_uniform(10, 32, 36, 4))
    assert lib.mm_render_views(ctx, other, 2, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == -1
    other = (mm.Uniform * 2)(us[0], mm.default_uniform(10, 32, 32, 2))
    assert lib.mm_render_views(ctx, other, 2, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == -1
    ok = (mm.Uniform * 2)(*us)
    assert lib.mm_render_views(ctx, ok, 2, C.byref(p), ch.ctypes.data, len(ch), None, None, None) == 0
    assert lib.mm_present_views(ctx, 2, None) == -1
    unpinned = np.empty((32, 32, 4), F)
    outs = (C.c_void_p * 2)(unpinned.ctypes.data, None)
    assert lib.mm_present_views(ctx, 0, outs) == -1
    assert lib.mm_present_views(ctx, 0, None) == 0
    assert lib.mm_wait_present(ctx) == 0
    r.close()
