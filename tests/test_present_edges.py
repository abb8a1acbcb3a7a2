"""The kernels that deliver and present pixels after tracing, against their models at block, grid and frame edges.

- The present blur (blur_kernel / blur_views_kernel: 256 threads of two pixels, so one block covers 512 columns; rows on grid.y
  in steps of 65535) against np_oracle.present_blur, across block columns, at 1..100000 rows and on every class of float value.
- The tile scatters (scatter_kernel, scatter_all_kernel) against a numpy model, on synthetic tiles and chunk lists that cross
  the frame's right and bottom edges or lie wholly outside it.
- The render kernels' frame-edge guards (deliver_pixel, the pool kernel's delivery, the tail's deferred pixels, the views
  kernels) on the same chunk lists, against the oracle; tiles of off-frame pixels against the reduction of the oracle's paths.
- Presents at the view-size limits (4 x 65536, 65536 x 4) and at 1920 x 1080, and a synchronous RGBA8 present issued while an
  asynchronous one is still reading its texels back.
"""
import numpy as np
import pytest

F = np.float32
FLT_MAX = np.finfo(F).max


def f32(bits):
    return np.array(bits, dtype=np.uint32).view(F)


def ulps_around(v, k):
    """v and its k neighbours on each side, float32."""
    b = np.array([F(v)]).view(np.uint32)[0].astype(np.int64)
    return f32(b + np.arange(-k, k + 1)).tolist()


def tie_values():
    """Every float32 v in (0, 1) with RN(v * 255) == k + 0.5 exactly: the round-half-even cases of quant8."""
    out = []
    for k in range(255):
        c = f32(np.array([F((k + 0.5) / 255)]).view(np.uint32)[0].astype(np.int64) + np.arange(-4, 5))
        out += c[c * F(255.0) == F(k + 0.5)].tolist()
    return out


# Value classes of the blur's inputs.  The guard of div3 is |sum| >= 1e-30 after the adds: an isolated pixel's sum is its own
# value, and the sum beside an isolated 2e-30 is half of it, so planting these values puts sums on both sides of the guard.
CLASSES = {
    "zero": [0.0, -0.0],
    "negative": [-0.25, -1.0, -3.0e5, -1.0e30],
    "above_one": [1.0, 1.5, 255.0, 3.0e7, 1.0e30],
    "near_max": [float(FLT_MAX), float(np.nextafter(FLT_MAX, F(0))), float(FLT_MAX / F(2)), float(FLT_MAX * F(0.75)), -float(FLT_MAX)],
    "inf": [np.inf, -np.inf],
    "nan": [np.nan],
    "subnormal": [float(f32(1)), float(f32(0x007FFFFF)), -float(f32(1)), -float(f32(0x007FFFFF))],
    "guard": ulps_around(1e-30, 4) + ulps_around(2e-30, 4) + ulps_around(3e-30, 4) + [-v for v in ulps_around(1e-30, 4)],
    "tie": tie_values(),
}
SPECIAL_CLASSES = [k for k in CLASSES if k != "guard"]
SPECIALS = np.array([v for k in SPECIAL_CLASSES for v in CLASSES[k]], dtype=F)
GUARD = np.array(CLASSES["guard"], dtype=F)
G = F(1e-30)


def edge_columns(W):
    """Columns at the image's sides and on both sides of every 512-column block boundary."""
    cols = {0, 1, W - 2, W - 1}
    for b in range(512, W + 2, 512):
        cols |= {b - 2, b - 1, b, b + 1}
    return sorted(c for c in cols if 0 <= c < W)


def edge_rows(H):
    """Rows at the image's top and bottom and around 65535, where the blur's rows wrap onto the first block row again."""
    rows = {0, 1, H - 2, H - 1, 65533, 65534, 65535, 65536, 65537}
    return sorted(r for r in rows if 0 <= r < H)


def special_values(rng, n):
    """n values of SPECIALS, their classes in turn from a random start (every class once in any run of 8), uniform within one."""
    k = (int(rng.integers(len(SPECIAL_CLASSES))) + np.arange(n)) % len(SPECIAL_CLASSES)
    out = np.empty(n, F)
    for i, name in enumerate(SPECIAL_CLASSES):
        vals = np.array(CLASSES[name], F)
        out[k == i] = vals[rng.integers(0, len(vals), int((k == i).sum()))]
    return out


def edge_image(H, W, seed):
    """[H, W, 4] float32: uniform [0, 1) values, with every edge row and edge column a mix of SPECIALS (each colour channel
    special with probability 1/2 on rows, 3/4 on columns, so specials sit next to each other and next to plain values), and guard
    values planted as isolated pixels (their four neighbours zero) on the edge columns."""
    rng = np.random.default_rng(seed)
    img = rng.random((H, W, 4), dtype=F)
    for y in edge_rows(H):
        m = rng.random((W, 3)) < 0.5
        img[y, :, :3][m] = special_values(rng, int(m.sum()))
    for x in edge_columns(W):
        m = rng.random((H, 3)) < 0.75
        img[:, x, :3][m] = special_values(rng, int(m.sum()))
    for i, x in enumerate(edge_columns(W)):
        for j in range(2):
            y = (3 * i + 7 * j) % H
            v = GUARD[(2 * i + j) % len(GUARD)]
            for yy, xx in ((y - 1, x), (y + 1, x), (y, x - 1), (y, x + 1)):
                if 0 <= yy < H and 0 <= xx < W:
                    img[yy, xx, :3] = 0.0
            img[y, x, :3] = v
    return img


def blur_sums(img):
    """present_blur's value before the divide by 3: c + (r + l) / 2 + (d + u) / 2 (the input of div3)."""
    H, W = img.shape[:2]
    pad = np.zeros((H + 2, W + 2, 4), F)
    pad[1:-1, 1:-1] = img
    with np.errstate(all="ignore"):
        return (pad[1:-1, 1:-1] + (pad[1:-1, 2:] + pad[1:-1, :-2]) / F(2.0)) + (pad[2:, 1:-1] + pad[:-2, 1:-1]) / F(2.0)


def blur_model(img, rgba8=False, band=8192):
    """np_oracle.present_blur over row bands with a one-row halo (the same bits; keeps the temporaries of tall images small)."""
    from oracle import np_oracle

    H = img.shape[0]
    out = np.empty_like(img)
    with np.errstate(all="ignore"):
        for a in range(0, H, band):
            b = min(a + band, H)
            lo, hi = max(a - 1, 0), min(b + 1, H)
            out[a:b] = np_oracle.present_blur(img[lo:hi], rgba8=rgba8)[a - lo:a - lo + b - a]
    return out


def same_bits(a, b):
    """Bit for bit, except that any NaN matches any NaN."""
    a, b = np.asarray(a, F), np.asarray(b, F)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def texels(img):
    return np.rint(img * F(255.0)).astype(np.uint8)


# ---- chunk lists that cross the frame's edges ----------------------------------------------------------------------------------

CHUNK_WIDTHS = [1, 3, 4, 5, 64]


def frame_for(c):
    """A frame that is not a multiple of the chunk width and holds a few whole chunks of width c."""
    return (23, 17) if c == 1 else (7 * c + 5, 5 * c + 3)


def edge_chunks(W, H, c, seed, limit=None):
    """Non-overlapping chunks of width c in a W x H frame, shuffled, with their kinds: chunks crossing the right edge, the bottom
    edge and the corner (c > 1), chunks wholly outside the frame, chunks off the chunk grid (c > 1) and grid chunks.  limit caps
    the count; the edge and outside chunks are always kept."""
    from mirror_maze_b200.host import CHUNK_DTYPE

    rng = np.random.default_rng(seed)
    cross = (lambda n: n - c + int(rng.integers(1, c))) if c > 1 else None
    cand = [("outside", W, 0), ("outside", 0, H), ("outside", W + c, H + 2 * c), ("outside", W + 1000 * c, 5)]
    if c > 1:
        cand.append(("corner", cross(W), cross(H)))
        for _ in range(3):
            cand.append(("right", cross(W), c * int(rng.integers(0, H // c))))
            cand.append(("bottom", c * int(rng.integers(0, W // c)), cross(H)))
    grid = [(c * i, c * j) for i in range(W // c) for j in range(H // c)]
    rng.shuffle(grid)
    if c > 1:
        for x, y in grid[: max(2, len(grid) // 3)]:
            x2, y2 = x + int(rng.integers(1, c)), y + int(rng.integers(1, c))
            if x2 + c <= W and y2 + c <= H:
                cand.append(("off_grid", x2, y2))
    cand += [("grid", x, y) for x, y in grid]
    kept = []
    for kind, x, y in cand:
        if limit is not None and len(kept) >= limit and kind in ("off_grid", "grid"):
            continue
        if all(abs(x - x2) >= c or abs(y - y2) >= c for _, x2, y2 in kept):
            kept.append((kind, x, y))
    order = rng.permutation(len(kept))
    kept = [kept[i] for i in order]
    ch = np.zeros(len(kept), CHUNK_DTYPE)
    ch["x"] = [k[1] for k in kept]
    ch["y"] = [k[2] for k in kept]
    return ch, [k[0] for k in kept]


def chunk_pixels(ch, c):
    """(x, y) of pixel pn of every chunk: [n, c * c] each; pixel pn sits at (x + pn // c, y + pn % c)."""
    pn = np.arange(c * c)
    return ch["x"].astype(np.int64)[:, None] + pn // c, ch["y"].astype(np.int64)[:, None] + pn % c


def scatter_model(image, tiles, ch, c, first, step, count):
    """Tile k holds the chunk of group first + k * step; off-frame pixels are dropped."""
    H, W = image.shape[:2]
    out = image.copy()
    x, y = chunk_pixels(ch[first + step * np.arange(count)], c)
    ok = (x < W) & (y < H)
    out[y[ok], x[ok]] = np.asarray(tiles).reshape(-1, c * c, 4)[:count][ok]
    return out


def gathered_model(image, gathered, ch, c, world, max_count):
    """The all-gather layout: row r * max_count + k is rank r's tile k, group r + k * world; rows past the last group are padding."""
    n = len(ch)
    rows = np.arange(world * max_count)
    g = rows % max_count * world + rows // max_count
    keep = g < n
    H, W = image.shape[:2]
    out = image.copy()
    x, y = chunk_pixels(ch[g[keep]], c)
    ok = (x < W) & (y < H)
    out[y[ok], x[ok]] = np.asarray(gathered).reshape(-1, c * c, 4)[keep][ok]
    return out


# ---- without a GPU ----------------------------------------------------------------------------------------------------------------

def test_edge_image_reaches_every_class_at_block_edges():
    """At 17 x 1025 every value class sits on a column of each side of both block boundaries, specials sit next to specials, and
    the sums before the divide land on both sides of div3's guard; at 65537 rows the specials reach the rows around 65535."""
    img = edge_image(17, 1025, seed=1)
    bits = img.view(np.uint32)

    def has(cols, name):
        sub = img[:, cols, :3]
        vals = np.array(CLASSES[name], F)
        return bool(np.isnan(sub).any()) if name == "nan" else bool(np.isin(sub.view(np.uint32), vals.view(np.uint32)).any())

    for name in SPECIAL_CLASSES:
        for cols in ([0, 1], [510, 511], [512, 513], [1022, 1023], [1024]):
            assert has(cols, name), (name, cols)
    ties = np.array(CLASSES["tie"], F)
    assert len(ties) >= 255 and (ties * F(255.0) == np.floor(ties * F(255.0)) + F(0.5)).all()
    special = np.isin(bits[..., 0], SPECIALS.view(np.uint32)) | np.isnan(img[..., 0])
    assert (special[:, 511] & special[:, 512]).sum() >= 2 and (special[:, 1023] & special[:, 1024]).sum() >= 2
    assert (special[:, 511] & special[:, 510]).sum() >= 2 and (special[:, 512] & special[:, 513]).sum() >= 2
    sums = blur_sums(img)[..., :3]
    s = np.abs(sums)
    g = int(np.array([G]).view(np.uint32)[0])
    below = (s < G) & (s >= f32(g - 8))
    above = (s >= G) & (s <= f32(g + 8))
    assert below.sum() >= 3 and above.sum() >= 3                                        # both sides of div3's guard
    assert (np.isinf(sums) & np.isfinite(img[..., :3])).sum() >= 3                       # finite values whose adds overflow
    assert (np.isnan(sums) & ~np.isnan(img[..., :3])).sum() >= 1                          # inf - inf
    tall = edge_image(65537, 2, seed=2)
    for y in (65534, 65535, 65536):
        assert (np.isin(tall[y].view(np.uint32), SPECIALS.view(np.uint32)) | np.isnan(tall[y])).any(), y


def test_banded_blur_model_equals_the_whole_image_model():
    from oracle import np_oracle

    img = edge_image(37, 9, seed=3)
    with np.errstate(all="ignore"):
        for rgba8 in (False, True):
            assert same_bits(blur_model(img, rgba8, band=5), np_oracle.present_blur(img, rgba8))


@pytest.mark.parametrize("c", CHUNK_WIDTHS)
def test_chunk_lists_reach_their_edges(mm, c):
    """Every kind the generator claims, counted; no two chunks overlap; the order is not the grid's."""
    W, H = frame_for(c)
    for seed in range(3):
        ch, kinds = edge_chunks(W, H, c, seed)
        x0, y0 = ch["x"].astype(np.int64), ch["y"].astype(np.int64)
        apart = (np.abs(x0[:, None] - x0[None]) >= c) | (np.abs(y0[:, None] - y0[None]) >= c)
        assert (apart | np.eye(len(ch), dtype=bool)).all()                            # no two chunks overlap
        inside = (x0 + c <= W) & (y0 + c <= H)
        right, bottom = (x0 < W) & (x0 + c > W), (y0 < H) & (y0 + c > H)
        outside = (x0 >= W) | (y0 >= H)
        counts = {k: kinds.count(k) for k in set(kinds)}
        assert counts["outside"] == outside.sum() == 4
        assert counts["grid"] >= 2 and (x0[inside] % c == 0).sum() >= 2
        if c > 1:
            assert counts["right"] >= 1 and (right & ~bottom).sum() == counts["right"]
            assert counts["bottom"] >= 1 and (bottom & ~right).sum() == counts["bottom"]
            assert counts["corner"] == (right & bottom).sum() == 1
            assert counts["off_grid"] >= 1 and (((x0 % c) != 0) & ((y0 % c) != 0) & inside).sum() == counts["off_grid"]
        order = [k for k in kinds if k == "grid"]
        assert len(order) < 2 or list(np.argsort(x0 * 100000 + y0)) != list(range(len(ch)))   # shuffled
    ch, kinds = edge_chunks(W, H, c, 0, limit=5)
    assert set(kinds) - {"grid", "off_grid"} == set(edge_chunks(W, H, c, 0)[1]) - {"grid", "off_grid"}


def test_scatter_models_place_tiles_as_the_host_scatter_does(mm):
    """The numpy models against the product's host twin (scatter_tiles_host) and the padding rule of the all-gather layout."""
    from mirror_maze_b200.renderer import scatter_tiles_host, tile_partition

    c = 3
    W, H = frame_for(c)
    ch, _ = edge_chunks(W, H, c, 4)
    n = len(ch)
    rng = np.random.default_rng(0)
    tiles = rng.random((n, c * c, 4), dtype=F)
    base = np.full((H, W, 4), -7.0, F)
    for first, step, count in ((0, 1, n), (1, 3, (n - 1 + 2) // 3), (2, 2, 3)):
        want = scatter_tiles_host(tiles[:count], ch, first, step, count, c, base.copy())
        assert scatter_model(base, tiles, ch, c, first, step, count).tobytes() == want.tobytes()
    world = 8
    max_count = max(tile_partition(n, r, world)[2] for r in range(world))
    assert n % world != 0
    gathered = rng.random((world * max_count, c * c, 4), dtype=F)
    want = base.copy()
    for r in range(world):
        first, step, count = tile_partition(n, r, world)
        want = scatter_model(want, gathered[r * max_count:(r + 1) * max_count], ch, c, first, step, count)
    assert gathered_model(base, gathered, ch, c, world, max_count).tobytes() == want.tobytes()


# ---- the blur on the GPU ----------------------------------------------------------------------------------------------------------

BLUR_SHAPES = [(h, w) for w in (1, 2, 3, 511, 512, 513, 514, 1023, 1024, 1025, 1536, 1537, 1920) for h in (1, 2, 3, 17)]
TALL_SHAPES = [(h, w) for w in (1, 2, 513) for h in (65535, 65536, 65537, 100000)]


def blur_on_gpu(renderer, img):
    import torch

    src = torch.from_numpy(img).cuda()
    dst = torch.full_like(src, float("nan"))
    torch.cuda.synchronize()
    renderer.present_blur_device(src.data_ptr(), dst.data_ptr(), img.shape[1], img.shape[0])
    renderer.sync()
    return dst.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", BLUR_SHAPES, ids=[f"{h}x{w}" for h, w in BLUR_SHAPES])
def test_blur_across_block_columns_matches_model(renderer, shape):
    H, W = shape
    img = edge_image(H, W, seed=H * 7919 + W)
    assert same_bits(blur_on_gpu(renderer, img), blur_model(img))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", TALL_SHAPES, ids=[f"{h}x{w}" for h, w in TALL_SHAPES])
def test_blur_of_tall_images_matches_model(renderer, shape):
    """Heights at and past grid.y's 65535: rows 65535 and beyond are blurred by the first block rows' second pass."""
    H, W = shape
    img = edge_image(H, W, seed=H + W)
    assert same_bits(blur_on_gpu(renderer, img), blur_model(img))


# ---- presents at the view-size limits and across block columns ---------------------------------------------------------------------

def check_presents(mm, r, H, W, screen, what):
    """mm_present, mm_present_rgba8, mm_present_async and mm_present_async_rgba8 in turn on r's screen, each against the next step
    of the blur model; returns the model screen."""
    out = np.empty((H, W, 4), F)
    r.present(out)
    screen = blur_model(screen)
    assert out.tobytes() == screen.tobytes(), f"{what}: present"
    out8 = np.empty((H, W, 4), np.uint8)
    r.present_rgba8(out, out8)
    screen = blur_model(screen, rgba8=True)
    assert out.tobytes() == screen.tobytes() and out8.tobytes() == texels(screen).tobytes(), f"{what}: present_rgba8"
    hf = mm.HostFrame(H, W)
    r.present_async(hf.ptr)
    r.wait_present()
    screen = blur_model(screen)
    assert hf.array.tobytes() == screen.tobytes(), f"{what}: present_async"
    r.present_async_rgba8(hf.ptr)
    r.wait_present()
    screen = blur_model(screen, rgba8=True)
    assert hf.array.reshape(-1).view(np.uint8)[: H * W * 4].tobytes() == texels(screen).tobytes(), f"{what}: present_async_rgba8"
    hf.close()
    return screen


def check_present_views(r, hfs, models, rgba8, what):
    H, W = models[0].shape[:2]
    r.present_views(hfs, rgba8=rgba8)
    r.wait_present()
    for v, hf in enumerate(hfs):
        models[v] = blur_model(models[v], rgba8=rgba8)
        want = texels(models[v]).tobytes() if rgba8 else models[v].tobytes()
        assert hf.array.reshape(-1).view(np.uint8)[: len(want)].tobytes() == want, f"{what}: present_views rgba8 {rgba8} view {v}"


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(4, 65536), (65536, 4)], ids=["4x65536", "65536x4"])
def test_views_at_the_size_limits_render_and_present(mm, oracle, noise, scenes, size):
    """A 4 x 65536 and a 65536 x 4 view (W x H), chunk 4, spp 1, 2 bounces: the render equals the oracle, and every present of
    the screen, and of two views of the same size, equals the blur model."""
    W, H = size
    sc = scenes(16)
    u = mm.default_uniform(16, W, H, 4, 5)
    ch = mm.gen_chunks(W, H, 4)
    p = mm.full_frame_params(u, spp=1, bounce_limit=2)
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    img = r.render(u, p, ch)[0]
    ref = oracle.render(sc, noise, u, p, ch)[0]
    assert img.tobytes() == ref.tobytes()
    check_presents(mm, r, H, W, ref, f"{W}x{H}")
    us = [mm.default_uniform(16, W, H, 4, t) for t in (5, 6)]
    r.render_views(us, p, [ch, ch])
    models = [oracle.render(sc, noise, v, p, ch)[0] for v in us]
    hfs = [mm.HostFrame(H, W) for _ in us]
    check_present_views(r, hfs, models, False, f"{W}x{H}")
    check_present_views(r, hfs, models, True, f"{W}x{H}")
    for hf in hfs:
        hf.close()
    r.close()


HD = dict(W=1920, H=1080, maze=16, center=(0.0, 0.0, -45.0), half_theta=0.0, spp=1, bounce=4)


@pytest.mark.gpu
def test_progressive_refresh_at_1080p(mm, oracle, noise, scenes):
    """1920 x 1080, three and a half block columns: frames of 1/64 of the chunks each, presented with present, present_async,
    and present_rgba8 (whose clamp the frame's values above 1 reach), then two views through present_views; every present
    against the oracle's chunks composed with the blur model."""
    W, H = HD["W"], HD["H"]
    sc = scenes(HD["maze"])
    u = mm.default_uniform(HD["maze"], W, H, 4, 0, camera_center=HD["center"], half_theta=HD["half_theta"])
    n = (W // 4) * (H // 4) // 64
    p = mm.Params(spp=HD["spp"], bounce_limit=HD["bounce"], mirror_limit=15, grid_x=n, grid_y=1)
    bag = mm.ChunkBag(W, H, 4, seed=3)
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    screen = np.zeros((H, W, 4), F)
    hf = mm.HostFrame(H, W)
    above_one = 0
    for frame, how in enumerate(("present", "present_async", "present_rgba8", "present_rgba8")):
        u.time = frame
        ch = bag.next(n)
        r.render(u, p, ch)
        oracle.render(sc, noise, u, p, ch, out=screen)
        if how == "present":
            out = np.empty((H, W, 4), F)
            r.present(out)
            screen = blur_model(screen)
            assert out.tobytes() == screen.tobytes(), frame
        elif how == "present_async":
            r.present_async(hf.ptr)
            r.wait_present()
            screen = blur_model(screen)
            assert hf.array.tobytes() == screen.tobytes(), frame
        else:
            out, out8 = np.empty((H, W, 4), F), np.empty((H, W, 4), np.uint8)
            r.present_rgba8(out, out8)
            above_one += int((blur_model(screen)[..., :3] > 1).sum())
            screen = blur_model(screen, rgba8=True)
            assert out.tobytes() == screen.tobytes() and out8.tobytes() == texels(screen).tobytes(), frame
    assert above_one > 0
    hf.close()
    us = [mm.default_uniform(HD["maze"], W, H, 4, t, camera_center=HD["center"], half_theta=h) for t, h in ((1, 0.0), (2, 0.4))]
    bags = [mm.ChunkBag(W, H, 4, seed=10 + v) for v in range(2)]
    models = [np.zeros((H, W, 4), F) for _ in us]
    hfs = [mm.HostFrame(H, W) for _ in us]
    for rgba8 in (False, True):
        lists = [b.next(n) for b in bags]
        r.render_views(us, p, lists)
        for v in range(2):
            oracle.render(sc, noise, us[v], p, lists[v], out=models[v])
        check_present_views(r, hfs, models, rgba8, "1080p")
    for h in hfs:
        h.close()
    r.close()


# ---- the scatter kernels on synthetic tiles --------------------------------------------------------------------------------------

SENTINEL = -7.0


@pytest.mark.gpu
@pytest.mark.parametrize("c", CHUNK_WIDTHS)
def test_scatter_kernels_match_model(mm, renderer, c):
    """mm_scatter_tiles_device for every rank's interleaved share (worlds 1, 3, 8; group counts not a multiple of the world) and
    the whole range; mm_scatter_gathered_device for the all-gather layout with its padding rows.  Unwritten pixels keep the
    sentinel."""
    import torch

    from mirror_maze_b200.renderer import tile_partition

    W, H = frame_for(c)
    torch.manual_seed(c)
    for seed in range(2):
        ch, kinds = edge_chunks(W, H, c, seed)
        while len(ch) % 3 == 0 or len(ch) % 8 == 0:                  # a group count that worlds 3 and 8 do not divide
            drop = kinds.index("grid")
            ch, kinds = np.delete(ch, drop), kinds[:drop] + kinds[drop + 1:]
        n = len(ch)
        u = mm.default_uniform(16, W, H, c)
        renderer.set_chunks(ch)
        base = np.full((H, W, 4), SENTINEL, F)
        for world in (1, 3, 8):
            assert world == 1 or n % world != 0
            parts = [tile_partition(n, r, world) for r in range(world)]
            max_count = max(pt[2] for pt in parts)
            gathered = torch.rand((world * max_count, c * c, 4), device="cuda")
            host = gathered.cpu().numpy()
            for r, (first, step, count) in enumerate(parts):
                p = mm.Params(spp=1, bounce_limit=1, mirror_limit=15, grid_x=n, grid_y=1, group_first=first, group_step=step,
                              group_count=count)
                image = torch.full((H, W, 4), SENTINEL, device="cuda")
                tiles = gathered[r * max_count:]
                renderer.scatter_tiles_device(u, p, tiles.data_ptr(), image.data_ptr())
                renderer.sync()
                want = scatter_model(base, host[r * max_count:], ch, c, first, step, count)
                assert image.cpu().numpy().tobytes() == want.tobytes(), (seed, world, r)
            p = mm.Params(spp=1, bounce_limit=1, mirror_limit=15, grid_x=n, grid_y=1)
            image = torch.full((H, W, 4), SENTINEL, device="cuda")
            renderer.scatter_gathered_device(u, p, world, max_count, gathered.data_ptr(), image.data_ptr())
            renderer.sync()
            assert image.cpu().numpy().tobytes() == gathered_model(base, host, ch, c, world, max_count).tobytes(), (seed, world)
        tiles = torch.rand((n, c * c, 4), device="cuda")
        image = torch.full((H, W, 4), SENTINEL, device="cuda")
        renderer.scatter_tiles_device(u, mm.Params(spp=1, bounce_limit=1, mirror_limit=15, grid_x=n, grid_y=1), tiles.data_ptr(),
                                      image.data_ptr())
        renderer.sync()
        assert image.cpu().numpy().tobytes() == scatter_model(base, tiles.cpu().numpy(), ch, c, 0, 1, n).tobytes(), seed


# ---- the render kernels on edge-crossing chunk lists -----------------------------------------------------------------------------

def edge_spp(c):
    """8 samples, or 32 where c * c * 8 is neither at most 32 nor a multiple of 32 (the launch's virtual-threadgroup rule)."""
    return 8 if c * c * 8 <= 32 or c * c * 8 % 32 == 0 else 32


def path_tiles(u, p, radiance):
    """Every tile pixel from the oracle's per-path radiance, in or out of the frame: the reference's per-pixel reduction
    (shaders.metal:344-366) as tests/test_high_spp.py's restated_image restates it: tone-map, pairwise sums at strides 1, 2, 4
    within each group of 8, the octets summed serially, divided by spp."""
    c, s = int(u.chunk_width), int(p.spp)
    v = np.sqrt(np.fmax(np.asarray(radiance, F).reshape(-1, c * c, s, 3), F(0.0)))
    for stride in (1, 2, 4):
        v[:, :, ::2 * stride] = v[:, :, ::2 * stride] + v[:, :, stride::2 * stride]
    acc = v[:, :, 0].copy()
    for o in range(8, s, 8):
        acc = acc + v[:, :, o]
    out = np.ones(v.shape[:2] + (4,), F)
    out[..., :3] = acc / F(s)
    return out


def edge_case(mm, c, time=77):
    W, H = frame_for(c)
    u = mm.default_uniform(16, W, H, c, time, camera_center=(25.0, 0.0, -15.0), half_theta=1.1)
    spp = edge_spp(c)
    ch, _ = edge_chunks(W, H, c, seed=c, limit=max(12, 300_000 // (c * c * spp)))
    p = mm.Params(spp=spp, bounce_limit=3, mirror_limit=15, grid_x=len(ch), grid_y=1)
    return u, p, ch


KERNEL_PATHS = {
    "default": (0, {}),
    "no_y_table": ("FLAG_NO_Y_TABLE", {}),
    "no_tail": ("FLAG_NO_TAIL", {}),
    "tail_k32_cap64": (0, {"MM_TAIL_K": "32", "MM_TAIL_CAP": "64"}),
    "pool": ("FLAG_POOL_KERNEL", {}),
    "regroup": ("FLAG_REGROUP", {}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("c", CHUNK_WIDTHS)
def test_render_kernels_on_edge_crossing_chunks(mm, oracle, noise, scenes, renderer, monkeypatch, c):
    """Each kernel path on a chunk list with chunks across the right and bottom edges, in the corner and wholly outside: the image
    (sentinel-filled, so pixels outside every chunk are checked too) equals the oracle's bit for bit; in-frame tile pixels equal
    the image and off-frame ones the reduction of the oracle's paths.  render_views on the same list equals the oracle per view."""
    import torch

    sc = scenes(16)
    u, p, ch = edge_case(mm, c)
    W, H = int(u.view_width), int(u.view_height)
    n = len(ch)
    ref_img, _, dbg = oracle.render(sc, noise, u, p, ch, debug=True, out=np.full((H, W, 4), SENTINEL, F))
    ref_tiles = path_tiles(u, p, dbg["radiance"])
    x, y = chunk_pixels(ch, c)
    inside = (x < W) & (y < H)
    assert inside.any() and not inside.all()
    assert same_bits(ref_tiles[inside], ref_img[y[inside], x[inside]])   # the restated reduction is the oracle's pixel
    renderer.upload_scene(sc, noise)
    renderer.set_chunks(ch)
    deferred = 0
    for name, (flag, env) in KERNEL_PATHS.items():
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        q = mm.Params.from_buffer_copy(bytes(p))
        q.flags = getattr(mm, flag) if flag else 0
        image = torch.full((H, W, 4), SENTINEL, device="cuda")
        tiles = torch.full((n, c * c, 4), SENTINEL, device="cuda")
        renderer.render_device(u, q, image_ptr=image.data_ptr(), tiles_ptr=tiles.data_ptr())
        renderer.sync()
        if env:
            deferred += renderer.last_tail()[1]
        for k in env:
            monkeypatch.delenv(k)
        got, gt = image.cpu().numpy(), tiles.cpu().numpy()
        assert got.tobytes() == ref_img.tobytes(), name
        assert gt[inside].tobytes() == got[y[inside], x[inside]].tobytes(), name
        assert gt[~inside].tobytes() == ref_tiles[~inside].tobytes(), name
    assert deferred > 0
    us = [u, mm.default_uniform(16, W, H, c, 78, camera_center=(25.0, 0.0, -15.0), half_theta=1.1)]
    outs, _, _ = renderer.render_views(us, p, [ch, ch], outs=[np.empty((H, W, 4), F) for _ in us])
    for v in range(2):
        want = oracle.render(sc, noise, us[v], p, ch)[0]
        assert outs[v].tobytes() == want.tobytes(), f"view {v}"


# ---- a synchronous RGBA8 present while an asynchronous one reads back ----------------------------------------------------------

@pytest.mark.gpu
def test_present_rgba8_waits_for_the_texels_of_present_async_rgba8(mm, noise, scenes):
    """An 8K screen: present_async_rgba8 queues the read-back of the texel buffer, and present_rgba8, called at once, blurs into
    the same buffer; it must wait for the read-back.  The pinned texels are the first step of the model, present_rgba8's
    outputs the second."""
    W, H = 7680, 4320
    sc = scenes(16)
    u = mm.default_uniform(16, W, H, 4, 3)
    p = mm.full_frame_params(u, spp=1, bounce_limit=1)
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    screen = r.render(u, p, mm.gen_chunks(W, H, 4))[0]
    hf = mm.HostFrame(H, W)
    out, out8 = np.empty((H, W, 4), F), np.empty((H, W, 4), np.uint8)
    r.present_async_rgba8(hf.ptr)
    r.present_rgba8(out, out8)
    r.wait_present()
    first = blur_model(screen, rgba8=True)
    second = blur_model(first, rgba8=True)
    got = hf.array.reshape(-1).view(np.uint8)[: H * W * 4]
    assert (texels(first) != texels(second)).any()
    assert got.tobytes() == texels(first).tobytes()
    assert out.tobytes() == second.tobytes() and out8.tobytes() == texels(second).tobytes()
    hf.close()
    r.close()
