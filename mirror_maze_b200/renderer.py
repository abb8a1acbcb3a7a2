"""Dispatch side of the drop-in: what the reference's frame loop does at src/main.rs:778-784 and 867-894
(rewrite the chunk list, set the uniform, dispatch compute_shader, read the screen), through the C-ABI.

Renderer          one context = one GPU = one stream (the reference has one device and one queue, main.rs:616-623).
tile_partition    the multi-GPU split: interleaved groups of the virtual grid; seeds depend on the group index,
                  not on the rank, so the union of all ranks' tiles is bit-identical to a one-GPU frame.
TiledFrameRenderer  one process per GPU: render own tiles -> all-gather over NCCL (NVLink) -> scatter into the frame.

No CPU fallback: constructing a Renderer without the built library or without a B200 raises MMError.
"""
import ctypes as C

import numpy as np

from . import abi
from .abi import Counters, Debug, MMError, Params, SceneInfo
from .host import CHUNK_DTYPE, NODE_DTYPE, PLANE_DTYPE


def tile_partition(n_groups, rank, world):
    """(group_first, group_step, group_count) of `rank`: groups rank, rank+world, ... (load-balanced stripes)."""
    if not (0 <= rank < world):
        raise ValueError("rank outside world")
    count = (n_groups - rank + world - 1) // world if n_groups > rank else 0
    return rank, world, count


def scatter_tiles_host(tiles, chunks, first, step, count, chunk_width, image):
    """Host twin of mm_scatter_tiles_device for callers that keep gathered tiles on the host:
    tile k -> chunk of group first + k*step; pixel pn of a tile sits at (x + pn // chunk, y + pn % chunk)
    (reference src/shaders.metal:272-275)."""
    ppc = chunk_width * chunk_width
    t = np.asarray(tiles, dtype=np.float32).reshape(-1, ppc, 4)
    H, W = image.shape[:2]
    pn = np.arange(ppc)
    dx, dy = pn // chunk_width, pn % chunk_width
    for k in range(count):
        ch = chunks[first + k * step]
        x, y = int(ch["x"]) + dx, int(ch["y"]) + dy
        ok = (x < W) & (y < H)
        image[y[ok], x[ok]] = t[k][ok]
    return image


class HostFrame:
    """A frame buffer in mapped pinned host memory (mm_host_alloc): mm_render / mm_multi_render write into it zero-copy.
    `array` is the [H, W, 4] float32 view; keep the HostFrame alive while the array is in use."""

    def __init__(self, height, width):
        self._lib = abi.load_library()
        self._ptr = C.c_void_p()
        self.nbytes = int(height) * int(width) * 16
        rc = self._lib.mm_host_alloc(self.nbytes, C.byref(self._ptr))
        if rc != 0:
            raise MMError(rc, "mm_host_alloc")
        buf = (C.c_float * (self.nbytes // 4)).from_address(self._ptr.value)
        self.array = np.ctypeslib.as_array(buf).reshape(int(height), int(width), 4)
        self.array[...] = 0.0

    @property
    def ptr(self):
        return self._ptr.value

    def close(self):
        if getattr(self, "_ptr", None) and self._ptr.value:
            self.array = None
            self._lib.mm_host_free(self._ptr)
            self._ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Renderer:
    def __init__(self, device=0):
        self._lib = abi.load_library()
        self._ctx = C.c_void_p()
        rc = self._lib.mm_create(device, C.byref(self._ctx))
        if rc != 0:
            raise MMError(rc, (self._lib.mm_last_error(None) or b"").decode())
        self.device = device
        self._chunks = None

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.mm_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise MMError(rc, (self._lib.mm_last_error(self._ctx) or b"").decode())

    # -- scene -------------------------------------------------------------------------------------------------
    def upload_scene(self, scene, noise):
        """make_buf x6 + noise texture (src/main.rs:667-695, 723-730)."""
        planes = np.ascontiguousarray(scene.planes, dtype=PLANE_DTYPE)
        nodes = np.ascontiguousarray(scene.nodes, dtype=NODE_DTYPE)
        indices = np.ascontiguousarray(scene.indices, dtype=np.uint32)
        materials = np.ascontiguousarray(scene.materials, dtype=np.uint8)
        emissions = np.ascontiguousarray(scene.emissions, dtype=np.float32)
        noise = np.ascontiguousarray(noise, dtype=np.uint8)
        nh, nw = noise.shape[:2]
        self._ck(self._lib.mm_upload_scene(self._ctx, planes.ctypes.data, len(planes), nodes.ctypes.data, len(nodes),
                                           indices.ctypes.data, materials.ctypes.data, emissions.ctypes.data,
                                           noise.ctypes.data, nw, nh))

    def scene_info(self):
        info = SceneInfo()
        self._ck(self._lib.mm_get_scene_info(self._ctx, C.byref(info)))
        return info.as_dict()

    # -- host-buffer render (the reference-facing call) -------------------------------------------------------------
    def render(self, uniform, params, chunks, out=None, debug=False):
        """One dispatch with HOST buffers in and out.  Returns (image[H,W,4] float32, counters dict, debug dict|None)."""
        chunks = np.ascontiguousarray(chunks, dtype=CHUNK_DTYPE)
        H, W = int(uniform.view_height), int(uniform.view_width)
        if out is None:
            out = np.empty((H, W, 4), dtype=np.float32)
        assert out.dtype == np.float32 and out.size == H * W * 4 and out.flags["C_CONTIGUOUS"]
        cnt = Counters()
        dbg_struct, dbg = None, None
        if debug:
            n_groups = params.group_count or params.grid_x * params.grid_y
            n_paths = n_groups * uniform.chunk_width ** 2 * params.spp
            dbg = {"first_hit": np.empty(n_paths, np.uint32), "segments": np.empty(n_paths, np.uint32),
                   "mirror_hits": np.empty(n_paths, np.uint32), "radiance": np.empty((n_paths, 3), np.float32)}
            dbg_struct = Debug(dbg["first_hit"].ctypes.data_as(C.POINTER(C.c_uint32)),
                               dbg["segments"].ctypes.data_as(C.POINTER(C.c_uint32)),
                               dbg["mirror_hits"].ctypes.data_as(C.POINTER(C.c_uint32)),
                               dbg["radiance"].ctypes.data_as(C.POINTER(C.c_float)))
        self._ck(self._lib.mm_render(self._ctx, C.byref(uniform), C.byref(params), chunks.ctypes.data, len(chunks),
                                     out.ctypes.data, C.byref(cnt), C.byref(dbg_struct) if dbg_struct else None))
        return out, cnt.as_dict(), dbg

    def render_into(self, uniform, params, chunks_ptr, n_chunks, out_ptr):
        """mm_render on raw host pointers; returns counters dict.  chunks_ptr None keeps the device chunk list."""
        cnt = Counters()
        self._ck(self._lib.mm_render(self._ctx, C.byref(uniform), C.byref(params), chunks_ptr, n_chunks, out_ptr,
                                     C.byref(cnt), None))
        return cnt.as_dict()

    def render_async(self, uniform, params, chunks_ptr, n_chunks, out_ptr):
        """mm_render_async: returns once the frame is enqueued (the reference commits without waiting, main.rs:894)."""
        self._ck(self._lib.mm_render_async(self._ctx, C.byref(uniform), C.byref(params), chunks_ptr, n_chunks, out_ptr, None))

    def wait(self):
        """mm_wait: the frame of the last render_async is in the caller's buffer; returns its counters."""
        cnt = Counters()
        self._ck(self._lib.mm_wait(self._ctx, C.byref(cnt)))
        return cnt.as_dict()

    def render_multicast_device(self, uniform, params, mc_ptr):
        """mm_render_multicast_device: every finished pixel is one multimem.st to an NVSwitch multicast address."""
        self._ck(self._lib.mm_render_multicast_device(self._ctx, C.byref(uniform), C.byref(params), mc_ptr))

    # -- device-resident path ------------------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self._lib.mm_set_stream(self._ctx, cuda_stream_ptr))

    def set_chunks(self, chunks):
        chunks = np.ascontiguousarray(chunks, dtype=CHUNK_DTYPE)
        self._chunks = chunks          # keep alive until the async copy has run
        self._ck(self._lib.mm_set_chunks(self._ctx, chunks.ctypes.data, len(chunks)))

    def render_device(self, uniform, params, image_ptr=None, tiles_ptr=None):
        self._ck(self._lib.mm_render_device(self._ctx, C.byref(uniform), C.byref(params), image_ptr, tiles_ptr))

    def render_peers_device(self, uniform, params, frame_ptrs):
        """mm_render_peers_device: render this rank's groups and store every pixel into each frame (peer / multicast)."""
        arr = (C.c_void_p * len(frame_ptrs))(*[int(p) for p in frame_ptrs])
        self._ck(self._lib.mm_render_peers_device(self._ctx, C.byref(uniform), C.byref(params), arr, len(frame_ptrs)))

    def scatter_tiles_device(self, uniform, params, tiles_ptr, image_ptr):
        self._ck(self._lib.mm_scatter_tiles_device(self._ctx, C.byref(uniform), C.byref(params), tiles_ptr, image_ptr))

    def scatter_gathered_device(self, uniform, params, world, max_count, gathered_ptr, image_ptr):
        self._ck(self._lib.mm_scatter_gathered_device(self._ctx, C.byref(uniform), C.byref(params), world, max_count, gathered_ptr, image_ptr))

    def sync(self):
        self._ck(self._lib.mm_sync(self._ctx))

    def last_counters(self):
        cnt = Counters()
        self._ck(self._lib.mm_last_counters(self._ctx, C.byref(cnt)))
        return cnt.as_dict()

    def present(self, out=None, copy=True):
        """The present pass' 5-tap blur over the persistent screen (src/shaders.metal:214-225, src/main.rs:888-892);
        returns the blurred screen as a host array when copy is true."""
        if copy and out is None:
            raise ValueError("pass the host array that receives the frame")
        self._ck(self._lib.mm_present(self._ctx, out.ctypes.data if copy else None))
        return out

    def present_async(self, out_ptr):
        """mm_present_async: blur + read-back into pinned host memory on a second stream; returns at once."""
        self._ck(self._lib.mm_present_async(self._ctx, out_ptr))

    def present_async_rgba8(self, out_ptr):
        """mm_present_async_rgba8: the quantising blur; the texels (4 bytes per pixel) are read back on a second stream."""
        self._ck(self._lib.mm_present_async_rgba8(self._ctx, out_ptr))

    def wait_present(self):
        self._ck(self._lib.mm_wait_present(self._ctx))

    def present_rgba8(self, out=None, out_bytes=None):
        """mm_present_rgba8: the present blur on an RGBA8Unorm screen; fills the float frame (values k/255) and / or the
        uint8 [H, W, 4] texel array."""
        self._ck(self._lib.mm_present_rgba8(self._ctx, None if out is None else out.ctypes.data,
                                            None if out_bytes is None else out_bytes.ctypes.data))
        return out, out_bytes

    def present_blur_device(self, src_ptr, dst_ptr, width, height):
        self._ck(self._lib.mm_present_blur_device(self._ctx, src_ptr, dst_ptr, width, height))

    def microbench(self, kind, table_bytes=0):
        """kind 0: GB/s of the traversal's per-visit fetch pattern from a table of table_bytes; kind 1: T FP32 FMA lane-instr/s."""
        out = C.c_double()
        self._ck(self._lib.mm_microbench(self._ctx, kind, table_bytes, C.byref(out)))
        return float(out.value)

    def selftest_quotient(self, n_pairs, seed=1):
        """Mismatches between the shared-reciprocal slab quotient and __fdiv_rn over n_pairs samples (must be 0)."""
        bad = C.c_uint64()
        self._ck(self._lib.mm_selftest_quotient(self._ctx, n_pairs, seed, C.byref(bad)))
        return int(bad.value)

    def selftest_div3(self):
        """Mismatches between the blur's exact x / 3 sequence and __fdiv_rn(x, 3) over all 2^32 floats (must be 0)."""
        bad = C.c_uint64()
        self._ck(self._lib.mm_selftest_div3(self._ctx, C.byref(bad)))
        return int(bad.value)

    def trace_rays(self, rays, slots=None, flags=0):
        """mm_trace_rays: one traversal per ray of the uploaded scene, 32 rays to a warp in the order given.  rays [n, 8] float32
        (ori.xyz, dir.xyz, t, alive), slots [n] starting leaf-order slots or None.  Returns a dict of numpy arrays: t, index
        (plane index of the hit), inner, leaf, rect, max_stack, lit and form (the traversal the ray's warp ran, bits
        1 mixed literal, 2 reciprocal-multiply, 4 axis-aligned rects, 8 y-table)."""
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
        n = len(rays)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.uint32)
        t, index, tally = np.empty(n, np.float32), np.empty(n, np.uint32), np.empty((n, 6), np.uint32)
        self._ck(self._lib.mm_trace_rays(self._ctx, flags, rays.ctypes.data, None if sl is None else sl.ctypes.data, n,
                                         t.ctypes.data, index.ctypes.data, tally.ctypes.data))
        out = {"t": t, "index": index}
        for i, k in enumerate(("inner", "leaf", "rect", "max_stack", "lit", "form")):
            out[k] = tally[:, i]
        return out

    def last_ms(self):
        ms = C.c_float()
        self._ck(self._lib.mm_last_ms(self._ctx, C.byref(ms)))
        return float(ms.value)

    def last_tail(self):
        """mm_last_tail: (paths queued for the straggler kernel, pixels deferred to it) in the most recent render."""
        q, px = C.c_uint64(), C.c_uint64()
        self._ck(self._lib.mm_last_tail(self._ctx, C.byref(q), C.byref(px)))
        return int(q.value), int(px.value)


class MultiRenderer:
    """mm_multi: one process, several GPUs behind the C-ABI (no torch involved): scene replicated, the frame's groups
    interleaved over the devices, pixels exchanged by the render kernel's peer stores ("peer"), an NCCL all-gather of
    tiles ("nccl") or assembled only in the caller's pinned host frame ("none")."""

    EXCHANGE = {"peer": abi.EXCHANGE_PEER, "nccl": abi.EXCHANGE_NCCL, "none": abi.EXCHANGE_NONE}

    def __init__(self, devices, exchange="peer"):
        self._lib = abi.load_library()
        self._m = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        rc = self._lib.mm_multi_create(devs, len(devices), self.EXCHANGE[exchange], C.byref(self._m))
        if rc != 0:
            raise MMError(rc, (self._lib.mm_multi_last_error(None) or b"").decode())
        self.devices, self.exchange = list(devices), exchange

    def close(self):
        if getattr(self, "_m", None):
            self._lib.mm_multi_destroy(self._m)
            self._m = None

    def __del__(self):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise MMError(rc, (self._lib.mm_multi_last_error(self._m) or b"").decode())

    def upload_scene(self, scene, noise):
        planes = np.ascontiguousarray(scene.planes, dtype=PLANE_DTYPE)
        nodes = np.ascontiguousarray(scene.nodes, dtype=NODE_DTYPE)
        indices = np.ascontiguousarray(scene.indices, dtype=np.uint32)
        materials = np.ascontiguousarray(scene.materials, dtype=np.uint8)
        emissions = np.ascontiguousarray(scene.emissions, dtype=np.float32)
        noise = np.ascontiguousarray(noise, dtype=np.uint8)
        nh, nw = noise.shape[:2]
        self._ck(self._lib.mm_multi_upload_scene(self._m, planes.ctypes.data, len(planes), nodes.ctypes.data, len(nodes),
                                                 indices.ctypes.data, materials.ctypes.data, emissions.ctypes.data,
                                                 noise.ctypes.data, nw, nh))

    def render(self, uniform, params, chunks, out):
        """One frame over all devices into the host array / HostFrame `out`; returns the summed counters."""
        chunks_ptr, n = (None, 0) if chunks is None else (np.ascontiguousarray(chunks, dtype=CHUNK_DTYPE), len(chunks))
        self._chunks = chunks_ptr
        cnt = Counters()
        out_ptr = out.ptr if isinstance(out, HostFrame) else out.ctypes.data
        self._ck(self._lib.mm_multi_render(self._m, C.byref(uniform), C.byref(params), None if chunks_ptr is None else chunks_ptr.ctypes.data,
                                           n, out_ptr, C.byref(cnt)))
        return cnt.as_dict()

    def render_async(self, uniform, params, chunks, out_ptr):
        chunks_ptr, n = (None, 0) if chunks is None else (np.ascontiguousarray(chunks, dtype=CHUNK_DTYPE), len(chunks))
        self._chunks = chunks_ptr
        self._ck(self._lib.mm_multi_render_async(self._m, C.byref(uniform), C.byref(params),
                                                 None if chunks_ptr is None else chunks_ptr.ctypes.data, n, out_ptr))

    def wait(self):
        cnt = Counters()
        self._ck(self._lib.mm_multi_wait(self._m, C.byref(cnt)))
        return cnt.as_dict()

    def frame_device_ptr(self, index):
        p = C.c_void_p()
        self._ck(self._lib.mm_multi_frame_device(self._m, index, C.byref(p)))
        return p.value

    def selftest_div3(self):
        """Mismatches between the blur's exact x / 3 sequence and __fdiv_rn(x, 3) over all 2^32 floats (must be 0)."""
        bad = C.c_uint64()
        self._ck(self._lib.mm_selftest_div3(self._ctx, C.byref(bad)))
        return int(bad.value)

    def last_ms(self):
        ms = C.c_float()
        self._ck(self._lib.mm_multi_last_ms(self._m, C.byref(ms)))
        return float(ms.value)


class TiledFrameRenderer:
    """One rank of the multi-GPU frame: scene replicated, groups interleaved over ranks.

    `dist` is torch.distributed (already initialised, backend nccl) or None for a single GPU.  Tensors are torch
    CUDA tensors used purely as device memory; the kernels are this library's.  Two ways to exchange the tiles:

    exchange="peer"   the render kernel stores each finished pixel straight into every rank's frame: the frames live in
                      torch symmetric memory, so each rank holds peer-mapped pointers to all of them (NVLink stores) and,
                      where the fabric supports it, ONE NVSwitch multicast address that replicates a single 16-B store
                      into all frames.  No gather, no scatter, the transfer overlaps the tracing; one barrier before (the
                      previous frame is no longer being read anywhere) and one after (every rank's stores have landed).
    exchange="gather" render into a compact tile buffer, NCCL all_gather_into_tensor, one scatter launch.
    exchange="auto"   "peer" when symmetric memory can be set up for this group and world <= MM_MAX_PEERS, else "gather".
    """

    MAX_PEERS = 8

    def __init__(self, renderer, uniform, params, chunks, rank=0, world=1, dist=None, exchange="auto", multicast=True):
        import torch

        self.torch = torch
        self.r = renderer
        self.uniform = uniform
        self.rank, self.world, self.dist = rank, world, dist
        self.n_groups = params.grid_x * params.grid_y
        self.ppc = uniform.chunk_width ** 2
        self.H, self.W = int(uniform.view_height), int(uniform.view_width)
        dev = torch.device("cuda", renderer.device)
        self.parts = [tile_partition(self.n_groups, r, world) for r in range(world)]
        self.max_count = max(p[2] for p in self.parts)
        first, step, count = self.parts[rank]
        self.my = Params.from_buffer_copy(bytes(params))
        self.my.group_first, self.my.group_step, self.my.group_count = first, step, count
        if exchange not in ("auto", "peer", "gather"):
            raise ValueError("exchange must be 'auto', 'peer' or 'gather'")
        # One stream for the kernel, the collective / barriers and the scatter: a dedicated torch stream (the legacy
        # default stream's handle is 0, which mm_set_stream reads as "use the context's own stream").
        self.stream = torch.cuda.Stream(dev)
        self.exchange, self.exchange_note = "none", ""
        self.handle, self.peer_ptrs, self.multicast_ptr = None, None, 0
        if world > 1 and exchange in ("auto", "peer"):
            try:
                self._setup_peer_frames(dev, multicast)
                self.exchange = "peer"
            except Exception as e:      # no symmetric memory on this system / group: fall back unless it was demanded
                if exchange == "peer":
                    raise
                self.exchange_note = f"peer exchange unavailable ({type(e).__name__}: {e})"
        if self.exchange != "peer":
            self.image = torch.zeros((self.H, self.W, 4), dtype=torch.float32, device=dev)
            if world > 1:
                self.exchange = "gather"
                self.tiles = torch.zeros((self.max_count, self.ppc, 4), dtype=torch.float32, device=dev)
                # concatenated all-gather layout [world * max_count, ppc, 4]; rank r's tiles are rows r*max_count ...
                self.gathered = torch.zeros((world * self.max_count, self.ppc, 4), dtype=torch.float32, device=dev)
        renderer.set_stream(self.stream.cuda_stream)
        renderer.set_chunks(chunks)

    def _setup_peer_frames(self, dev, multicast):
        import torch.distributed._symmetric_memory as symm

        if self.world > self.MAX_PEERS:
            raise RuntimeError(f"world {self.world} > MM_MAX_PEERS {self.MAX_PEERS}")
        self.image = symm.empty((self.H, self.W, 4), dtype=self.torch.float32, device=dev)
        self.image.zero_()
        self.handle = symm.rendezvous(self.image, self.dist.group.WORLD)
        mc = int(self.handle.multicast_ptr) if multicast else 0
        self.multicast_ptr = mc
        if mc:
            self.peer_ptrs, self.exchange_note = [mc], "NVSwitch multicast stores (multimem.st)"
        else:
            self.peer_ptrs, self.exchange_note = [int(p) for p in self.handle.buffer_ptrs], "NVLink peer stores"
        self.torch.cuda.synchronize(dev)
        self.dist.barrier()

    def render_frame(self, uniform=None):
        """Renders this rank's share and assembles the full frame on every rank (asynchronous on self.stream)."""
        u = uniform if uniform is not None else self.uniform
        if self.world == 1:
            self.r.render_device(u, self.my, image_ptr=self.image.data_ptr())
            return self.image
        if self.exchange == "peer":
            with self.torch.cuda.stream(self.stream):
                self.handle.barrier(channel=0)          # every rank is done reading its previous frame
            if self.my.group_count:
                if self.multicast_ptr:
                    self.r.render_multicast_device(u, self.my, self.multicast_ptr)
                else:
                    self.r.render_peers_device(u, self.my, self.peer_ptrs)
            with self.torch.cuda.stream(self.stream):
                self.handle.barrier(channel=1)          # every rank's stores have landed in this rank's frame
            return self.image
        if self.my.group_count:
            self.r.render_device(u, self.my, tiles_ptr=self.tiles.data_ptr())
        with self.torch.cuda.stream(self.stream):
            self.dist.all_gather_into_tensor(self.gathered, self.tiles)
        self.r.scatter_gathered_device(u, self.my, self.world, self.max_count, self.gathered.data_ptr(), self.image.data_ptr())
        return self.image
