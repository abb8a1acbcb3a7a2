#!/usr/bin/env python
"""bench.py — measures BASELINE.json's metric (Mrays/s and ms/frame at 1080p x 16 spp, 8 bounces) on N B200s.

A step = one frame of the hot path.  Default workload = BASELINE configs[1] (32x32 maze, 1920x1080, 16 spp, 8 bounces), the
configuration the metric is quoted on; --workload selects the other configurations (hl64 = the north-star 64x64 headline,
cfg3 = 64x64 / 4K / 64 spp / 16 bounces, cfg4 = 256x256 traversal stress, cfg5 = fly-throughs with progressive refresh).
N > 1 (one rank per GPU under torch.distributed.run): every rank renders its interleaved share of the frame's 4x4-pixel
chunk groups; the render kernel stores each finished pixel into every rank's frame through an NVSwitch multicast address /
NVLink peer mappings (--exchange peer, default) or into a tile buffer that is all-gathered over NCCL and scattered
(--exchange gather).  Total work per step is fixed as N grows ("strong" scaling: one frame, more GPUs).

  value / ms_per_step : device time (CUDA events on the launching stream, max over ranks), inputs resident in HBM.
  e2e                 : the same frame through the reference-facing C-ABI call with HOST buffers, wall clock: mm_render with
                        the uniform + parameters from the host and the frame delivered in mapped pinned HOST memory (the
                        kernel stores finished pixels straight into it over PCIe; N > 1: every rank's kernel writes its
                        share into ONE frame in shared pinned host memory, N PCIe links in parallel).  e2e.pageable is the
                        same call into an ordinary pageable buffer (staged copy + memcpy).
  roofline            : dominant kernel (trace kernel).  Top level = the BINDING bound: algorithmic FP32-pipe operations
                        (SURVEY 8 d: 50 per inner visit, 84 per rect test, exact oracle-identical counters) over the
                        kernel's CUDA-event duration against SMs x 128 lanes x max clock.  Sub-entries: hbm (algorithmic
                        bytes vs the measured HBM copy peak — not binding, the scene lives in L1/L2) and l1 (node bytes vs
                        the L1 bandwidth ceiling).
  cpu_baseline        : the CPU oracle (oracle/mm_oracle.cpp, a port of the reference's shader, -march=native build made on
                        this box) on every host core this process may use, on a bounded interleaved sample of the frame.
  parity_ok           : N > 1: sha256 of the N-GPU frame (device exchange) and of the shared host frame (e2e) == sha256 of
                        the frame rank 0 renders alone (untimed).
  mm_multi            : N > 1: the same frame through mm_multi (ONE process driving all N GPUs through the C-ABI, no torch in
                        the data path), timed by rank 0 while the other ranks' processes idle.
--impl reference      : the reference's own CPU implementation of the path = that oracle port, all host threads, rank 0
                        only, workload built with oracle/host_ref.py (no product library mapped).  (The reference's shader
                        source does compile as C++ here — oracle/_ref, which pins the port bit for bit — but it hard-wires 5
                        bounces and its own grid lookup, so it cannot run this workload.)
"""
import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the sources this imports

METRIC = "Mrays/s @1080p x16spp, 8 bounces"
UNIT = "Mrays/s"

WORKLOADS = {
    "cfg2": dict(maze=32, width=1920, height=1080, spp=16, bounces=8, note="BASELINE configs[1], the metric's configuration"),
    "hl64": dict(maze=64, width=1920, height=1080, spp=16, bounces=8, note="north-star headline: 64x64 maze"),
    "cfg3": dict(maze=64, width=3840, height=2160, spp=64, bounces=16, note="BASELINE configs[2]"),
    "cfg4": dict(maze=256, width=1920, height=1080, spp=16, bounces=8, note="BASELINE configs[3], traversal stress"),
    "cfg5": dict(maze=64, width=1920, height=1080, spp=16, bounces=8, note="BASELINE configs[4]: fly-throughs, one per GPU"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--maze", type=int, default=None, help="override the workload's maze size n")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--bounces", type=int, default=None)
    ap.add_argument("--mirror-limit", type=int, default=15)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-crop", type=int, default=0, help="CPU legs render every k-th chunk group (0 = sized from a probe so the run stays within minutes)")
    ap.add_argument("--no-extras", action="store_true", help="skip the 64x64 side measurement, mm_multi and the pageable e2e leg")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "gather"],
                    help="N > 1: fused peer/multicast stores from the render kernel, or NCCL all-gather + scatter")
    ap.add_argument("--flags", type=int, default=0, help="MM_FLAG_* for experiments (2 = literal divides for every ray, 64 = reciprocal-multiply slab arithmetic)")
    ap.add_argument("--screen", default="f32", choices=["f32", "rgba8"],
                    help="cfg5: fp32 screen and frames (default), or the reference's RGBA8Unorm screen: quantised stores, 4-byte texels read back")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frame the last timed step computed as DIR/<name>.npy (float32), "
                         "to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    w = WORKLOADS[a.workload]
    for k in ("maze", "width", "height", "spp", "bounces"):
        if getattr(a, k) is None:
            setattr(a, k, w[k])
    return a


def workload_name(a):
    return (f"{a.maze}x{a.maze} Kruskal maze (seed 0), {a.width}x{a.height}, {a.spp} spp, {a.bounces} bounces "
            f"(mirror_limit {a.mirror_limit}), chunk 4, start camera")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def algorithmic_work(cnt, spp):
    """SURVEY §8(d) per-unit figures x the exact counters of one frame."""
    bytes_ = 64 * cnt["inner_visits"] + 52 * cnt["rect_tests"] + 65 * cnt["hits"] + cnt["paths"] * (68 + 16 / spp)
    fp32_ops = 50 * cnt["inner_visits"] + 84 * cnt["rect_tests"]          # 2 slab tests x 25 ops; rect: 75 flops + 3 sqrt + 6 div
    return bytes_, fp32_ops


WHY_PORT = ("oracle/_ref (the reference's own shader compiled as C++) hard-wires bounce_limit 5 and a grid lookup valid only for "
            "grid_x = (width/2)/16, so it cannot run this workload; the port is bit-identical to it on every dispatch it can run "
            "(tests/test_ref_shader.py)")
N_CORES = len(os.sched_getaffinity(0))       # the host cores this process may use (OMP_NUM_THREADS is ignored on purpose)


def sha(a):
    return hashlib.sha256(memoryview(a).cast("B")).hexdigest()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy in float32, at most DUMP_BYTES in all.  An array over its share
    (a 4K frame) is stored as a fixed seeded sample of its pixels, [n, channels], with their flat pixel indices beside it
    as <name>_index.npy (float64, exact)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096                    # room for the .npy headers
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            px = a.reshape(-1, a.shape[-1])
            n = share // (px.shape[1] * 4 + 8)
            idx = np.sort(np.random.default_rng(0).choice(len(px), n, replace=False))
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
            a = px[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---- CPU legs (oracle; the only place bench.py executes oracle/) -----------------------------------------------------------

class _Scene:
    pass


def reference_inputs(a):
    """The workload built WITHOUT the product library: oracle/host_ref.py (scene, uniform, chunk list) and the C-ABI's ctypes
    struct definitions (pure Python)."""
    import gzip
    import numpy as np
    from oracle import host_ref
    from mirror_maze_b200 import abi            # struct layouts only; abi.load_library() is never called on this path

    sc = _Scene()
    if a.maze <= 64:
        d = host_ref.build_scene(a.maze, 0)
        sc.planes, sc.nodes, sc.indices, sc.materials, sc.emissions = d["planes"], d["nodes"], d["indices"], d["materials"], d["emissions"]
    else:                                       # the Python BVH build is quadratic per node: hours at n = 256; use the C++ host surface there
        import mirror_maze_b200 as mm
        m = mm.MazeScene(a.maze, 0)
        sc.planes, sc.nodes, sc.indices, sc.materials, sc.emissions = m.planes, m.nodes, m.indices, m.materials, m.emissions
    u = abi.Uniform.from_buffer_copy(host_ref.default_uniform_bytes(a.maze, a.width, a.height, 4, 0))
    chunks = host_ref.gen_chunks(a.width, a.height, 4)
    p = abi.Params(spp=a.spp, bounce_limit=a.bounces, mirror_limit=a.mirror_limit, grid_x=a.width // 4, grid_y=a.height // 4,
                   group_first=0, group_step=1, group_count=0, flags=a.flags & 64)          # same arithmetic mode
    with gzip.open(os.path.join(ROOT, "mirror_maze_b200", "assets", "noiseTexture-2.rgba8.gz"), "rb") as f:
        noise = np.frombuffer(f.read(), dtype=np.uint8).reshape(512, 512, 4).copy()
    return sc, u, p, chunks, noise


def cpu_reference_run(a, steps, warmup, inputs=None, budget_s=120.0):
    """Times the oracle port on the host cores over a bounded interleaved sample of the frame: every k-th chunk group, k
    sized from a short probe so that warmup + steps take about budget_s seconds.  Returns (Mrays/s, info)."""
    import numpy as np
    from oracle import oracle

    build = oracle.use_native()
    sc, u, p, chunks, noise = inputs if inputs is not None else reference_inputs(a)
    n_groups = p.grid_x * p.grid_y
    out = np.zeros((a.height, a.width, 4), dtype=np.float32)

    def render(stride):
        p.group_first, p.group_step = 0, stride
        p.group_count = (n_groups + stride - 1) // stride
        t0 = time.perf_counter()
        _, cnt, _ = oracle.render(sc, noise, u, p, chunks, threads=N_CORES, out=out)
        return time.perf_counter() - t0, cnt["rays"]

    stride = a.cpu_crop
    if stride <= 0:
        probe = max(1, n_groups // 2048)
        render(probe)                                                    # first touch: threads, pages
        dt, rays = render(probe)
        frame_s = dt * probe                                             # whole-frame time at the probed rate
        stride = max(1, int(np.ceil(frame_s / (budget_s / max(1, steps + warmup)))))
    times, rays = [], 0
    for i in range(warmup + steps):
        u.time = i
        dt, n = render(stride)
        if i >= warmup:
            times.append(dt); rays += n
    total = sum(times)
    sample = (f"every {p.group_step}th 4x4-chunk group of the frame ({p.group_count} of {n_groups} groups, "
              f"{rays // max(1, steps)} rays per step), {steps} steps")
    return rays / total / 1e6, {"cores": N_CORES, "sample": sample, "ms_per_step": 1e3 * total / max(1, steps),
                                "rays_per_step": rays // max(1, steps), "build": build}


def reference_shader_on_its_own_dispatch():
    """The compiled reference shader (oracle/_ref) and the port, timed on the one workload the unmodified shader can run at
    scale: its own dispatch (10x10 maze, 1024x768, 64 spp, 5 bounces, 768 chunks).  Informational: shows that the port the
    reference arm times is not slower than the reference's own code.  None when the library is not present."""
    try:
        from oracle import oracle, ref_shader, host_ref
        from mirror_maze_b200 import abi
        if not ref_shader.available():
            return None
        a = argparse.Namespace(maze=10, width=1024, height=768, spp=64, bounces=5, mirror_limit=15, flags=0)
        sc, u, p, chunks, noise = reference_inputs(a)
        u.time = 3
        p.grid_x, p.grid_y = 32, 24
        chunks = chunks[: 32 * 24].copy()
        t0 = time.perf_counter(); img, cnt, _ = oracle.render(sc, noise, u, p, chunks, threads=N_CORES); t_port = time.perf_counter() - t0
        t0 = time.perf_counter(); ref = ref_shader.render(sc, noise, u, p, chunks); t_ref = time.perf_counter() - t0
        return {"workload": "the reference's own dispatch: 10x10 maze, 1024x768, 64 spp, 5 bounces, 768 chunks", "rays": cnt["rays"],
                "reference_shader_Mrays_s": round(cnt["rays"] / t_ref / 1e6, 3), "port_Mrays_s": round(cnt["rays"] / t_port / 1e6, 3),
                "images_identical": bool(img.tobytes() == ref.tobytes())}
    except Exception as e:                      # informational only
        return {"error": f"{type(e).__name__}: {e}"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    val, info = cpu_reference_run(a, max(1, a.steps), max(0, a.warmup))
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(info["ms_per_step"], 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload_name(a), "note": "ms_per_step is for the bounded sample, not the whole frame"},
            "cpu_baseline": {"value": round(val, 3), "unit": UNIT, "cores": info["cores"], "kind": "port", "sample": info["sample"],
                             "build": info["build"], "why_port": WHY_PORT},
            "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    check = reference_shader_on_its_own_dispatch()
    if check is not None:
        line["cpu_baseline"]["reference_shader_check"] = check
    print(json.dumps(line), flush=True)
    return 0


# ---- GPU legs -----------------------------------------------------------------------------------------------------------------

class SharedHostFrame:
    """One frame buffer in host memory shared by every rank of the node (a file in /dev/shm mapped by all), pinned and mapped
    into each rank's CUDA context with mm_host_register: every rank's kernel stores its pixels straight into it."""

    def __init__(self, mm, name, nbytes, create, register=True):
        import mmap
        import numpy as np
        if os.environ.get("MM_BENCH_NO_SHM"):                      # test hook for the fallback leg
            raise OSError("shared host frame disabled by MM_BENCH_NO_SHM")
        self.path = os.path.join("/dev/shm", name)
        if create:
            with open(self.path, "wb") as f:
                f.truncate(nbytes)
        self.f = open(self.path, "r+b")
        self.map = mmap.mmap(self.f.fileno(), nbytes)
        self.array = np.frombuffer(self.map, dtype=np.float32)
        self.ptr = self.array.ctypes.data
        self.lib = mm.load_library() if register else None           # register=False: CPU tests of the plumbing
        if register:
            rc = self.lib.mm_host_register(self.ptr, nbytes)
            if rc != 0:
                raise RuntimeError(f"mm_host_register on the shared frame failed: {rc}")
        self.create = create

    def close(self):
        if self.lib is not None:
            self.lib.mm_host_unregister(self.ptr)
        self.array = None
        try:
            self.map.close()
        except BufferError:
            pass
        self.f.close()
        if self.create:
            try:
                os.unlink(self.path)
            except OSError:
                pass


def time_frames(r, frame, u, steps, warmup, flush, dist, torch, t0_time=0):
    """Device-timed frames (CUDA events on the launching stream, L2 flushed between iterations).  Returns per-step ms, the
    mean kernel ms of this rank and the rays this rank traced."""
    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup):
        u.time = t0_time + i
        flush.fill_(i & 255)
        frame.render_frame(u)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kernel_ms, rays = [], 0
    for i in range(steps):
        u.time = t0_time + warmup + i
        flush.fill_(i & 255)                       # L2 flush between timed iterations (outside the event pair)
        if dist is not None:
            dist.barrier()
        ev[i][0].record()
        frame.render_frame(u)
        ev[i][1].record()
        ev[i][1].synchronize()
        if frame.my.group_count:
            kernel_ms.append(r.last_ms())
            rays += r.last_counters()["rays"]
    barrier()
    return [s.elapsed_time(e) for s, e in ev], (statistics.mean(kernel_ms) if kernel_ms else 0.0), rays


def run_ours(a):
    import numpy as np
    import torch

    import mirror_maze_b200 as mm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch N > 1 with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the render path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    if a.workload == "cfg5":
        return run_flythroughs(a, mm, torch, dist, rank, world, local)

    noise = mm.load_noise()
    scene = mm.MazeScene(a.maze, 0)
    u = mm.default_uniform(a.maze, a.width, a.height, 4)
    chunks = mm.gen_chunks(a.width, a.height, 4)
    p = mm.full_frame_params(u, spp=a.spp, bounce_limit=a.bounces, mirror_limit=a.mirror_limit, flags=a.flags)
    r = mm.Renderer(local)
    r.upload_scene(scene, noise)
    frame = mm.TiledFrameRenderer(r, u, p, chunks, rank=rank, world=world, dist=dist, exchange=a.exchange)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)        # > 126 MB L2
    H, W = a.height, a.width

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # exact event counts of this rank's share (deterministic; counted once with the counting kernel variant, untimed)
    pc = mm.Params.from_buffer_copy(bytes(frame.my)); pc.flags = a.flags | mm.FLAG_COUNTERS
    if pc.group_count:
        scratch = torch.zeros((frame.max_count, frame.ppc, 4), dtype=torch.float32, device=dev)
        r.render_device(u, pc, tiles_ptr=scratch.data_ptr())
    r.sync()
    zero = {k: 0 for k in ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits", "literal_rays", "max_stack")}
    my_cnt = r.last_counters() if pc.group_count else zero

    torch.cuda.set_stream(frame.stream)            # every torch op below (flush, events, collectives) shares the kernel's stream
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    step_ms, kernel_mean, rays_timed = time_frames(r, frame, u, a.steps, a.warmup, flush, dist, torch)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"frame": frame.image.cpu().numpy()})        # the last timed step's whole frame
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    rays_all = torch.tensor([float(rays_timed)], dtype=torch.float64, device=dev)
    keys = ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits", "literal_rays")
    cnt_vec = torch.tensor([float(my_cnt[k]) for k in keys], dtype=torch.float64, device=dev)
    kms = torch.tensor([kernel_mean], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays_all, op=dist.ReduceOp.SUM)
        dist.all_reduce(cnt_vec, op=dist.ReduceOp.SUM)
        dist.all_reduce(kms, op=dist.ReduceOp.MAX)
    total_ms, rays_all, kernel_mean_ms = float(total_ms.item()), float(rays_all.item()), float(kms.item())
    cnt_frame = dict(zip(keys, [int(v) for v in cnt_vec.tolist()]))

    # ---- parity of the timed N-GPU frame: against the frame rank 0 renders alone (untimed) --------------------------------
    parity = None
    single_sha = None
    if world > 1:
        u.time = 4242
        img = frame.render_frame(u)
        frame.stream.synchronize()
        multi_sha = sha(img.cpu().numpy()) if rank == 0 else None
        if rank == 0:
            solo = mm.Renderer(local)
            solo.upload_scene(scene, noise)
            single = np.zeros((H, W, 4), dtype=np.float32)
            solo.render(u, p, chunks, out=single)
            solo.close()
            single_sha = sha(single)
            parity = {"device_exchange_frame": multi_sha == single_sha}
        barrier()

    # ---- e2e: host uniform/params in, frame delivered in HOST memory, wall clock ------------------------------------------
    e2e_steps = max(3, min(a.steps, 10))
    e2e_rays = 0
    frame_bytes = H * W * 16
    h2d = ctypes.sizeof(mm.Uniform) + ctypes.sizeof(mm.Params)          # the chunk list goes up once, before the timed region: it
    e2e_extra = {}                                                       # does not change from frame to frame (chunks = NULL keeps it)
    r.set_stream(None)                                                   # the context's own stream again
    torch.cuda.synchronize()
    if world == 1:
        hf = mm.HostFrame(H, W)
        chunk_arr = np.ascontiguousarray(chunks)
        r.render_into(u, p, chunk_arr.ctypes.data, len(chunk_arr), hf.ptr)
        r.render_into(u, p, None, 0, hf.ptr)
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            u.time = 1000 + i
            c = r.render_into(u, p, None, 0, hf.ptr)                     # mm_render: kernel stores pixels into the pinned host frame
            e2e_rays += c["rays"]
        e2e_s = time.perf_counter() - t0
        d2h = frame_bytes + ctypes.sizeof(mm.Counters)
        e2e_api = "mm_render (host uniform + params in; frame in mapped pinned host memory from mm_host_alloc, written by the kernel's zero-copy stores)"
        if not a.no_extras:
            # the same call with the buffer kinds a caller may have: pinned + DMA copy, and an ordinary pageable array (staged)
            q = mm.Params.from_buffer_copy(bytes(p)); q.flags = a.flags | mm.FLAG_NO_ZERO_COPY
            r.render_into(u, q, None, 0, hf.ptr)
            t1 = time.perf_counter()
            for i in range(e2e_steps):
                r.render_into(u, q, None, 0, hf.ptr)
            dma_ms = 1e3 * (time.perf_counter() - t1) / e2e_steps
            pageable = np.zeros((H, W, 4), dtype=np.float32)
            r.render_into(u, p, None, 0, pageable.ctypes.data)
            t1 = time.perf_counter()
            for i in range(e2e_steps):
                r.render_into(u, p, None, 0, pageable.ctypes.data)
            pg_ms = 1e3 * (time.perf_counter() - t1) / e2e_steps
            e2e_extra = {"pinned_dma_copy_ms_per_step": round(dma_ms, 4), "pageable_staged_ms_per_step": round(pg_ms, 4),
                         "frames_identical": bool(sha(hf.array) == sha(pageable))}
        hf.close()
    else:
        port = os.environ.get("MASTER_PORT", "0")
        shared, shared_err = None, ""
        try:
            if rank == 0:
                shared = SharedHostFrame(mm, f"mm_bench_frame_{port}", frame_bytes, create=True)
        except Exception as e:
            shared_err = f"{type(e).__name__}: {e}"
        barrier()
        try:
            if rank != 0:
                shared = SharedHostFrame(mm, f"mm_bench_frame_{port}", frame_bytes, create=False)
        except Exception as e:
            shared_err = f"{type(e).__name__}: {e}"
        ok_all = torch.tensor([1 if shared is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
        use_shared = int(ok_all.item()) == 1
        if not use_shared and shared is not None:
            shared.close(); shared = None
        mine = mm.Params.from_buffer_copy(bytes(frame.my))
        chunk_arr = np.ascontiguousarray(chunks)
        if use_shared:
            if mine.group_count:
                r.render_into(u, mine, chunk_arr.ctypes.data, len(chunk_arr), shared.ptr)
            barrier()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                u.time = 1000 + i
                if mine.group_count:
                    c = r.render_into(u, mine, None, 0, shared.ptr)          # this rank's groups -> the one shared host frame
                    e2e_rays += c["rays"]
                dist.barrier()
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            e2e_api = ("mm_render per rank (its interleaved groups) with out_rgba = ONE frame in shared pinned host memory (/dev/shm, "
                       "mm_host_register in every rank): each kernel stores its pixels straight into it, N PCIe links in parallel; barrier")
        else:
            # no shared pinned frame on this box (e.g. /dev/shm not writable): device exchange, then rank 0 copies the assembled
            # frame to its pinned memory (round 1's path)
            host_frame = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
            r.set_stream(frame.stream.cuda_stream)
            barrier()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                u.time = 1000 + i
                img = frame.render_frame(u)
                if rank == 0:
                    host_frame.copy_(img, non_blocking=True)
                torch.cuda.synchronize()
                e2e_rays += r.last_counters()["rays"] if frame.my.group_count else 0
            barrier()
            e2e_s = time.perf_counter() - t0
            r.set_stream(None)
            e2e_api = ("device exchange + assembled frame copied to rank 0's pinned host memory (shared pinned host frame unavailable: " + shared_err + ")")
        t = torch.tensor([e2e_s, float(e2e_rays)], dtype=torch.float64, device=dev)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e2e_s, e2e_rays = float(tmax[0].item()), int(t[1].item())
        d2h = frame_bytes + world * ctypes.sizeof(mm.Counters)
        # parity of the host frame: one more frame at the parity time stamp
        if use_shared:
            u.time = 4242
            if mine.group_count:
                r.render_into(u, mine, None, 0, shared.ptr)
            barrier()
            if rank == 0:
                parity["shared_host_frame"] = sha(shared.array) == single_sha
            barrier()
            shared.close()

    # ---- mm_multi: the same frame from ONE process over all N GPUs (rank 0 drives, the other ranks idle on the store) ------
    multi_info = None
    if world > 1 and not a.no_extras:
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                multi_info = run_mm_multi(mm, np, scene, noise, u, p, chunks, list(range(world)), single_sha, e2e_steps)
            except Exception as e:
                multi_info = {"error": f"{type(e).__name__}: {e}"}
            store.set("mm_multi_done", "1")
        else:
            store.wait(["mm_multi_done"])
        barrier()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    value = rays_all / (total_ms * 1e-3) / 1e6
    ms_per_step = total_ms / a.steps
    info = r.scene_info()
    roofline = build_roofline(a, r, info, cnt_frame, kernel_mean_ms, world, clocks)

    # ---- the north-star headline (64x64 maze, same frame size) beside the metric's configuration ---------------------------
    north = None
    if world == 1 and a.workload == "cfg2" and not a.no_extras:
        north = side_measurement(a, mm, torch, r, noise, flush, frame.stream, clocks)

    exchange_desc = (f", exchange fused into the render kernel ({frame.exchange_note})" if frame.exchange == "peer" else
                     ", NCCL all-gather + one scatter launch" + (f" [{frame.exchange_note}]" if frame.exchange_note else ""))
    line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(a), "workload_id": a.workload, "paths_per_frame": cnt_frame["paths"], "rays_per_frame": cnt_frame["rays"],
                       "parallelism": f"image tiles x{world} (interleaved 4x4-chunk groups), scene replicated" + (exchange_desc if world > 1 else ""),
                       "exchange": frame.exchange if world > 1 else None,
                       "l2_flush": "256 MiB device fill between timed iterations", "fast_slab_ok": info["fast_slab_ok"], "fast_rect_ok": info["fast_rect_ok"],
                       "blocks_per_sm": info["blocks_per_sm"], "bvh_nodes": info["n_nodes"], "planes": info["n_planes"],
                       "literal_rays_per_frame": cnt_frame["literal_rays"],
                       "arithmetic": "opt-in (b-o)*RN(1/d) slab quotients (MM_FLAG_RCP_SLAB)" if (a.flags & 64) else "IEEE fp32, slab quotients bit-identical to the literal (b-o)/d"},
            "clocks": clocks, "roofline": roofline,
            "e2e": dict({"value": round(e2e_rays / e2e_s / 1e6, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                         "ms_per_step": round(1e3 * e2e_s / e2e_steps, 4), "steps": e2e_steps, "api": e2e_api}, **e2e_extra),
            "gpu_launches": a.steps * (2 if frame.exchange == "gather" else 1), "counters": cnt_frame}
    if north is not None:
        line["config"]["north_star_64"] = north
    if parity is not None:
        line["parity_ok"] = bool(all(parity.values()))
        line["parity"] = parity
    if multi_info is not None:
        line["mm_multi"] = multi_info
    if not a.no_cpu_baseline and world == 1:
        pr = mm.Params.from_buffer_copy(bytes(p)); pr.flags = a.flags & 64
        u.time = 0
        val, cinfo = cpu_reference_run(a, 1, 0, inputs=(scene, u, pr, chunks, noise), budget_s=20.0)
        line["cpu_baseline"] = {"value": round(val, 3), "unit": UNIT, "cores": cinfo["cores"], "kind": "port", "sample": cinfo["sample"],
                                "build": cinfo["build"], "why_port": WHY_PORT}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def build_roofline(a, r, info, cnt_frame, kernel_mean_ms, world, clocks):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    alg_bytes, alg_ops = algorithmic_work(cnt_frame, a.spp)
    # per launch: one launch per rank renders 1/world of the frame; the slowest rank's kernel time bounds the step
    bytes_per_launch, ops_per_launch = alg_bytes / world, alg_ops / world
    sec = kernel_mean_ms * 1e-3
    achieved_gbs = bytes_per_launch / sec / 1e9 if sec else 0.0
    sm_max = (clocks or {}).get("sm_max_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    sm_now = (clocks or {}).get("sm_mhz") or sm_max
    issue_peak_max = info["n_sms"] * 128 * sm_max * 1e6 / 1e12            # T lane-ops/s at max clock
    issue_peak_now = info["n_sms"] * 128 * sm_now * 1e6 / 1e12            # at the clock seen under load
    achieved_tops = ops_per_launch / sec / 1e12 if sec else 0.0
    ffma_peak = r.microbench(1)                                           # measured T FP32 FMA lane-instr/s (library micro-benchmark)
    node_bytes = (64 * cnt_frame["inner_visits"] + 52 * cnt_frame["rect_tests"]) / world
    node_gbs = node_bytes / sec / 1e9 if sec else 0.0
    l1_peak = info["n_sms"] * 128 * sm_max * 1e6 / 1e9                    # GB/s: 128 B per clock per SM
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = prof.get(f"maze{a.maze}", {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    return {"bound": "fp32_issue", "achieved": round(achieved_tops, 3), "peak": round(issue_peak_max, 2), "unit": "T lane-op/s",
            "frac": round(achieved_tops / issue_peak_max, 4), "traffic": traffic,
            "traffic_note": "dram__bytes_read+write per launch from ncu --set full of this kernel and maze (profiles/traffic.json); the frame write-back only",
            "kernel": "trace kernel", "kernel_ms": round(kernel_mean_ms, 4),
            "peak_source": f"{info['n_sms']} SMs x 128 FP32 lanes x {sm_max:.0f} MHz (max SM clock); no entry for this bound in MEASURED_PEAKS.json",
            "peak_at_load_clock": round(issue_peak_now, 2), "frac_at_load_clock": round(achieved_tops / issue_peak_now, 4),
            "peak_measured_ffma": round(ffma_peak, 2), "frac_of_measured_ffma": round(achieved_tops / ffma_peak, 4) if ffma_peak else None,
            "algorithmic_ops_per_launch": int(ops_per_launch),
            "def": "ALGORITHMIC FP32-pipe operations of the reference's algorithm: 50 per inner visit (2 slab tests x 25, a divide = 1 op) + 84 per "
                   "rect test (SURVEY 8d), from the exact oracle-identical counters, over the kernel's CUDA-event time.  The kernel EXECUTES more: "
                   "each literal divide is an exact 4-instruction sequence",
            "hbm": {"achieved": round(achieved_gbs, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(achieved_gbs / hbm_peak, 4),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": int(bytes_per_launch),
                    "note": "NOT the binding bound: algorithmic node+primitive bytes are served by L1/L2 (the scene is <= 9 MB); DRAM sees only the frame (see traffic)"},
            "l1": {"achieved": round(node_gbs, 1), "peak": round(l1_peak, 1), "unit": "GB/s", "frac": round(node_gbs / l1_peak, 4),
                   "def": "algorithmic node+primitive bytes (64 B per inner visit + 52 B per rect test) over the kernel time, against the L1 ceiling "
                          "SMs x 128 B/clk x max clock"}}


def side_measurement(a, mm, torch, r, noise, flush, stream, clocks):
    """The 64x64-maze frame (north-star headline) with the same frame size / spp / bounces, device-timed like the main leg."""
    try:
        sc = mm.MazeScene(64, 0)
        r.upload_scene(sc, noise)
        u = mm.default_uniform(64, a.width, a.height, 4)
        ch = mm.gen_chunks(a.width, a.height, 4)
        p = mm.full_frame_params(u, spp=a.spp, bounce_limit=a.bounces, mirror_limit=a.mirror_limit, flags=a.flags)
        fr = mm.TiledFrameRenderer(r, u, p, ch)
        pc = mm.Params.from_buffer_copy(bytes(p)); pc.flags = a.flags | mm.FLAG_COUNTERS
        r.render_device(u, pc, image_ptr=fr.image.data_ptr())
        r.sync()
        cnt = r.last_counters()
        torch.cuda.set_stream(fr.stream)
        steps = max(3, min(a.steps, 20))
        ms, kms, rays = time_frames(r, fr, u, steps, 3, flush, None, torch)
        info = r.scene_info()
        _, ops = algorithmic_work(cnt, a.spp)
        sm_max = (clocks or {}).get("sm_max_mhz") or 1965.0
        peak = info["n_sms"] * 128 * sm_max * 1e6 / 1e12
        return {"workload": f"64x64 maze, {a.width}x{a.height}, {a.spp} spp, {a.bounces} bounces", "value": round(rays / (sum(ms) * 1e-3) / 1e6, 2),
                "unit": UNIT, "ms_per_step": round(sum(ms) / steps, 4), "steps": steps, "rays_per_frame": cnt["rays"],
                "fp32_issue_frac": round(ops / (kms * 1e-3) / 1e12 / peak, 4), "bvh_nodes": info["n_nodes"], "planes": info["n_planes"]}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def run_mm_multi(mm, np, scene, noise, u, p, chunks, devices, single_sha, steps):
    """One process, all GPUs, through the C-ABI's mm_multi: frame into mapped pinned host memory, wall clock per frame."""
    out = {}
    for exchange in ("peer", "none"):
        m = mm.MultiRenderer(devices, exchange)
        m.upload_scene(scene, noise)
        hf = mm.HostFrame(int(u.view_height), int(u.view_width))
        u.time = 4242
        m.render(u, p, chunks, hf)
        ok = sha(hf.array) == single_sha
        m.render(u, p, None, hf)
        t0 = time.perf_counter()
        rays = 0
        for i in range(steps):
            u.time = 2000 + i
            rays += m.render(u, p, None, hf)["rays"]
        dt = time.perf_counter() - t0
        out[exchange] = {"e2e_ms_per_step": round(1e3 * dt / steps, 4), "e2e_Mrays_s": round(rays / dt / 1e6, 2), "kernel_ms_max": round(m.last_ms(), 4),
                         "parity_ok": bool(ok)}
        m.close(); hf.close()
    out["api"] = "mm_multi_render: one process, one call per frame, N devices; frame in mapped pinned host memory"
    return out


def run_flythroughs(a, mm, torch, dist, rank, world, local):
    """BASELINE configs[4]: camera fly-throughs with temporal sample accumulation, one fly-through per GPU, frames batched
    across the GPUs (no exchange until the final collect).  One fly-through = the reference's frame loop (reference
    src/main.rs:767-895) run headless: scripted WASD + yaw -> mm_move_camera (collision) / mm_update_quat_angle -> pop 1/64 of the
    screen's chunk origins (progressive refresh, main.rs:778-784) -> mm_render into the persistent screen -> mm_present (5-tap
    blur) -> frame read back to pinned host memory.  A step = one frame on every GPU: --warmup untimed frames, then the
    fly-through again from its start for --steps timed frames."""
    import math
    import numpy as np

    noise = mm.load_noise()
    sc = mm.MazeScene(a.maze, 0)
    r = mm.Renderer(local)
    r.upload_scene(sc, noise)
    u = mm.default_uniform(a.maze, a.width, a.height, 4)
    n_chunks = (a.width // 4) * (a.height // 4)
    per_frame = max(1, n_chunks // 64)
    gx = max(1, int(math.sqrt(per_frame * a.width / a.height)))
    while per_frame % gx:
        gx -= 1
    rgba8 = a.screen == "rgba8"
    p = mm.Params(spp=a.spp, bounce_limit=a.bounces, mirror_limit=a.mirror_limit, grid_x=gx, grid_y=per_frame // gx,
                  flags=mm.FLAG_SCREEN_RGBA8 if rgba8 else 0)
    hf = mm.HostFrame(a.height, a.width)            # fp32 frames; in the rgba8 mode their first quarter holds the texel bytes
    hf2 = mm.HostFrame(a.height, a.width)
    texels = np.zeros((a.height, a.width, 4), dtype=np.uint8)

    def fly(seed, frames, check=None):
        bag = mm.ChunkBag(a.width, a.height, 4, seed=1000 + seed)
        uu = mm.Uniform.from_buffer_copy(bytes(u))
        q = np.array([uu.cam.rotation.x, uu.cam.rotation.y, uu.cam.rotation.z, uu.cam.rotation.w], dtype=np.float32)
        half_theta = math.acos(float(q[3]))
        center = np.array([uu.cam.camera_center.x, uu.cam.camera_center.y, uu.cam.camera_center.z], dtype=np.float32)
        rng = np.random.default_rng(seed)
        rays = 0
        for f in range(frames):
            center, b = mm.move_camera(sc.nodes, center, q, [13], fps=60.0)          # hold W
            if b or f % 30 == 29:                                                   # turn when blocked, and now and then
                half_theta = (half_theta - float(rng.uniform(-0.6, 0.6))) % math.pi     # main.rs:923-924 rem_euclid(PI)
                nq = mm.update_quat_angle(q, half_theta)
                if not np.isnan(nq).any():                                              # main.rs:830-841
                    q = nq
                    bag.reshuffle()
            uu.cam.camera_center = mm.Float3(*[float(v) for v in center])
            uu.cam.rotation = mm.Float4(*[float(v) for v in q])
            uu.time = f
            ch = bag.next(per_frame)
            rays += r.render_into(uu, p, ch.ctypes.data, len(ch), None)["rays"]   # compute pass into the persistent screen
            if check is not None:
                if rgba8:
                    r.present_rgba8(hf.array, texels)                           # quantising blur; float frame and texel bytes
                else:
                    r.present(hf.array)                                         # present pass (blur) + read-back, synchronous
                check(f, uu, ch)
            elif rgba8:
                r.present_async_rgba8((hf if f & 1 else hf2).ptr)               # 4 bytes per pixel back to the host
            else:
                # present pass without the wait (main.rs:888-894): the frame's read-back overlaps the next frame's dispatch;
                # two pinned host frames alternate
                r.present_async((hf if f & 1 else hf2).ptr)
        r.wait_present()
        return rays

    if a.warmup:
        fly(rank, a.warmup)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rays = fly(rank, a.steps)
    dt = time.perf_counter() - t0
    if a.dump_outputs and rank == 0:
        last = hf if (a.steps - 1) & 1 else hf2                                  # the alternating read-back frames
        if rgba8:
            H, W = a.height, a.width
            dump_outputs(a.dump_outputs, {"texels": last.array.reshape(-1).view(np.uint8)[:H * W * 4].reshape(H, W, 4)})
        else:
            dump_outputs(a.dump_outputs, {"frame": last.array})
    # parity: the first 3 frames of this rank's fly-through against the oracle + the blur model, on a fresh renderer state —
    # AFTER the timed run: the oracle's OpenMP workers keep spinning for a while and would steal the cores the frame loop needs
    parity_ok = None
    if not a.no_cpu_baseline:
        from oracle import oracle
        model = np.zeros((a.height, a.width, 4), dtype=np.float32)
        ok = [True]

        def blur(img):
            z = np.zeros_like(img)
            rt, lf, dn, up = z.copy(), z.copy(), z.copy(), z.copy()
            rt[:, :-1], lf[:, 1:], dn[:-1], up[1:] = img[:, 1:], img[:, :-1], img[1:], img[:-1]
            c = (img + (rt + lf) / np.float32(2.0) + (dn + up) / np.float32(2.0)) / np.float32(3.0)
            c[..., 3] = 1.0
            return c.astype(np.float32)

        def check(f, uu, ch):
            nonlocal model
            if f >= 3:
                return
            q = mm.Params.from_buffer_copy(bytes(p))
            oracle.render(sc, noise, uu, q, ch, out=model)
            model = blur(model)
            if rgba8:
                from oracle import np_oracle
                model = np_oracle.quant8(model)
                ok[0] = ok[0] and np.array_equal(texels, np.rint(model * np.float32(255.0)).astype(np.uint8))
            ok[0] = ok[0] and model.tobytes() == hf.array.tobytes()

        r.close()
        r = mm.Renderer(local)
        r.upload_scene(sc, noise)
        fly(rank, 3, check)
        parity_ok = ok[0]
    tot = np.array([rays, a.steps, dt, 1.0 if parity_ok in (True, None) else 0.0], dtype=np.float64)
    if dist is not None:
        t = torch.tensor(tot, device=f"cuda:{local}")
        mx, mn = t.clone(), t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        tot = np.array([t[0].item(), t[1].item(), mx[2].item(), mn[3].item()])
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps({"metric": "frames/s, fly-throughs with temporal accumulation (BASELINE configs[4])", "value": round(tot[1] / tot[2], 2), "unit": "frames/s",
                          "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1e3 * tot[2] / a.steps, 4), "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": f"{world} fly-through(s) x {a.steps} frames, {a.maze}x{a.maze} maze, {a.width}x{a.height}, {a.spp} spp, {a.bounces} bounces, "
                                                 f"1/64 of the screen ({per_frame} chunks) re-rendered per frame + 5-tap present blur, every frame read back to pinned host memory "
                                                 f"(mm_present_async: the read-back overlaps the next frame's dispatch)",
                                     "workload_id": "cfg5", "parallelism": "one fly-through per GPU, no exchange until the final collect"},
                          "Mrays_per_s": round(tot[0] / tot[2] / 1e6, 1), "parity_ok": bool(tot[3] == 1.0) if parity_ok is not None else None,
                          "parity": "first 3 frames of every rank's fly-through == oracle render + blur model, bit for bit",
                          "screen": "RGBA8Unorm like the reference's (main.rs:702-709): quantised stores, texel bytes read back" if rgba8 else "fp32",
                          "e2e": {"value": round(tot[1] / tot[2], 2), "unit": "frames/s", "h2d_bytes_per_step": per_frame * 8 + 92,
                                  "d2h_bytes_per_step": a.width * a.height * (4 if rgba8 else 16)},
                          "gpu_launches": int(2 * a.steps)}), flush=True)
    return 0


if __name__ == "__main__":
    args = parse_args()
    sys.exit(run_reference(args) if args.impl == "reference" else run_ours(args))
