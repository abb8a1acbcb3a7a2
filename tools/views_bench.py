"""K camera fly-throughs on one GPU: K contexts with one launch per view (arm A) against one context with one launch for all
views (arm B, mm_render_views + mm_present_views).

Config 5's shape (BASELINE configs[4]): the 64x64 maze at 1920x1080, 16 spp, 8 bounces; every frame re-renders 1/64 of the
screen's chunks into each view's persistent screen, then the present blur runs and every view's frame is read back to pinned
host memory.  The camera script is bench.py's cfg5 one (hold W through mm_move_camera, a new yaw when blocked and every 30
frames, a ChunkBag per fly-through); view v flies seed v.  A step is one frame of every view:

  A  K Renderers, each: render_into (mm_render) + present_async / present_async_rgba8  (today's per-view loop)
  B  one Renderer:      render_views (mm_render_views) + present_views                  (one trace launch, one blur launch)

For every screen format and K the arms alternate, each from fresh contexts (zero screens), --rounds times.  Every line is JSON:
first the card (name, power limit, max SM clock, read with nvidia-smi in this call), then one line per timed run and one per
(screen, K) saying whether the last step's K frames of A and B are equal byte for byte.  Needs a GPU; there is no CPU path.

  python tools/views_bench.py --ks 1,2,4,8 --steps 120 --warmup 10 --rounds 2 --out /tmp/views.jsonl
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import mirror_maze_b200 as mm  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, power, max_sm, sm = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": max_sm, "sm_clock_at_start": sm}
    except Exception as e:                       # the measurement still stands; say that the card was not read
        return {"gpu": None, "note": f"nvidia-smi query failed: {type(e).__name__}: {e}"}


class Fly:
    """bench.py's cfg5 camera script for one fly-through (seed): position, yaw and chunk bag, one frame at a time."""

    def __init__(self, scene, u, W, H, per_frame, seed):
        self.nodes, self.per_frame = scene.nodes, per_frame
        self.bag = mm.ChunkBag(W, H, 4, seed=1000 + seed)
        self.u = mm.Uniform.from_buffer_copy(bytes(u))
        self.q = np.array([u.cam.rotation.x, u.cam.rotation.y, u.cam.rotation.z, u.cam.rotation.w], dtype=np.float32)
        self.half_theta = math.acos(float(self.q[3]))
        self.center = np.array([u.cam.camera_center.x, u.cam.camera_center.y, u.cam.camera_center.z], dtype=np.float32)
        self.rng = np.random.default_rng(seed)

    def next(self, f):
        self.center, b = mm.move_camera(self.nodes, self.center, self.q, [13], fps=60.0)       # hold W
        if b or f % 30 == 29:                                                                   # turn when blocked, and now and then
            self.half_theta = (self.half_theta - float(self.rng.uniform(-0.6, 0.6))) % math.pi
            nq = mm.update_quat_angle(self.q, self.half_theta)
            if not np.isnan(nq).any():
                self.q = nq
                self.bag.reshuffle()
        self.u.cam.camera_center = mm.Float3(*[float(v) for v in self.center])
        self.u.cam.rotation = mm.Float4(*[float(v) for v in self.q])
        self.u.time = f
        return mm.Uniform.from_buffer_copy(bytes(self.u)), self.bag.next(self.per_frame)


def run_arm(arm, K, scene, noise, u, p, W, H, per_frame, frames, steps, warmup, rgba8):
    """warmup + steps frames of K fly-throughs; returns (wall s of the timed steps, summed mm_last_ms of the timed steps,
    rays of the timed steps, the frames the last step read back)."""
    rs = [mm.Renderer(0) for _ in range(K if arm == "A" else 1)]
    for r in rs:
        r.upload_scene(scene, noise)
    flies = [Fly(scene, u, W, H, per_frame, v) for v in range(K)]
    t0 = dev_ms = 0.0
    rays = 0
    for f in range(warmup + steps):
        if f == warmup:
            for r in rs:
                r.wait_present()
            dev_ms, rays, t0 = 0.0, 0, time.perf_counter()
        views = [fl.next(f) for fl in flies]
        outs = [frames[v][f & 1] for v in range(K)]
        if arm == "A":
            for v, (r, (uu, ch)) in enumerate(zip(rs, views)):
                rays += r.render_into(uu, p, ch.ctypes.data, len(ch), None)["rays"]
                dev_ms += r.last_ms()
                (r.present_async_rgba8 if rgba8 else r.present_async)(outs[v].ptr)
        else:
            r = rs[0]
            rays += r.render_views([uu for uu, _ in views], p, [ch for _, ch in views])[1]["rays"]
            dev_ms += r.last_ms()
            r.present_views(outs, rgba8=rgba8)
    for r in rs:
        r.wait_present()
    wall = time.perf_counter() - t0
    last = (warmup + steps - 1) & 1
    nbytes = W * H * (4 if rgba8 else 16)
    got = [frames[v][last].array.reshape(-1).view(np.uint8)[:nbytes].copy() for v in range(K)]
    for r in rs:
        r.close()
    return wall, dev_ms, rays, got


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--screens", default="f32,rgba8")
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--maze", type=int, default=64)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--bounces", type=int, default=8)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    ks = [int(k) for k in a.ks.split(",")]
    W, H = a.width, a.height
    out = open(a.out, "a") if a.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    noise = mm.load_noise()
    scene = mm.MazeScene(a.maze, 0)
    u = mm.default_uniform(a.maze, W, H, 4)
    per_frame = max(1, (W // 4) * (H // 4) // 64)
    gx = max(1, int(math.sqrt(per_frame * W / H)))
    while per_frame % gx:
        gx -= 1
    emit({"tool": "views_bench", **card(), "workload": f"{a.maze}x{a.maze} maze, {W}x{H}, {a.spp} spp, {a.bounces} bounces, "
          f"{per_frame} chunks (1/64 of the screen) per view-frame, present blur + read-back of every view-frame",
          "grid": [gx, per_frame // gx], "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds})
    frames = [[mm.HostFrame(H, W), mm.HostFrame(H, W)] for _ in range(max(ks))]      # fp32 frames; rgba8 uses their first quarter
    for screen in a.screens.split(","):
        rgba8 = screen == "rgba8"
        p = mm.Params(spp=a.spp, bounce_limit=a.bounces, mirror_limit=15, grid_x=gx, grid_y=per_frame // gx,
                      flags=mm.FLAG_SCREEN_RGBA8 if rgba8 else 0)
        for K in ks:
            last = {}
            for rnd in range(a.rounds):
                for arm in ("A", "B"):
                    wall, dev_ms, rays, got = run_arm(arm, K, scene, noise, u, p, W, H, per_frame, frames, a.steps, a.warmup, rgba8)
                    last[arm] = got
                    emit({"screen": screen, "K": K, "arm": arm, "round": rnd,
                          "view_frames_per_s": round(K * a.steps / wall, 1), "ms_per_step": round(1e3 * wall / a.steps, 4),
                          "trace_device_ms_per_step": round(dev_ms / a.steps, 4), "Mrays_per_s": round(rays / wall / 1e6, 1),
                          "launches_per_step": {"A": 2 * K, "B": 2}[arm],
                          "d2h_bytes_per_step": K * W * H * (4 if rgba8 else 16)})
            emit({"screen": screen, "K": K, "last_step_frames_equal": all(x.tobytes() == y.tobytes() for x, y in zip(last["A"], last["B"]))})
    for fr in frames:
        for h in fr:
            h.close()
    if out:
        out.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
