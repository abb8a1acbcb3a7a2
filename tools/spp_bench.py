"""High sample counts on one GPU: the 1024-thread block shape (spp 512 and 1024) against spp 256's 256-thread blocks.

Workload: the 32x32 maze at 1920x1080, 8 bounces, mirror limit 15, the default pose.  Shapes, as (chunk_width, spp):
(2, 256), (1, 512), (1, 1024) (the reference's one-pixel-per-threadgroup dispatch at 1024 samples) and (4, 1024); each with
the straggler tail on and under MM_FLAG_NO_TAIL.  After one warm-up launch of every arm, the arms alternate, --rounds times.
Every line is JSON: first the card (name, power limit, max SM clock, read with nvidia-smi in this call), then one line per
timed launch with its device time (mm_last_ms: trace kernel plus tail kernel), Grays/s from the `rays` counter, and the
tail's queued paths and deferred pixels (mm_last_tail), then per shape a check of a group range (a crop of the frame) against
a CPU reference, bit for bit: image, counters and the per-path arrays.  The reference is the C++ oracle up to spp 256, its
range, and oracle/np_oracle.py above it (tests/test_high_spp.py pins the two together path by path).  The whole 1024-spp
frame is about 17 G rays, hours in numpy, hence the crop.  Needs a GPU; there is no CPU path.

  python tools/spp_bench.py --rounds 3 --out /tmp/spp.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import mirror_maze_b200 as mm  # noqa: E402

SHAPES = [(2, 256), (1, 512), (1, 1024), (4, 1024)]
ARMS = [("tail", 0), ("no_tail", mm.FLAG_NO_TAIL)]


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, power, max_sm, sm = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": max_sm, "sm_clock_at_start": sm}
    except Exception as e:                       # the measurement still stands; say that the card was not read
        return {"gpu": None, "note": f"nvidia-smi query failed: {type(e).__name__}: {e}"}


def crop_check(r, sc, noise, u, p, ch, crop_paths):
    """A contiguous group range from the middle of the frame, about crop_paths paths, against the CPU reference, tail on and
    off."""
    from oracle import np_oracle, oracle

    T = u.chunk_width ** 2 * p.spp
    n_groups = p.grid_x * p.grid_y
    q = mm.Params.from_buffer_copy(bytes(p))
    q.group_count = max(1, min(n_groups, crop_paths // T))
    q.group_first = (n_groups - q.group_count) // 2
    q.group_step = 1
    if p.spp <= 256:
        ref_img, ref_cnt, ref_dbg = oracle.render(sc, noise, u, q, ch, debug=True)
    else:
        ref_img, ref_cnt, ref_dbg = np_oracle.render(sc, noise, u, q, ch)
    out = {"groups": [int(q.group_first), 1, int(q.group_count)], "paths": int(q.group_count) * T,
           "reference": "oracle/mm_oracle.cpp" if p.spp <= 256 else "oracle/np_oracle.py"}
    for arm, flags in ARMS:
        q.flags = flags
        hf = mm.HostFrame(int(u.view_height), int(u.view_width))
        try:
            img, cnt, dbg = r.render(u, q, ch, out=hf.array, debug=True)
            same = img.tobytes() == ref_img.tobytes() and all(cnt[k] == ref_cnt[k] for k in ("paths", "rays", "hits", "max_stack")) \
                and all(dbg[k].tobytes() == np.ascontiguousarray(ref_dbg[k], dtype=dbg[k].dtype).tobytes() for k in dbg)
        finally:
            hf.close()
        out[arm] = {"bit_identical": bool(same), "tail": list(r.last_tail())}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--maze", type=int, default=32)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--bounces", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--crop-paths", type=int, default=1 << 18, help="paths of the reference-checked group range per shape")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()

    sink = open(a.out, "a") if a.out else None

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if sink:
            sink.write(s + "\n")
            sink.flush()

    W, H = a.width, a.height
    emit({"kind": "card", **card(), "workload": f"maze {a.maze}, {W}x{H}, {a.bounces} bounces, mirror limit 15"})
    noise = mm.load_noise()
    sc = mm.MazeScene(a.maze, 0)
    r = mm.Renderer(0)
    r.upload_scene(sc, noise)
    frame = mm.HostFrame(H, W)
    setups = {}
    for chunk, spp in SHAPES:
        u = mm.default_uniform(a.maze, W, H, chunk)
        setups[(chunk, spp)] = (u, mm.full_frame_params(u, spp=spp, bounce_limit=a.bounces, mirror_limit=15), mm.gen_chunks(W, H, chunk))

    def launch(chunk, spp, flags):
        u, p, ch = setups[(chunk, spp)]
        q = mm.Params.from_buffer_copy(bytes(p))
        q.flags = flags
        cnt = r.render(u, q, ch, out=frame.array)[1]
        info = r.scene_info()
        return cnt, r.last_ms(), r.last_tail(), info

    for chunk, spp in SHAPES:                    # warm-up: module load, function attributes, tail buffers at their largest
        for _, flags in ARMS:
            launch(chunk, spp, flags)
    for rnd in range(a.rounds):
        for chunk, spp in SHAPES:
            for arm, flags in ARMS:
                cnt, ms, tail, info = launch(chunk, spp, flags)
                emit({"kind": "launch", "round": rnd, "chunk": chunk, "spp": spp, "arm": arm, "ms": round(ms, 3),
                      "grays_per_s": round(cnt["rays"] / (ms * 1e-3) / 1e9, 3), "rays": cnt["rays"], "paths": cnt["paths"],
                      "tail_queued": tail[0], "tail_deferred_pixels": tail[1], "block_threads": info["block_threads"],
                      "blocks_per_sm": info["blocks_per_sm"], "smem_bytes": info["smem_bytes"]})
    for chunk, spp in SHAPES:
        u, p, ch = setups[(chunk, spp)]
        emit({"kind": "reference_crop", "chunk": chunk, "spp": spp, **crop_check(r, sc, noise, u, p, ch, a.crop_paths)})
    emit({"kind": "card_end", **card()})
    frame.close()
    r.close()
    if sink:
        sink.close()


if __name__ == "__main__":
    main()
