"""Developer tool (CPU): how much of the segment-synchronous trace kernel's work goes into the warp segments that run past
bounce_limit (paths kept alive by mirror hits), and what moving those paths into a dense second kernel could save.

Replays the oracle's exact per-path traversal traces (tools/sched_sim.py:get_traces: maze 32, 1920x1080, 16 spp, 8 bounces,
every EVERY-th 4x4-chunk group), forms warps the way trace_kernel does (32 consecutive virtual threads = two pixels x 16
samples) and prices every warp segment with the per-body costs of tools/sched_sim_r2.py (59 warp instructions per interior
visit, 80 per rect test, 8 per vote, 330 + 40 per shaded segment and set-up).

Trigger K: at a segment boundary past bounce_limit, a warp with 1..K live lanes writes those paths to a queue and stops.  The
tail kernel then runs the queued paths 32 to a warp in queue order.  Saving = the warp segments removed from the trace kernel
- the same paths' segments in the tail kernel - the spill / reload / deferred-pixel traffic (priced as SPILL per spilling
warp, RELOAD per tail warp, PIXEL per deferred pixel, in warp instructions).

    python tools/tail_replay.py [EVERY]          (default 797, about 41k paths; the output is committed under profiles/)
"""
import os
import sys
from collections import Counter

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sched_sim                                        # noqa: E402
from sched_sim_r2 import C_S, seg_cost                  # noqa: E402

BOUNCES, SPP = 8, 16
SEG_FIXED = C_S + 40            # shade + next segment's set-up, as sched_sim_r2's model of the shipped kernel
SPILL, RELOAD, PIXEL = 120.0, 120.0, 60.0


def warp_rounds(w):
    """Per segment round of one warp: (live lanes, warp instructions)."""
    out = []
    for s in range(max(len(p) for p in w)):
        live = [p[s] for p in w if len(p) > s]
        out.append((len(live), seg_cost(live)[0] + SEG_FIXED))
    return out


def main():
    every = int(sys.argv[1]) if len(sys.argv) > 1 else 797
    paths, _ = sched_sim.get_traces(maze=32, spp=SPP, bounces=BOUNCES, every=every)
    warps = [paths[i:i + 32] for i in range(0, len(paths), 32)]
    rounds = [warp_rounds(w) for w in warps]
    total = sum(c for r in rounds for _, c in r)
    rays = sum(len(p) for p in paths)
    tail_rounds = [(n, c) for r in rounds for n, c in r[BOUNCES:]]
    tail_cost = sum(c for _, c in tail_rounds)
    warps_with_tail = sum(1 for r in rounds if len(r) > BOUNCES)
    print(f"{len(paths)} paths, {rays} rays ({rays / len(paths):.4f} segments per path), {len(warps)} warps; "
          f"paths with a segment past bounce_limit {BOUNCES}: {sum(1 for p in paths if len(p) > BOUNCES) / len(paths):.2%}")
    print(f"warps that run past bounce_limit: {warps_with_tail / len(warps):.2%}; "
          f"warp segments past bounce_limit per warp: {len(tail_rounds) / len(warps):.3f}")
    hist = Counter(n for n, _ in tail_rounds)
    print("live lanes in a warp segment past bounce_limit: " + ", ".join(f"{k}:{hist[k]}" for k in sorted(hist)))
    print(f"modelled warp instructions: {total / rays:.1f} per ray; share in segments past bounce_limit: {tail_cost / total:.2%} "
          f"(their lane-segments are {sum(n for n, _ in tail_rounds) / rays:.2%} of the rays)")
    print(f"{'K':>3} {'spilled paths':>14} {'removed':>9} {'tail kernel':>12} {'overhead':>9} {'saving':>8}")
    for K in range(1, 17):
        removed, queue, n_spill, n_pix = 0.0, [], 0, 0
        for w, r in zip(warps, rounds):
            for s in range(BOUNCES, len(r)):
                if r[s][0] <= K:
                    removed += sum(c for _, c in r[s:])
                    live = [i for i, p in enumerate(w) if len(p) > s]
                    queue.extend(w[i][s:] for i in live)
                    n_spill += 1
                    n_pix += len({i // SPP for i in live})
                    break
        tail = 0.0
        for q0 in range(0, len(queue), 32):
            tail += sum(c for _, c in warp_rounds(queue[q0:q0 + 32])) + RELOAD
        over = n_spill * SPILL + n_pix * PIXEL
        print(f"{K:3d} {len(queue):14d} {removed / total:9.2%} {tail / total:12.2%} {over / total:9.2%} {(removed - tail - over) / total:8.2%}")


if __name__ == "__main__":
    main()
