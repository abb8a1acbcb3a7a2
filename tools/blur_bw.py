"""Developer tool (GPU box): achieved HBM bandwidth of the present pass' 5-tap blur (blur_kernel; reference src/shaders.metal:214-225),
the one HBM-bound kernel on the path: 16 B read + 16 B written per pixel (the four neighbour taps hit L1 / L2)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import mirror_maze_b200 as mm

r = mm.Renderer(0)
peaks_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
peak = json.load(open(peaks_path)).get("hbm_gbs", 6650.0) if os.path.exists(peaks_path) else 6650.0   # the file is written per machine, not committed
stream = torch.cuda.Stream()
r.set_stream(stream.cuda_stream)
for W, H in ((1920, 1080), (3840, 2160), (7680, 4320)):
    a = torch.rand((H, W, 4), device="cuda"); b = torch.empty_like(a)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(stream):
        for _ in range(3):
            r.present_blur_device(a.data_ptr(), b.data_ptr(), W, H)
        ms = []
        for i in range(10):
            flush.fill_(i)                                   # L2 flush between timed launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r.present_blur_device(a.data_ptr(), b.data_ptr(), W, H); e1.record(); e1.synchronize()
            ms.append(e0.elapsed_time(e1))
    best = sorted(ms)[len(ms) // 2]
    gbs = 2 * W * H * 16 / (best * 1e-3) / 1e9
    print(json.dumps({"kernel": "blur_kernel", "frame": f"{W}x{H}", "ms_median": round(best, 4), "algorithmic_GBs": round(gbs, 1),
                      "hbm_peak_measured_GBs": peak, "frac": round(gbs / peak, 3)}))
