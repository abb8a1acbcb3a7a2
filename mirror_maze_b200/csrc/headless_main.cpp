// headless_main.cpp — headless driver over the C-ABI, the C++ stand-in for the Rust driver north_star asks for (no Rust
// toolchain on the build or GPU boxes).  It walks the same steps as the reference's main() (reference src/main.rs:356-895)
// with the window, event loop and Metal calls removed:
//   maze + walls + scene + BVH (:357-588)  ->  mm_scene_build
//   device, queue, pipelines, buffers, noise texture (:616-730)  ->  mm_create + mm_upload_scene
//   uniform (:732-755, 846-858), chunk list (:713-723, 778-784), dispatch (:867-886)  ->  mm_render
//   present pass (:888-893)  ->  mm_present (optional)
// and writes the frame as a binary PPM (sqrt tone-map already applied by the kernel, as in the shader) or raw fp32.
//
//   mm_headless [--maze N] [--width W] [--height H] [--spp S] [--chunk C] [--bounces B] [--frames F] [--blur]
//               [--noise file.rgba8] [--out frame.ppm] [--raw frame.f32] [--gpus N] [--exchange peer|nccl|none] [--pageable]
// --chunk C is the uniform's chunk_width (default 4, the reference's): each virtual threadgroup renders a C x C chunk, so
// --chunk 1 --spp 1024 is the reference's one-pixel-per-threadgroup shape (1024 / C^2 samples fill its 32 x 32 threads).
// --gpus N > 1 renders through mm_multi (one process, N devices: the frame's groups interleaved over the devices).  The
// frame buffer is mapped pinned memory from mm_host_alloc (zero-copy output) unless --pageable asks for a plain vector.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/mirror_maze_cuda.h"

static int fail(mm_ctx *ctx, const char *what, int rc) {
    std::fprintf(stderr, "%s failed: %d (%s)\n", what, rc, mm_last_error(ctx));
    return 1;
}

int main(int argc, char **argv) {
    uint32_t maze = 10, W = 1024, H = 768, spp = 64, chunk = 4, bounces = 5, frames = 1;   // the reference's literals
    int gpus = 1, exchange = MM_EXCHANGE_PEER;
    bool blur = false, pageable = false;
    std::string out_ppm, out_raw, noise_file;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto next = [&]() -> const char * { return i + 1 < argc ? argv[++i] : ""; };
        if (a == "--maze") maze = (uint32_t)std::atoi(next());
        else if (a == "--width") W = (uint32_t)std::atoi(next());
        else if (a == "--height") H = (uint32_t)std::atoi(next());
        else if (a == "--spp") spp = (uint32_t)std::atoi(next());
        else if (a == "--chunk") chunk = (uint32_t)std::atoi(next());
        else if (a == "--bounces") bounces = (uint32_t)std::atoi(next());
        else if (a == "--frames") frames = (uint32_t)std::atoi(next());
        else if (a == "--blur") blur = true;
        else if (a == "--pageable") pageable = true;
        else if (a == "--gpus") gpus = std::atoi(next());
        else if (a == "--exchange") {
            std::string e = next();
            exchange = e == "nccl" ? MM_EXCHANGE_NCCL : (e == "none" ? MM_EXCHANGE_NONE : MM_EXCHANGE_PEER);
        }
        else if (a == "--out") out_ppm = next();
        else if (a == "--raw") out_raw = next();
        else if (a == "--noise") noise_file = next();
        else { std::fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    // noise texture: raw 512x512 RGBA8 if given, else a flat 128 texture (only texel (0,0) is ever sampled: the shader
    // samples with integer coordinates, normalised + repeat + nearest, shaders.metal:288-291)
    std::vector<uint8_t> noise(512 * 512 * 4, 128);
    for (size_t i = 3; i < noise.size(); i += 4) noise[i] = 255;
    if (!noise_file.empty()) {
        FILE *f = std::fopen(noise_file.c_str(), "rb");
        if (!f || std::fread(noise.data(), 1, noise.size(), f) != noise.size()) { std::fprintf(stderr, "cannot read %s\n", noise_file.c_str()); return 2; }
        std::fclose(f);
    }

    mm_scene *scene = nullptr;
    int rc = mm_scene_build(maze, 0, 1, &scene);
    if (rc != MM_OK) { std::fprintf(stderr, "mm_scene_build failed: %d\n", rc); return 1; }
    mm_ctx *ctx = nullptr;
    mm_multi *multi = nullptr;
    if (gpus > 1) {
        if (blur) { std::fprintf(stderr, "--blur needs --gpus 1 (the present pass runs on one device's screen)\n"); return 2; }
        std::vector<int> devs(gpus);
        for (int i = 0; i < gpus; i++) devs[i] = i;
        rc = mm_multi_create(devs.data(), gpus, exchange, &multi);
        if (rc != MM_OK) { std::fprintf(stderr, "mm_multi_create failed: %d (%s)\n", rc, mm_multi_last_error(nullptr)); return 1; }
        rc = mm_multi_upload_scene(multi, mm_scene_planes(scene), mm_scene_n_planes(scene), mm_scene_nodes(scene), mm_scene_n_nodes(scene),
                                   mm_scene_indices(scene), mm_scene_materials(scene), mm_scene_emissions(scene), noise.data(), 512, 512);
        if (rc != MM_OK) { std::fprintf(stderr, "mm_multi_upload_scene failed: %d (%s)\n", rc, mm_multi_last_error(multi)); return 1; }
    } else {
        rc = mm_create(0, &ctx);
        if (rc != MM_OK) { std::fprintf(stderr, "mm_create failed: %d (%s)\n", rc, mm_last_error(nullptr)); return 1; }   // no CPU fallback
        rc = mm_upload_scene(ctx, mm_scene_planes(scene), mm_scene_n_planes(scene), mm_scene_nodes(scene), mm_scene_n_nodes(scene),
                             mm_scene_indices(scene), mm_scene_materials(scene), mm_scene_emissions(scene), noise.data(), 512, 512);
        if (rc != MM_OK) return fail(ctx, "mm_upload_scene", rc);
    }

    mm_uniform uni;
    if (chunk == 0 || chunk > W || chunk > H) { std::fprintf(stderr, "--chunk must be in 1..min(width, height)\n"); return 2; }
    rc = mm_default_uniform(maze, (float)W, (float)H, chunk, 0, &uni);
    if (rc != MM_OK) { std::fprintf(stderr, "mm_default_uniform failed: %d\n", rc); return 1; }
    const uint32_t n_chunks = mm_gen_chunks((float)W, (float)H, chunk, nullptr, 0);
    std::vector<mm_chunk> chunks(n_chunks);
    mm_gen_chunks((float)W, (float)H, chunk, chunks.data(), n_chunks);
    mm_params par;
    std::memset(&par, 0, sizeof(par));
    par.spp = spp; par.bounce_limit = bounces; par.mirror_limit = 15;
    par.grid_x = W / chunk; par.grid_y = H / chunk;         // one virtual threadgroup per chunk, whole frame

    const size_t frame_floats = (size_t)W * H * 4;
    std::vector<float> frame_vec;
    float *frame = nullptr;
    if (pageable) {
        frame_vec.assign(frame_floats, 0.0f);
        frame = frame_vec.data();
    } else {
        void *p = nullptr;
        rc = mm_host_alloc(frame_floats * sizeof(float), &p);
        if (rc != MM_OK) { std::fprintf(stderr, "mm_host_alloc failed: %d\n", rc); return 1; }
        frame = static_cast<float *>(p);
        std::memset(frame, 0, frame_floats * sizeof(float));
    }
    mm_counters cnt;
    double total_ms = 0.0, total_rays = 0.0;
    for (uint32_t f = 0; f < frames; f++) {
        uni.time = f;                                        // main.rs:857
        auto t0 = std::chrono::steady_clock::now();
        // the chunk list goes to the device with the first frame; later frames keep it (it does not change here)
        const mm_chunk *cl = f == 0 ? chunks.data() : nullptr;
        if (multi) {
            rc = mm_multi_render(multi, &uni, &par, cl, n_chunks, frame, &cnt);
            if (rc != MM_OK) { std::fprintf(stderr, "mm_multi_render failed: %d (%s)\n", rc, mm_multi_last_error(multi)); return 1; }
        } else {
            rc = mm_render(ctx, &uni, &par, cl, n_chunks, frame, &cnt, nullptr);
            if (rc != MM_OK) return fail(ctx, "mm_render", rc);
        }
        if (blur) {
            rc = mm_present(ctx, frame);
            if (rc != MM_OK) return fail(ctx, "mm_present", rc);
        }
        total_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        total_rays += (double)cnt.rays;
    }
    float kernel_ms = 0.0f;
    if (multi) mm_multi_last_ms(multi, &kernel_ms); else mm_last_ms(ctx, &kernel_ms);
    std::printf("%d GPU(s)%s; ", gpus, multi ? (exchange == MM_EXCHANGE_NCCL ? " [nccl gather]" : exchange == MM_EXCHANGE_NONE ? " [host assembly]" : " [peer stores]") : "");
    std::printf("maze %ux%u: %u planes, %u nodes; %ux%u x%u spp, chunk %u, %u bounces; %u frame(s): %.3f ms/frame end to end (last kernel %.3f ms), "
                "%.1f Mrays/s, %llu rays/frame\n", maze, maze, mm_scene_n_planes(scene), mm_scene_n_nodes(scene), W, H, spp, chunk, bounces, frames,
                total_ms / frames, kernel_ms, total_rays / total_ms / 1e3, (unsigned long long)cnt.rays);

    if (!out_raw.empty()) {
        FILE *f = std::fopen(out_raw.c_str(), "wb");
        if (!f) { std::fprintf(stderr, "cannot write %s\n", out_raw.c_str()); return 2; }
        std::fwrite(frame, sizeof(float), frame_floats, f);
        std::fclose(f);
    }
    if (!out_ppm.empty()) {
        FILE *f = std::fopen(out_ppm.c_str(), "wb");
        if (!f) { std::fprintf(stderr, "cannot write %s\n", out_ppm.c_str()); return 2; }
        std::fprintf(f, "P6\n%u %u\n255\n", W, H);
        std::vector<uint8_t> row(W * 3);
        for (uint32_t y = 0; y < H; y++) {
            for (uint32_t x = 0; x < W; x++)
                for (int c = 0; c < 3; c++) {                // RGBA8Unorm store of the reference's texture (main.rs:704)
                    float v = frame[((size_t)y * W + x) * 4 + c];
                    v = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
                    row[x * 3 + c] = (uint8_t)std::lround(v * 255.0f);
                }
            std::fwrite(row.data(), 1, row.size(), f);
        }
        std::fclose(f);
    }
    if (!pageable) mm_host_free(frame);
    mm_multi_destroy(multi);
    mm_destroy(ctx);
    mm_scene_free(scene);
    return 0;
}
