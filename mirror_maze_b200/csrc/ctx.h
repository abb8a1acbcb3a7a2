// ctx.h — the context behind include/mirror_maze_cuda.h's opaque mm_ctx, shared by api.cu (one device) and multi.cu
// (a device list in one process).  Private to the library.
#pragma once
#include <string>
#include "render_kernel.cuh"

struct mm_ctx {
    int device = -1;
    cudaStream_t stream = nullptr;       // stream in use
    cudaStream_t own_stream = nullptr;   // created by mm_create
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;   // kernel start, kernel end, counter copy done
    bool timed = false;
    std::string err;
    int n_sms = 0;
    size_t smem_optin = 0;
    // scene
    bool have_scene = false;
    mmk::PairRec *d_pairs = nullptr;
    mmk::PairRecY *d_pairs_y = nullptr;   // n_pairs_y y-table records followed by n_yiv y-intervals; present when n_yiv > 0
    uint32_t n_pairs_y = 0, n_yiv = 0;
    mmk::RectI *d_rects = nullptr;
    mmk::RectS *d_shade = nullptr;
    mmk::RectA *d_rects_axis = nullptr;   // present when every rect is axis-aligned
    uint8_t *d_noise = nullptr;
    uint32_t n_pairs = 0, n_slots = 0, n_nodes = 0, root_link = 0, root_count = 0, depth = 0, max_leaf = 0, noise_w = 0, noise_h = 0;
    bool fast_ok = false, rect_fast_ok = false;
    // per-frame
    mm_chunk *d_chunks = nullptr;
    uint32_t chunks_cap = 0, n_chunks = 0;
    mmk::Counters *d_counters = nullptr;
    mmk::Counters *h_counters = nullptr;   // pinned
    float *d_screen = nullptr;        // persistent screen image (the reference's private screen texture, main.rs:702-709)
    float *d_screen2 = nullptr;       // ping-pong partner for the present blur
    uint8_t *d_screen8 = nullptr;     // RGBA8Unorm copy of the screen (mm_present_rgba8)
    uint32_t screen_w = 0, screen_h = 0;
    uint32_t *d_dbg_u32[3] = {nullptr, nullptr, nullptr};
    float *d_dbg_rad = nullptr;
    size_t dbg_cap = 0;
    mmk::TailPath *d_tail_q = nullptr;  // straggler queue and deferred-pixel slots (trace_kernel -> trace_tail_kernel)
    float *d_tail_pix = nullptr;
    size_t tail_q_cap = 0, tail_pix_bytes = 0;
    // asynchronous host-buffer frames (mm_render_async / mm_wait)
    float *h_stage = nullptr;         // pinned staging for callers whose buffer the library does not know to be pinned
    size_t stage_bytes = 0;
    float *pending_out = nullptr;     // caller buffer that receives h_stage at mm_wait
    size_t pending_bytes = 0;
    bool in_flight = false;
    uint32_t last_zero_copy = 0;
    // asynchronous present (mm_present_async): the blurred screen is snapshot on the main stream and read back on a second one
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_snap = nullptr, ev_copy = nullptr;
    float *d_snap = nullptr;
    bool present_in_flight = false;
    // last launch facts
    uint32_t last_smem = 0, last_blocks_per_sm = 0, last_block_threads = 0, last_tail_cap = 0;
    uint32_t last_y_table = 0;        // y-table entries of the last launch, 0 when it ran without the table
    const void *cfg_fn = nullptr;     // kernel variant whose attributes / occupancy were last set up
    size_t cfg_smem = 0;
};

namespace mmapi {

struct Launch {
    mmk::KParams p;
    mmk::KernelChoice choice;
    unsigned blocks;
    size_t smem;
};

int fail(mm_ctx *ctx, int code, const std::string &msg);
bool traversal_params(const mm_ctx *ctx, uint32_t flags, mmk::KParams &p);
int build_launch(mm_ctx *ctx, const mm_uniform *uni, const mm_params *par, bool debug, Launch &L);
int do_launch(mm_ctx *ctx, Launch &L);
int ensure_screen(mm_ctx *ctx, uint32_t W, uint32_t H);
void counters_out(const mmk::Counters *h, mm_counters *o);
// Device alias of [p, p + bytes) when the range lies inside mapped pinned memory the library allocated or registered
// (mm_host_alloc / mm_host_register); nullptr otherwise.
void *host_device_alias(const void *p, size_t bytes);

}  // namespace mmapi

#define MM_CK(call)                                                                                       \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) {                                                                         \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                               \
            return MM_ERR_CUDA;                                                                           \
        }                                                                                                 \
    } while (0)
