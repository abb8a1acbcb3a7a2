//! `extern "C"` bindings of include/mirror_maze_cuda.h (subset used by the headless driver).
//! NOT compiled in this environment.  Layouts: reference src/main.rs:32-90, src/maths.rs:3-16,50-52.
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int};

#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Float2(pub f32, pub f32);
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Float3(pub f32, pub f32, pub f32);
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Float4(pub f32, pub f32, pub f32, pub f32);
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Plane { pub origin: Float3, pub v: Float3, pub u: Float3, pub color: Float3 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct BVHNode { pub aabb_min: Float3, pub aabb_max: Float3, pub left_first: u32, pub tri_count: u32 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Camera { pub camera_center: Float3, pub focal_length: f32, pub rotation: Float4, pub viewport: Float2 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Uniform { pub cam: Camera, pub view_width: f32, pub view_height: f32, pub chunk_width: u32, pub time: u32 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct Chunk { pub x: u32, pub y: u32 }
/// `spp`: a power of two in 1..=1024 (`chunk_width^2 * spp <= 2^20`); `chunk_width = 1, spp = 1024` is the reference's
/// one-pixel-per-threadgroup dispatch.  Anything else returns `MM_ERR_UNSUPPORTED`.
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct Params { pub spp: u32, pub bounce_limit: u32, pub mirror_limit: u32, pub grid_x: u32, pub grid_y: u32,
                    pub group_first: u32, pub group_step: u32, pub group_count: u32, pub flags: u32 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)]
pub struct Counters { pub paths: u64, pub rays: u64, pub inner_visits: u64, pub leaf_visits: u64, pub rect_tests: u64,
                      pub hits: u64, pub literal_rays: u64, pub max_stack: u64 }

const _: () = assert!(std::mem::size_of::<Plane>() == 48 && std::mem::size_of::<BVHNode>() == 32
    && std::mem::size_of::<Camera>() == 40 && std::mem::size_of::<Uniform>() == 56 && std::mem::size_of::<Params>() == 36);

#[repr(C)] pub struct mm_ctx { _p: [u8; 0] }
#[repr(C)] pub struct mm_multi { _p: [u8; 0] }
#[repr(C)] pub struct mm_scene { _p: [u8; 0] }
pub const MM_EXCHANGE_PEER: c_int = 0;
pub const MM_EXCHANGE_NCCL: c_int = 1;
pub const MM_EXCHANGE_NONE: c_int = 2;
pub const MM_MAX_VIEWS: u32 = 64;

extern "C" {
    pub fn mm_create(cuda_device: c_int, out: *mut *mut mm_ctx) -> c_int;
    pub fn mm_destroy(ctx: *mut mm_ctx) -> c_int;
    pub fn mm_last_error(ctx: *const mm_ctx) -> *const c_char;
    pub fn mm_upload_scene(ctx: *mut mm_ctx, planes: *const Plane, n_planes: u32, nodes: *const BVHNode, n_nodes: u32,
                           indices: *const u32, materials: *const u8, emissions: *const Float4,
                           noise_rgba8: *const u8, noise_w: u32, noise_h: u32) -> c_int;
    pub fn mm_render(ctx: *mut mm_ctx, uni: *const Uniform, params: *const Params, chunks: *const Chunk, n_chunks: u32,
                     out_rgba: *mut f32, counters: *mut Counters, debug: *const std::ffi::c_void) -> c_int;
    // commit() without wait (main.rs:894) / the wait the reference never needs because it presents a drawable
    pub fn mm_render_async(ctx: *mut mm_ctx, uni: *const Uniform, params: *const Params, chunks: *const Chunk, n_chunks: u32,
                           out_rgba: *mut f32, debug: *const std::ffi::c_void) -> c_int;
    pub fn mm_wait(ctx: *mut mm_ctx, counters: *mut Counters) -> c_int;
    // several camera views in one launch, each with its own uniform, chunk list and persistent view screen (MM_MAX_VIEWS = 64)
    pub fn mm_render_views_async(ctx: *mut mm_ctx, unis: *const Uniform, n_views: u32, params: *const Params, chunks: *const Chunk,
                                 n_chunks: u32, out_rgba: *const *mut f32, debug: *const std::ffi::c_void) -> c_int;
    pub fn mm_render_views(ctx: *mut mm_ctx, unis: *const Uniform, n_views: u32, params: *const Params, chunks: *const Chunk,
                           n_chunks: u32, out_rgba: *const *mut f32, counters: *mut Counters, debug: *const std::ffi::c_void) -> c_int;
    // the blur of every view screen in one launch; out: null or one pinned pointer (or null) per view, done at mm_wait_present
    pub fn mm_present_views(ctx: *mut mm_ctx, rgba8: u32, out: *const *mut std::ffi::c_void) -> c_int;
    // pin + map a Vec<f32> frame once: the kernel then stores finished pixels straight into it (zero-copy output)
    pub fn mm_host_register(ptr: *mut std::ffi::c_void, bytes: usize) -> c_int;
    pub fn mm_host_unregister(ptr: *mut std::ffi::c_void) -> c_int;
    // one process, several GPUs
    pub fn mm_multi_create(devices: *const c_int, n: c_int, exchange: c_int, out: *mut *mut mm_multi) -> c_int;
    pub fn mm_multi_destroy(m: *mut mm_multi) -> c_int;
    pub fn mm_multi_last_error(m: *const mm_multi) -> *const c_char;
    pub fn mm_multi_upload_scene(m: *mut mm_multi, planes: *const Plane, n_planes: u32, nodes: *const BVHNode, n_nodes: u32,
                                 indices: *const u32, materials: *const u8, emissions: *const Float4,
                                 noise_rgba8: *const u8, noise_w: u32, noise_h: u32) -> c_int;
    pub fn mm_multi_render(m: *mut mm_multi, uni: *const Uniform, params: *const Params, chunks: *const Chunk, n_chunks: u32,
                           out_rgba: *mut f32, counters: *mut Counters) -> c_int;
    pub fn mm_multi_last_ms(m: *mut mm_multi, ms: *mut f32) -> c_int;
    pub fn mm_present(ctx: *mut mm_ctx, out_rgba: *mut f32) -> c_int;
    // present_drawable + commit without wait (main.rs:893-894): blur now, read-back on a second stream
    pub fn mm_present_async(ctx: *mut mm_ctx, out_rgba_pinned: *mut f32) -> c_int;
    pub fn mm_present_async_rgba8(ctx: *mut mm_ctx, out_rgba8_pinned: *mut u8) -> c_int;
    pub fn mm_wait_present(ctx: *mut mm_ctx) -> c_int;
    pub fn mm_host_alloc(bytes: usize, out: *mut *mut std::ffi::c_void) -> c_int;
    pub fn mm_host_free(ptr: *mut std::ffi::c_void) -> c_int;
    pub fn mm_last_ms(ctx: *mut mm_ctx, ms: *mut f32) -> c_int;
    pub fn mm_scene_build(maze_n: u32, seed: u64, fast_bvh: c_int, out: *mut *mut mm_scene) -> c_int;
    pub fn mm_scene_free(s: *mut mm_scene) -> c_int;
    pub fn mm_scene_n_planes(s: *const mm_scene) -> u32;
    pub fn mm_scene_n_nodes(s: *const mm_scene) -> u32;
    pub fn mm_scene_planes(s: *const mm_scene) -> *const Plane;
    pub fn mm_scene_nodes(s: *const mm_scene) -> *const BVHNode;
    pub fn mm_scene_indices(s: *const mm_scene) -> *const u32;
    pub fn mm_scene_materials(s: *const mm_scene) -> *const u8;
    pub fn mm_scene_emissions(s: *const mm_scene) -> *const Float4;
    pub fn mm_gen_chunks(view_width: f32, view_height: f32, chunk_width: u32, out: *mut Chunk, cap: u32) -> u32;
    pub fn mm_default_uniform(maze_n: u32, view_width: f32, view_height: f32, chunk_width: u32, time: u32, out: *mut Uniform) -> c_int;
}
