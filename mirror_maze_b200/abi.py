"""ctypes binding of include/mirror_maze_cuda.h (the C-ABI drop-in boundary).

Struct layouts are the reference's #[repr(C)] types (reference src/main.rs:32-90, src/maths.rs:3-16,50-52); sizes
are asserted at import.  The library is built in-tree by `make -C mirror_maze_b200` (see __graft_entry__.build).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libmirror_maze_cuda.so"

MAX_STACK = 52
MAX_BVH_DEPTH = 51
FLAG_COUNTERS = 1
FLAG_FORCE_LITERAL = 2
FLAG_RCP_SLAB = 64
FLAG_NO_ZERO_COPY = 128
FLAG_POOL_KERNEL = 256
FLAG_SCREEN_RGBA8 = 512
FLAG_REGROUP = 1024
FLAG_GENERAL_RECTS = 2048
FLAG_NO_TAIL = 4096
FLAG_NO_Y_TABLE = 8192
EXCHANGE_PEER, EXCHANGE_NCCL, EXCHANGE_NONE = 0, 1, 2
MAX_PEERS = 8
MAX_VIEWS = 64

ERR_NAMES = {0: "MM_OK", -1: "MM_ERR_INVALID", -2: "MM_ERR_CUDA", -3: "MM_ERR_NO_SCENE", -4: "MM_ERR_BVH",
             -5: "MM_ERR_UNSUPPORTED", -6: "MM_ERR_NOMEM"}


class MMError(RuntimeError):
    """A C-ABI call returned a negative MM_ERR_* code (the reference panics instead, e.g. src/utils.rs:19)."""

    def __init__(self, code, msg=""):
        self.code = code
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}" if msg else str(ERR_NAMES.get(code, code)))


class Float2(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float)]


class Float3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class Float4(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float), ("w", C.c_float)]


class Plane(C.Structure):          # main.rs:51-58
    _fields_ = [("origin", Float3), ("v", Float3), ("u", Float3), ("color", Float3)]


class BVHNode(C.Structure):        # main.rs:74-81
    _fields_ = [("aabb_min", Float3), ("aabb_max", Float3), ("left_first", C.c_uint32), ("tri_count", C.c_uint32)]


class Camera(C.Structure):         # main.rs:32-39
    _fields_ = [("camera_center", Float3), ("focal_length", C.c_float), ("rotation", Float4), ("viewport", Float2)]


class Uniform(C.Structure):        # main.rs:41-49
    _fields_ = [("cam", Camera), ("view_width", C.c_float), ("view_height", C.c_float), ("chunk_width", C.c_uint32),
                ("time", C.c_uint32)]


class Chunk(C.Structure):
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32)]


class Params(C.Structure):
    _fields_ = [("spp", C.c_uint32), ("bounce_limit", C.c_uint32), ("mirror_limit", C.c_uint32), ("grid_x", C.c_uint32),
                ("grid_y", C.c_uint32), ("group_first", C.c_uint32), ("group_step", C.c_uint32), ("group_count", C.c_uint32),
                ("flags", C.c_uint32)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits",
                                          "literal_rays", "max_stack")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class Debug(C.Structure):
    _fields_ = [("first_hit", C.POINTER(C.c_uint32)), ("segments", C.POINTER(C.c_uint32)),
                ("mirror_hits", C.POINTER(C.c_uint32)), ("radiance", C.POINTER(C.c_float))]


class SceneInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("n_planes", "n_nodes", "bvh_depth", "max_leaf", "fast_rect_ok", "fast_slab_ok",
                                          "smem_bytes", "block_threads", "blocks_per_sm", "n_sms", "axis_rects",
                                          "y_table")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


assert C.sizeof(Float2) == 8 and C.sizeof(Float3) == 12 and C.sizeof(Float4) == 16
assert C.sizeof(Plane) == 48 and C.sizeof(BVHNode) == 32 and C.sizeof(Camera) == 40 and C.sizeof(Uniform) == 56
assert C.sizeof(Chunk) == 8 and C.sizeof(Params) == 36 and C.sizeof(Counters) == 64

_P = C.POINTER
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/mirror_maze_cuda.h declares.
PROTOTYPES = {
    "mm_create": (C.c_int, [C.c_int, _P(_vp)]),
    "mm_destroy": (C.c_int, [_vp]),
    "mm_last_error": (C.c_char_p, [_vp]),
    "mm_upload_scene": (C.c_int, [_vp, _vp, C.c_uint32, _vp, C.c_uint32, _vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32]),
    "mm_render": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, C.c_uint32, _vp, _P(Counters), _P(Debug)]),
    "mm_render_async": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, C.c_uint32, _vp, _P(Debug)]),
    "mm_wait": (C.c_int, [_vp, _P(Counters)]),
    "mm_render_views_async": (C.c_int, [_vp, _P(Uniform), C.c_uint32, _P(Params), _vp, C.c_uint32, _P(_vp), _P(Debug)]),
    "mm_render_views": (C.c_int, [_vp, _P(Uniform), C.c_uint32, _P(Params), _vp, C.c_uint32, _P(_vp), _P(Counters), _P(Debug)]),
    "mm_present_views": (C.c_int, [_vp, C.c_uint32, _P(_vp)]),
    "mm_host_alloc": (C.c_int, [C.c_size_t, _P(_vp)]),
    "mm_host_free": (C.c_int, [_vp]),
    "mm_host_register": (C.c_int, [_vp, C.c_size_t]),
    "mm_host_unregister": (C.c_int, [_vp]),
    "mm_render_multicast_device": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp]),
    "mm_multi_create": (C.c_int, [_P(C.c_int), C.c_int, C.c_int, _P(_vp)]),
    "mm_multi_destroy": (C.c_int, [_vp]),
    "mm_multi_last_error": (C.c_char_p, [_vp]),
    "mm_multi_n_devices": (C.c_int, [_vp]),
    "mm_multi_upload_scene": (C.c_int, [_vp, _vp, C.c_uint32, _vp, C.c_uint32, _vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32]),
    "mm_multi_render": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, C.c_uint32, _vp, _P(Counters)]),
    "mm_multi_render_async": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, C.c_uint32, _vp]),
    "mm_multi_wait": (C.c_int, [_vp, _P(Counters)]),
    "mm_multi_frame_device": (C.c_int, [_vp, C.c_int, _P(_vp)]),
    "mm_multi_last_ms": (C.c_int, [_vp, _P(C.c_float)]),
    "mm_multi_ctx": (_vp, [_vp, C.c_int]),
    "mm_set_chunks": (C.c_int, [_vp, _vp, C.c_uint32]),
    "mm_render_device": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, _vp]),
    "mm_scatter_tiles_device": (C.c_int, [_vp, _P(Uniform), _P(Params), _vp, _vp]),
    "mm_scatter_gathered_device": (C.c_int, [_vp, _P(Uniform), _P(Params), C.c_uint32, C.c_uint32, _vp, _vp]),
    "mm_sync": (C.c_int, [_vp]),
    "mm_set_stream": (C.c_int, [_vp, _vp]),
    "mm_last_counters": (C.c_int, [_vp, _P(Counters)]),
    "mm_last_ms": (C.c_int, [_vp, _P(C.c_float)]),
    "mm_last_tail": (C.c_int, [_vp, _P(C.c_uint64), _P(C.c_uint64)]),
    "mm_stream": (C.c_int, [_vp, _P(_vp)]),
    "mm_get_scene_info": (C.c_int, [_vp, _P(SceneInfo)]),
    "mm_selftest_quotient": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _P(C.c_uint64)]),
    "mm_selftest_div3": (C.c_int, [_vp, _P(C.c_uint64)]),
    "mm_render_peers_device": (C.c_int, [_vp, _P(Uniform), _P(Params), _P(C.c_void_p), C.c_uint32]),
    "mm_rect_edge_thresholds": (C.c_int, [C.c_float, _P(C.c_float), _P(C.c_float)]),
    "mm_axis_rect": (C.c_int, [_P(Plane), _P(C.c_float), _P(C.c_uint32)]),
    "mm_trace_rays": (C.c_int, [_vp, C.c_uint32, _vp, _vp, C.c_uint32, _vp, _vp, _vp]),
    "mm_microbench": (C.c_int, [_vp, C.c_int, C.c_uint64, _P(C.c_double)]),
    "mm_present": (C.c_int, [_vp, _vp]),
    "mm_present_rgba8": (C.c_int, [_vp, _vp, _vp]),
    "mm_present_async": (C.c_int, [_vp, _vp]),
    "mm_present_async_rgba8": (C.c_int, [_vp, _vp]),
    "mm_wait_present": (C.c_int, [_vp]),
    "mm_present_blur_device": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint32]),
    "mm_move_camera": (C.c_int, [_vp, C.c_uint32, Float3, Float4, _vp, C.c_uint32, C.c_float, _P(Float3)]),
    "mm_bag_new": (C.c_int, [C.c_float, C.c_float, C.c_uint32, C.c_uint64, _P(_vp)]),
    "mm_bag_free": (C.c_int, [_vp]),
    "mm_bag_next": (C.c_int, [_vp, C.c_uint32, _vp]),
    "mm_bag_reshuffle": (C.c_int, [_vp]),
    "mm_bag_size": (C.c_uint32, [_vp]),
    "mm_scene_build": (C.c_int, [C.c_uint32, C.c_uint64, C.c_int, _P(_vp)]),
    "mm_scene_free": (C.c_int, [_vp]),
    "mm_scene_n_planes": (C.c_uint32, [_vp]),
    "mm_scene_n_nodes": (C.c_uint32, [_vp]),
    "mm_scene_planes": (_vp, [_vp]),
    "mm_scene_nodes": (_vp, [_vp]),
    "mm_scene_indices": (_vp, [_vp]),
    "mm_scene_materials": (_vp, [_vp]),
    "mm_scene_emissions": (_vp, [_vp]),
    "mm_scene_grid": (_vp, [_vp]),
    "mm_scene_n_vert_walls": (C.c_uint32, [_vp]),
    "mm_scene_n_hori_walls": (C.c_uint32, [_vp]),
    "mm_scene_vert_walls": (_vp, [_vp]),
    "mm_scene_hori_walls": (_vp, [_vp]),
    "mm_build_bvh": (C.c_int, [_vp, C.c_uint32, C.c_int, _vp, _P(C.c_uint32), _vp]),
    "mm_stdrng_new": (C.c_int, [C.c_uint64, _P(_vp)]),
    "mm_stdrng_free": (C.c_int, [_vp]),
    "mm_stdrng_next_u32": (C.c_uint32, [_vp]),
    "mm_stdrng_gen_f32": (C.c_float, [_vp]),
    "mm_stdrng_gen_range_u32": (C.c_uint32, [_vp, C.c_uint32, C.c_uint32]),
    "mm_chacha_block": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_int, _vp]),
    "mm_calculate_quaternion": (Float4, [Float3]),
    "mm_update_quat_angle": (Float4, [Float4, C.c_float]),
    "mm_quat_mult": (Float3, [Float3, Float4]),
    "mm_gen_chunks": (C.c_uint32, [C.c_float, C.c_float, C.c_uint32, _vp, C.c_uint32]),
    "mm_default_uniform": (C.c_int, [C.c_uint32, C.c_float, C.c_float, C.c_uint32, C.c_uint32, _P(Uniform)]),
    "mm_check_collision": (C.c_int, [_vp, C.c_uint32, Float3, Float3]),
    "mm_version": (C.c_char_p, []),
}

_lib = None


def library_path():
    return os.path.join(_HERE, _LIB_NAME)


def load_library():
    """Load the in-tree CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("MM_LIBRARY") or library_path()      # MM_LIBRARY: developer override for A/B builds
    if not os.path.exists(path):
        raise MMError(-2, f"{path} is missing: build it with `make -C {_HERE}` (or __graft_entry__.build()); "
                          "there is no CPU fallback for the render path")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)       # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
