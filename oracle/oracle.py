"""ctypes wrapper of oracle/libmm_oracle.so (mm_oracle.cpp): the scalar fp32 transcription of the reference's
`compute_shader` (reference src/shaders.metal:245-368) and its helpers.  TEST INFRASTRUCTURE — see mm_oracle.cpp."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libmm_oracle.so")
_lib = None
_native_dir = None


class _Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("paths", "rays", "inner_visits", "leaf_visits", "rect_tests", "hits",
                                          "literal_rays", "max_stack")]


class _Debug(C.Structure):
    _fields_ = [("first_hit", C.c_void_p), ("segments", C.c_void_p), ("mirror_hits", C.c_void_p), ("radiance", C.c_void_p)]


def build():
    subprocess.check_call(["make", "-C", _HERE, "-s"])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        _lib = C.CDLL(_LIB)
        _lib.mmo_render.restype = C.c_int
        _lib.mmo_render.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                    C.c_void_p, C.POINTER(_Counters), C.POINTER(_Debug), C.c_int]
        _lib.mmo_random.restype = C.c_float
        _lib.mmo_random.argtypes = [C.POINTER(C.c_uint32)]
        _lib.mmo_random_word.restype = C.c_uint32
        _lib.mmo_random_word.argtypes = [C.POINTER(C.c_uint32)]
        _lib.mmo_seed.restype = C.c_uint32
        _lib.mmo_seed.argtypes = [C.c_float, C.c_float, C.c_uint32, C.c_uint32, C.c_uint32]
        _lib.mmo_intersect_aabb.restype = C.c_float
        _lib.mmo_intersect_aabb.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
        _lib.mmo_ray_rect.restype = C.c_int
        _lib.mmo_ray_rect.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_float)]
        _lib.mmo_quat_mult.restype = None
        _lib.mmo_quat_mult.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.mmo_num_threads.restype = C.c_int
        _lib.mmo_trace_rays.restype = C.c_int
        _lib.mmo_trace_rays.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                        C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    return _lib


def use_native():
    """bench.py only: build libmm_oracle.so for THIS machine (g++ -march=native, same source, still no contraction and
    no fast-math) in a temporary directory, so that the tree may be read-only, and use it for every later call.  Returns
    a one-line description of what is in use.  Must run before the first lib() call of the process."""
    global _LIB, _lib, _native_dir
    _native_dir = tempfile.TemporaryDirectory(prefix="mm_oracle_native_")       # removed when the process exits
    native = os.path.join(_native_dir.name, "libmm_oracle.so")
    try:
        subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"NATIVE_DIR={_native_dir.name}"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    except Exception as e:
        return f"portable build (native build failed: {type(e).__name__})"
    if _lib is not None or not os.path.exists(native):
        return "portable build"
    _LIB = native
    return "g++ -O2 -march=native -ffp-contract=off -fopenmp, built on this machine"


def num_threads():
    return int(lib().mmo_num_threads())


def render(scene, noise, uniform, params, chunks, debug=False, threads=0, out=None):
    """Same contract as Renderer.render: (image[H,W,4], counters dict, debug dict|None).  `uniform`/`params` are the
    ctypes structs of the C-ABI (byte layouts are shared; the oracle reads them through the same header)."""
    L = lib()
    planes = np.ascontiguousarray(scene.planes)
    nodes = np.ascontiguousarray(scene.nodes)
    indices = np.ascontiguousarray(scene.indices, dtype=np.uint32)
    materials = np.ascontiguousarray(scene.materials, dtype=np.uint8)
    emissions = np.ascontiguousarray(scene.emissions, dtype=np.float32)
    noise = np.ascontiguousarray(noise, dtype=np.uint8)
    chunks = np.ascontiguousarray(chunks)
    nh, nw = noise.shape[:2]
    H, W = int(uniform.view_height), int(uniform.view_width)
    if out is None:
        out = np.zeros((H, W, 4), dtype=np.float32)
    cnt = _Counters()
    dbg, dstruct = None, None
    if debug:
        n_groups = params.group_count or params.grid_x * params.grid_y
        n_paths = n_groups * uniform.chunk_width ** 2 * params.spp
        dbg = {"first_hit": np.empty(n_paths, np.uint32), "segments": np.empty(n_paths, np.uint32),
               "mirror_hits": np.empty(n_paths, np.uint32), "radiance": np.empty((n_paths, 3), np.float32)}
        dstruct = _Debug(dbg["first_hit"].ctypes.data, dbg["segments"].ctypes.data, dbg["mirror_hits"].ctypes.data,
                         dbg["radiance"].ctypes.data)
    rc = L.mmo_render(planes.ctypes.data, len(planes), nodes.ctypes.data, len(nodes), indices.ctypes.data,
                      materials.ctypes.data, emissions.ctypes.data, noise.ctypes.data, nw, nh,
                      C.addressof(uniform), C.addressof(params), chunks.ctypes.data, len(chunks), out.ctypes.data,
                      C.byref(cnt), C.byref(dstruct) if dstruct else None, threads)
    if rc != 0:
        raise RuntimeError(f"mmo_render failed: {rc}")
    return out, {n: int(getattr(cnt, n)) for n, _ in cnt._fields_}, dbg


def trace_rays(scene, rays, index=None, flags=0, threads=0):
    """intersect_bvh_iterative per ray (mmo_trace_rays): rays [n, 8] float32 (ori.xyz, dir.xyz, t, alive), index [n] starting
    plane indices or None.  Returns a dict of numpy arrays: t, index, inner, leaf, rect, max_stack, overflow."""
    planes = np.ascontiguousarray(scene.planes)
    nodes = np.ascontiguousarray(scene.nodes)
    indices = np.ascontiguousarray(scene.indices, dtype=np.uint32)
    rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 8)
    n = len(rays)
    idx = None if index is None else np.ascontiguousarray(index, dtype=np.uint32)
    t, out_idx, counts = np.empty(n, np.float32), np.empty(n, np.uint32), np.empty((n, 5), np.uint64)
    rc = lib().mmo_trace_rays(planes.ctypes.data, len(planes), nodes.ctypes.data, len(nodes), indices.ctypes.data, flags,
                              rays.ctypes.data, None if idx is None else idx.ctypes.data, n, t.ctypes.data, out_idx.ctypes.data,
                              counts.ctypes.data, threads)
    if rc not in (0, -4):
        raise RuntimeError(f"mmo_trace_rays failed: {rc}")
    out = {"t": t, "index": out_idx}
    for i, k in enumerate(("inner", "leaf", "rect", "max_stack", "overflow")):
        out[k] = counts[:, i]
    return out


def random_words(seed, n):
    st = C.c_uint32(seed)
    return [int(lib().mmo_random_word(C.byref(st))) for _ in range(n)], int(st.value)


def random_floats(seed, n):
    st = C.c_uint32(seed)
    return [float(lib().mmo_random(C.byref(st))) for _ in range(n)]


def seed(nx, ny, texid_x, texid_y, time):
    return int(lib().mmo_seed(nx, ny, texid_x, texid_y, time))


def intersect_aabb(ori, direction, t, bmin, bmax):
    a = [np.ascontiguousarray(v, dtype=np.float32) for v in (ori, direction, bmin, bmax)]
    return float(lib().mmo_intersect_aabb(a[0].ctypes.data, a[1].ctypes.data, t, a[2].ctypes.data, a[3].ctypes.data))


def ray_rect(ori, direction, t, plane_record):
    o = np.ascontiguousarray(ori, dtype=np.float32)
    d = np.ascontiguousarray(direction, dtype=np.float32)
    p = np.ascontiguousarray(plane_record)
    tout = C.c_float()
    hit = lib().mmo_ray_rect(o.ctypes.data, d.ctypes.data, t, p.ctypes.data, C.byref(tout))
    return bool(hit), float(tout.value)


def quat_mult(v, q):
    v = np.ascontiguousarray(v, dtype=np.float32)
    q = np.ascontiguousarray(q, dtype=np.float32)
    out = np.zeros(3, dtype=np.float32)
    lib().mmo_quat_mult(v.ctypes.data, q.ctypes.data, out.ctypes.data)
    return out
