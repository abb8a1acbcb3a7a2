"""mirror_maze_b200 (the task's `mirror-maze_b200/`, a symlink to this importable directory) — B200-native drop-in for mirror-maze's per-pixel render kernel.

Only what the hot path needs: `csrc/` (hand-written sm_100a CUDA + the C-ABI of include/mirror_maze_cuda.h),
`abi.py` (ctypes binding of that ABI), `host.py` (mirror of the reference's host surface: maze -> scene -> BVH ->
uniform -> chunk list, reference src/main.rs:357-588,732-755) and `renderer.py` (the dispatch the reference encodes
at src/main.rs:867-886, including the multi-GPU tile partition).  There is no CPU fallback: rendering raises when
the CUDA library or a B200 is missing.
"""
from .abi import (MMError, load_library, library_path, Float2, Float3, Float4, Plane, BVHNode, Camera, Uniform, Chunk,
                  Params, Counters, SceneInfo, FLAG_COUNTERS, FLAG_FORCE_LITERAL, FLAG_RCP_SLAB, FLAG_NO_ZERO_COPY, FLAG_POOL_KERNEL, FLAG_SCREEN_RGBA8, FLAG_REGROUP, FLAG_GENERAL_RECTS, FLAG_NO_TAIL, FLAG_NO_Y_TABLE, MAX_STACK, MAX_BVH_DEPTH,
                  EXCHANGE_PEER, EXCHANGE_NCCL, EXCHANGE_NONE, MAX_VIEWS)
from .host import (MazeScene, StdRng, default_uniform, gen_chunks, calculate_quaternion, update_quat_angle, quat_mult,
                   load_noise, full_frame_params, check_collision, chacha_block, ChunkBag, move_camera, rect_edge_thresholds, axis_rect)
from .renderer import Renderer, MultiRenderer, HostFrame, TiledFrameRenderer, tile_partition

__all__ = [n for n in dir() if not n.startswith("_")]
