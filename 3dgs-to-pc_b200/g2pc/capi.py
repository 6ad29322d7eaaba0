"""ctypes binding of libg2pc.so (the C-ABI CUDA library declared in include/g2pc.h).

This is the stub a maintainer of the reference would add in place of
`from gaussian_pointcloud_rasterization import _C` (gaussian_pointcloud_rasterization/__init__.py:14) and of
the torch call chains in gauss_to_pc.py:140-275.  There is NO fallback: if the library is missing or a call
fails, an exception is raised.
"""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libg2pc.so")

F32, F64 = 0, 1
CULL_EPS_NORM, CULL_EXPLICIT = 0, 1
ST_OVERFLOW, ST_CHOLFAIL, ST_CHOLREG, ST_WORDS = 0, 1, 2, 4

_c_void_p = ctypes.c_void_p
_i32, _i64, _u32, _u64, _f32 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_float

# name -> argtypes, exactly as declared in include/g2pc.h
SIGNATURES = {
    "g2pc_version": ([], ctypes.c_int),
    "g2pc_last_error": ([], ctypes.c_char_p),
    "g2pc_cov_build": ([_c_void_p, _c_void_p, ctypes.c_int, _f32, _i64, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_normals": ([_c_void_p, _c_void_p, ctypes.c_int, _i64, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_eigvals_sym3": ([_c_void_p, _i64, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_sample_count": ([_c_void_p, _c_void_p, _c_void_p, ctypes.c_int, _c_void_p, _c_void_p, _c_void_p, _i64, _i64,
                           _c_void_p, _i32, _i32, _i32, _f32, _i32, _u64, _u32, _c_void_p, _c_void_p, _c_void_p,
                           _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_sample_emit_chunk_points": ([], ctypes.c_int),
    "g2pc_sample_emit": ([_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p, _i32, _u64, _u32, _c_void_p,
                          _c_void_p, _c_void_p, ctypes.c_int, _i64, _c_void_p], ctypes.c_int),
    "g2pc_dump_eps": ([_c_void_p, _i64, _i32, _i32, _u64, _u32, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_cull_workspace_bytes": ([_i64], ctypes.c_int64),
    "g2pc_cull_select": ([_c_void_p, _f32, _c_void_p, _f32, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                          _c_void_p, _i64, _i64, _i64, _c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p], ctypes.c_int),
    "g2pc_gather_rows": ([_c_void_p, _i64, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_ppg_workspace_bytes": ([_i64], ctypes.c_int64),
    "g2pc_points_per_gaussian": ([_c_void_p, _c_void_p, _i64, ctypes.c_double, _c_void_p, _c_void_p, _c_void_p, _i64,
                                  _c_void_p], ctypes.c_int),
    "g2pc_knn_workspace_bytes": ([_i64, _i32], ctypes.c_int64),
    "g2pc_knn_mean_distance": ([_c_void_p, _i64, _i32, _c_void_p, _c_void_p, _i64, _c_void_p], ctypes.c_int),
    "g2pc_outlier_workspace_bytes": ([_i64], ctypes.c_int64),
    "g2pc_outlier_mask": ([_c_void_p, _i64, ctypes.c_double, _c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p],
                          ctypes.c_int),
    "g2pc_pack_geometry": ([_c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_preprocess": ([_c_void_p, _c_void_p, _c_void_p, _i32, _i32, _i64, _c_void_p, _c_void_p, _c_void_p, _i32, _u32,
                         _u32, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_depth_sort_workspace_bytes": ([_i64], ctypes.c_int64),
    "g2pc_depth_sort": ([_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _i64, _c_void_p], ctypes.c_int),
    "g2pc_build_tree": ([_c_void_p, _i32, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i32, _i64, _i64,
                         _i64, _i32, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_multisplit_chunk": ([_i32], ctypes.c_int32),
    "g2pc_multisplit_rows": ([_i64, _i32], ctypes.c_int32),
    "g2pc_multisplit": ([_c_void_p, _i64, _c_void_p, _i32, _i32, _c_void_p, _i32, _u32, _u32, _c_void_p, _c_void_p,
                         _c_void_p, _c_void_p, _i32, _i32, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_blend": ([_c_void_p, _c_void_p, _c_void_p, _c_void_p, _i32, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                    _c_void_p, _c_void_p, _i32, _i32, _f32, _f32, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_blend_set_compact": ([ctypes.c_int], None),
    "g2pc_accumulate": ([_c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p, _i32, _c_void_p], ctypes.c_int),
    "g2pc_tiles_preprocess": ([_c_void_p, _c_void_p, _c_void_p, _i32, _i32, _i32, _i64, _c_void_p, _c_void_p, _c_void_p,
                               _c_void_p, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_tiles_build": ([_c_void_p, _i32, _i32, _c_void_p, _c_void_p, _i32, _i64, _i64, _i32, _i32, _c_void_p,
                          _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_multisplit_grid": ([_c_void_p, _i64, _i32, _i32, _c_void_p, _c_void_p, _c_void_p, _i32, _i32, _c_void_p,
                              _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_tiles_blend": ([_c_void_p, _c_void_p, _c_void_p, _c_void_p, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                          _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i32, _i32, _c_void_p, _c_void_p, _c_void_p,
                          _c_void_p], ctypes.c_int),
    "g2pc_tiles_accumulate": ([_c_void_p, _c_void_p, _c_void_p, _i32, _i32, _i64, _c_void_p, _c_void_p, _c_void_p,
                               _c_void_p, _c_void_p, _i32, _c_void_p, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    "g2pc_fill_u32": ([_c_void_p, _u32, _i64, _c_void_p], ctypes.c_int),
    "g2pc_compose_image": ([_c_void_p, _c_void_p, _i32, _i32, _f32, _c_void_p, _c_void_p], ctypes.c_int),
}


class Raster(ctypes.Structure):
    """g2pc_raster_t"""
    _fields_ = [("viewmatrix", _f32 * 16), ("projmatrix", _f32 * 16), ("campos", _f32 * 3), ("tan_fovx", _f32),
                ("tan_fovy", _f32), ("width", _i32), ("height", _i32)]


class Camera(ctypes.Structure):
    """g2pc_camera_t"""
    _fields_ = [("view", _f32 * 16), ("proj", _f32 * 16), ("campos", _f32 * 3), ("tan_fovx", _f32),
                ("tan_fovy", _f32), ("focal_x", _f32), ("focal_y", _f32), ("width", _i32), ("height", _i32)]


(HDR_NUM_LEAVES, HDR_TOTAL_INST, HDR_TOTAL_PIX, HDR_NEED_DEEPER, HDR_LEAF_OVERFLOW, HDR_CAP_OVERFLOW, HDR_POISON,
 HDR_FRAME, HDR_TOTAL_INST_HI) = range(9)
HDR_WORDS = 16
WORK_COUNTERS = 4
STAT_WARP_GAUSSIANS, STAT_WORDS = 0, 4
LEAF_WORDS = 8  # g2pc_leaf_t = 8 x int32

_lib = None


class G2pcError(RuntimeError):
    pass


def load(path=None):
    """Load libg2pc.so and attach the argument types.  Raises if the library is absent (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise G2pcError(
            f"{path} not found: build it with `python -m g2pc.build` (or __graft_entry__.build()). "
            "There is no CPU fallback for the g2pc kernels.")
    lib = ctypes.CDLL(path)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


# ---- launch accounting (bench.py reads these) -------------------------------------------------------------------
LAUNCHES = 0      # number of hand-written g2pc kernels launched since the last reset
TIMING = None     # None, or a dict filled as {entry point name: [(start_event, end_event), ...]}: every launch is
                  # bracketed with CUDA events on the current stream (bench.py)
# hand-written kernels launched per entry point (default 1); the radix sorts inside g2pc_depth_sort and
# g2pc_knn_mean_distance are cub's (library)
_OWN_KERNELS = {"g2pc_multisplit": 5, "g2pc_multisplit_grid": 5, "g2pc_depth_sort": 0, "g2pc_cull_select": 3,
                "g2pc_points_per_gaussian": 5, "g2pc_knn_mean_distance": 6, "g2pc_outlier_mask": 5}
_NOT_KERNELS = {"g2pc_version", "g2pc_last_error", "g2pc_sample_emit_chunk_points", "g2pc_multisplit_chunk",
                "g2pc_multisplit_rows", "g2pc_blend_set_compact", "g2pc_cull_workspace_bytes", "g2pc_ppg_workspace_bytes",
                "g2pc_depth_sort_workspace_bytes", "g2pc_knn_workspace_bytes", "g2pc_outlier_workspace_bytes"}


def call(name, *args):
    """Invoke entry point `name` (must be declared in SIGNATURES), check its status, count it, and — when TIMING is a
    dict — bracket it with CUDA events on the current stream."""
    global LAUNCHES
    fn = getattr(load(), name)
    if TIMING is not None and name not in _NOT_KERNELS:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        status = fn(*args)
        b.record()
        TIMING.setdefault(name, []).append((a, b))
    else:
        status = fn(*args)
    LAUNCHES += _OWN_KERNELS.get(name, 1)
    check(status, name)


def check(status, what):
    if status != 0:
        msg = load().g2pc_last_error()
        raise G2pcError(f"{what} failed (status {status}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def dtype_code(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise G2pcError(f"unsupported dtype {t.dtype} (need float32 or float64)")


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise G2pcError("g2pc kernels need CUDA tensors; there is no CPU fallback "
                            f"(got a tensor on {t.device})")
