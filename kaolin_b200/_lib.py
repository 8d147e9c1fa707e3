"""ctypes binding of the C ABI (include/dibr_b200.h) + in-tree build of libdibr_b200.so.

PyTorch is used for device memory and streams only; every compute call goes
through the ``extern "C"`` entry points with raw device pointers.  There is no
fallback: a missing library is an error.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# DIBR_B200_LIB: an alternative build of the same sources (A/B experiments on the GPU box only)
LIB_PATH = os.environ.get("DIBR_B200_LIB") or os.path.join(CSRC, "libdibr_b200.so")
SOURCES = [os.path.join(CSRC, "dibr_b200.cu"), os.path.join(CSRC, "mesh_pipeline.cu"),
           os.path.join(CSRC, "deftet.cu"), os.path.join(CSRC, "peer_push.cu")]
HEADERS = [os.path.join(CSRC, "dibr_math.cuh"), os.path.join(CSRC, "dibr_math_f64.cuh"),
           os.path.join(CSRC, "dibr_f64.cuh"),
           os.path.join(_HERE, "..", "include", "dibr_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]

EINVAL, EWORKSPACE, ESIZE = -1, -3, -4
ALIGNMENT = 16                      # DIBR_B200_ALIGNMENT: bytes, every device tensor pointer
RASTER, SOFT_MASK = 1, 2
BINS_VALID, ACCUMULATE = 1, 2      # dibr_b200_backward flags

_lock = threading.Lock()
_lib = None

_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_f = ctypes.c_float
_d = ctypes.c_double
_sz = ctypes.c_size_t
_fp3 = ctypes.POINTER(ctypes.c_float)      # HOST pointer to 3 floats (camera_proj)

SIGNATURES = {
    "dibr_b200_version": (_i, []),
    "dibr_b200_trace_begin": (_i, []),
    "dibr_b200_peer_push": (_i, [_vp, _sz, ctypes.POINTER(ctypes.c_void_p), _i, _sz, _i, _vp]),
    "dibr_b200_peer_push_multicast": (_i, [_vp, _sz, _vp, _sz, _i, _vp]),
    "dibr_b200_trace_end": (_i, [ctypes.c_char_p, _sz, ctypes.POINTER(ctypes.c_float), _i]),
    "dibr_b200_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "dibr_b200_workspace_bytes_cached": (_sz, [_i, _i64, _i, _i, _i, _i64]),
    "dibr_b200_forward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _f, _f, _i,
                               _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_backward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _i, _vp]),
    "dibr_b200_backward_views": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i,
                                      _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _i, _i, _i, _vp]),
    "dibr_b200_workspace_bytes_f64": (_sz, [_i, _i64, _i, _i]),
    "dibr_b200_forward_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _f, _d, _i,
                                   _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_backward_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                    _f, _f, _f, _d, _i, _vp, _vp, _vp, _sz, _i, _vp]),
    "dibr_b200_forward_bf16": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _f, _f, _i,
                                    _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_backward_bf16": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _i, _vp]),
    "dibr_b200_packed_rasterize_forward": (_i, [_i, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f,
                                                _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_rasterize_backward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f,
                                          _vp, _vp, _vp]),
    "dibr_b200_soft_mask_forward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _f, _f,
                                         _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_soft_mask_backward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _f, _f, _vp, _vp]),
    "dibr_b200_packed_rasterize_forward_f64": (_i, [_i, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f,
                                                    _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_rasterize_backward_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f,
                                              _vp, _vp, _vp]),
    "dibr_b200_soft_mask_forward_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _f, _f,
                                             _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_soft_mask_backward_f64": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                              _f, _f, _vp, _vp]),
    # SURVEY.md §8(f): the steps either side of the rasterizer (csrc/mesh_pipeline.cu)
    "dibr_b200_prepare_vertices_forward": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _fp3, _vp, _vp, _vp, _vp]),
    "dibr_b200_prepare_vertices_backward": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _fp3, _vp, _vp, _vp,
                                                 _vp, _vp]),
    "dibr_b200_texture_mapping_forward": (_i, [_i, _i64, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "dibr_b200_texture_mapping_backward": (_i, [_i, _i64, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "dibr_b200_mask_iou_forward": (_i, [_i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "dibr_b200_mask_iou_backward": (_i, [_i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    # SURVEY.md §8(f) rank 3: DefTet volumetric renderer operators (csrc/deftet.cu)
    "dibr_b200_deftet_workspace_bytes": (_sz, [_i, _i]),
    "dibr_b200_deftet_sparse_render_forward": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f,
                                                    _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dibr_b200_deftet_sparse_render_backward": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f,
                                                     _vp, _vp, _vp]),
}


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.exists(p) and os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a -> kaolin_b200/csrc/libdibr_b200.so."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH] + SOURCES
    if verbose:
        cmd += ["-Xptxas", "-v"]
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB_PATH


def lib():
    """The loaded library; raises if it has not been built (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"kaolin_b200: CUDA library {LIB_PATH} is missing; build it with "
                    "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                    "There is no CPU fallback.")
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def trace_begin():
    """Per-kernel CUDA-event timing of every launch made by THIS thread until trace_end()."""
    lib().dibr_b200_trace_begin()


def trace_end(capacity=256):
    """-> [(kernel name, milliseconds), ...] in launch order (synchronises the recorded events)."""
    names = ctypes.create_string_buffer(64 * capacity)
    ms = (ctypes.c_float * capacity)()
    n = lib().dibr_b200_trace_end(names, len(names), ms, capacity)
    if n < 0:
        raise RuntimeError("dibr_b200_trace_end failed")
    got = names.value.decode().split("\n")[:n]
    return [(got[i], float(ms[i])) for i in range(min(n, capacity))]


def check(status, what):
    if status == 0:
        return
    if status == EINVAL:
        raise RuntimeError(f"{what}: invalid argument (null or misaligned pointer, non-positive size or multiplier)")
    if status == EWORKSPACE:
        raise RuntimeError(f"{what}: workspace too small")
    if status == ESIZE:
        raise RuntimeError(f"{what}: image larger than 16384 px per side or index overflow")
    raise RuntimeError(f"{what}: CUDA error {status}")
