"""CPU-side checks of the boundary: the C-ABI library loads and exports every
symbol include/dibr_b200.h declares, argument errors are detected on the host
without a GPU, the Python layer mirrors the reference signatures and refuses to
run without CUDA (no CPU fallback)."""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest
import torch

from kaolin_b200 import _lib, _C
from kaolin_b200.render.mesh import rasterize, dibr_soft_mask, dibr_rasterization

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dibr_b200.h")).read()
    declared = set(re.findall(r"\b(dibr_b200_[a-z_0-9]+)\s*\(", hdr))
    assert {"dibr_b200_forward", "dibr_b200_backward", "dibr_b200_packed_rasterize_forward",
            "dibr_b200_rasterize_backward", "dibr_b200_soft_mask_forward",
            "dibr_b200_soft_mask_backward", "dibr_b200_workspace_bytes",
            "dibr_b200_version"} <= declared
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert set(_lib.SIGNATURES) == declared
    assert lib.dibr_b200_version() >= 200


def test_header_cites_reference_interfaces():
    hdr = open(os.path.join(ROOT, "include", "dibr_b200.h")).read()
    for cite in ("rasterization.h:23-32", "rasterization.h:34-41", "dibr_soft_mask.h:23-30",
                 "dibr_soft_mask.h:32-42", "bindings.cpp:111-115"):
        assert cite in hdr


def test_workspace_query_and_host_side_errors():
    lib = _lib.lib()
    n = lib.dibr_b200_workspace_bytes(32, 32 * 20480, 1024, 1024)
    assert 50e6 < n < 200e6
    assert lib.dibr_b200_workspace_bytes(0, 10, 64, 64) == 0          # bad batch
    assert lib.dibr_b200_workspace_bytes(1, 10, 20000, 64) == 0       # image too large
    # null pointers / bad sizes are rejected before any CUDA call (no GPU needed)
    st = lib.dibr_b200_forward(1, 4, 8, 8, 1, None, None, None, None, None, 1000.0, 1e-8, 3,
                               7000.0, 20.0, 30, None, None, None, None, None, 0, None)
    assert st == _lib.EINVAL
    st = lib.dibr_b200_forward(1, 4, 20000, 8, 1, None, None, None, None, None, 1000.0, 1e-8, 3,
                               7000.0, 20.0, 30, None, None, None, None, None, 0, None)
    assert st == _lib.ESIZE
    with pytest.raises(RuntimeError):
        _lib.check(st, "dibr_b200_forward")
    # float64 entry points: same host-side contract
    n64 = lib.dibr_b200_workspace_bytes_f64(4, 4 * 20480, 1024, 1024)
    assert 0 < n64 < 200e6
    assert lib.dibr_b200_workspace_bytes_f64(0, 10, 64, 64) == 0
    st = lib.dibr_b200_forward_f64(1, 4, 8, 8, 1, None, None, None, None, None, 1000.0, 1e-8, 3,
                                   7000.0, 20.0, 30, None, None, None, None, None, 0, None)
    assert st == _lib.EINVAL
    st = lib.dibr_b200_backward_f64(1, 4, 20000, 8, 1, None, None, None, None, None, None, None,
                                    1000.0, 1e-8, 7000.0, 20.0, 30, None, None, None, 0, 0, None)
    assert st == _lib.ESIZE
    # peer push: argument errors are host-side
    import ctypes
    arr = (ctypes.c_void_p * 1)(ctypes.c_void_p(4096))
    assert lib.dibr_b200_peer_push(None, 32, arr, 1, 0, 0, None) == _lib.EINVAL           # no source
    assert lib.dibr_b200_peer_push(ctypes.c_void_p(4096), 24, arr, 1, 0, 0, None) == _lib.EINVAL   # not 16-byte units
    assert lib.dibr_b200_peer_push(ctypes.c_void_p(4096), 32, arr, 17, 0, 0, None) == _lib.EINVAL  # > 16 destinations
    assert lib.dibr_b200_peer_push(ctypes.c_void_p(4096), 0, arr, 1, 0, 0, None) == 0              # nothing to do
    assert lib.dibr_b200_peer_push_multicast(ctypes.c_void_p(4096), 32, None, 0, 0, None) == _lib.EINVAL
    assert lib.dibr_b200_peer_push_multicast(ctypes.c_void_p(4096), 32, ctypes.c_void_p(4104), 0, 0, None) == _lib.EINVAL


def test_image_size_limit_is_inclusive():
    """DIBR_B200_MAX_IMAGE_DIM = 16384 px per side is accepted (6 bin levels), 16385 is not."""
    lib = _lib.lib()
    for h, w in ((16384, 16384), (16384, 36), (40, 16384)):
        assert lib.dibr_b200_workspace_bytes(1, 100, h, w) > 0, (h, w)
        assert lib.dibr_b200_workspace_bytes_f64(1, 100, h, w) > 0, (h, w)
    for h, w in ((16385, 64), (64, 16385), (16385, 16385)):
        assert lib.dibr_b200_workspace_bytes(1, 100, h, w) == 0, (h, w)
        assert lib.dibr_b200_workspace_bytes_f64(1, 100, h, w) == 0, (h, w)


def test_misaligned_tensor_pointers_are_rejected_on_the_host():
    """Every device tensor pointer must be 16-byte aligned (include/dibr_b200.h): the kernels use
    16-byte vector and cp.async accesses.  A pointer 4 bytes off is refused with EINVAL before any
    CUDA call.  The calls are built so that, without the alignment check, they would stop at a
    different host-side result (a too-small workspace, or nothing to do) instead of launching."""
    lib = _lib.lib()
    A, M = ctypes.c_void_p(4096), ctypes.c_void_p(4096 + 4)     # aligned / misaligned fake device pointers
    acc = _lib.ACCUMULATE

    def fwd(fn, **bad):
        p = {k: A for k in ("fvz", "fvi", "ff", "fnz", "valid", "feat", "idx", "w", "soft")}
        p.update(bad)
        return fn(1, 4, 8, 8, 1, p["fvz"], p["fvi"], p["ff"], p["fnz"], p["valid"], 1000.0, 1e-8, 3,
                  7000.0, 20.0, 30, p["feat"], p["idx"], p["w"], p["soft"], A, 0, None)

    for fn in (lib.dibr_b200_forward, lib.dibr_b200_forward_bf16):
        assert fwd(fn) == _lib.EWORKSPACE                                # aligned: reaches the workspace check
        for name in ("fvz", "fvi", "ff", "fnz", "valid", "feat", "idx", "w", "soft"):
            assert fwd(fn, **{name: M}) == _lib.EINVAL, name
    assert lib.dibr_b200_forward_f64(1, 4, 8, 8, 1, A, A, A, A, A, 1000.0, 1e-8, 3, 7000.0, 20.0, 30,
                                     A, A, A, A, A, 0, None) == _lib.EWORKSPACE
    assert lib.dibr_b200_forward_f64(1, 4, 8, 8, 1, A, M, A, A, A, 1000.0, 1e-8, 3, 7000.0, 20.0, 30,
                                     A, A, A, A, A, 0, None) == _lib.EINVAL

    # backward, soft-mask branch only, accumulating: the next host check is the workspace size
    def bwd(fn, **bad):
        p = {k: A for k in ("gs", "idx", "w", "soft", "fvi", "ff", "gxy", "gff")}
        p.update(bad)
        return fn(1, 4, 8, 8, 1, None, p["gs"], p["idx"], p["w"], p["soft"], p["fvi"], p["ff"],
                  1000.0, 1e-8, 7000.0, 20.0, 30, p["gxy"], p["gff"], A, 0, acc, None)

    for fn in (lib.dibr_b200_backward, lib.dibr_b200_backward_bf16):
        assert bwd(fn) == _lib.EWORKSPACE
        for name in ("gs", "idx", "w", "soft", "fvi", "ff", "gxy", "gff"):
            assert bwd(fn, **{name: M}) == _lib.EINVAL, name
    # an upstream feature gradient at a 4-byte storage offset (no faces: nothing else to do)
    for fn in (lib.dibr_b200_backward, lib.dibr_b200_backward_bf16):
        assert fn(1, 0, 8, 8, 2, M, None, A, A, None, A, A, 1000.0, 1e-8, 7000.0, 20.0, 30,
                  A, A, None, 0, acc, None) == _lib.EINVAL
    assert lib.dibr_b200_backward_views(2, 0, 8, 8, 2, M, None, A, A, None, A, A, 1, 1000.0, 1e-8, 7000.0,
                                        20.0, 30, A, A, None, 0, acc, 1, 2, None) == _lib.EINVAL
    assert lib.dibr_b200_backward_f64(1, 4, 8, 8, 1, None, M, A, A, A, A, A, 1000.0, 1e-8, 7000.0, 20.0, 30,
                                      A, A, A, 0, acc, None) == _lib.EINVAL
    # operators
    assert lib.dibr_b200_packed_rasterize_forward(1, 4, 8, 8, 1, A, A, M, A, A, 1000.0, 1e-8, A, A, A,
                                                  A, 0, None) == _lib.EINVAL
    assert lib.dibr_b200_packed_rasterize_forward(1, 4, 8, 8, 1, A, A, A, A, A, 1000.0, 1e-8, A, A, A,
                                                  A, 0, None) == _lib.EWORKSPACE
    assert lib.dibr_b200_rasterize_backward(1, 0, 8, 8, 2, M, A, A, A, A, 1e-8, A, A, None) == _lib.EINVAL
    assert lib.dibr_b200_soft_mask_forward(1, 4, 8, 8, 30, A, A, A, 7000.0, 1000.0, A, A, M, A,
                                           A, 0, None) == _lib.EINVAL
    assert lib.dibr_b200_soft_mask_forward(1, 4, 8, 8, 30, A, A, A, 7000.0, 1000.0, A, A, A, A,
                                           A, 0, None) == _lib.EWORKSPACE
    assert lib.dibr_b200_soft_mask_backward(1, 4, 8, 8, 30, A, A, A, A, A, A, M, 7000.0, 1000.0,
                                            A, None) == _lib.EINVAL
    assert lib.dibr_b200_deftet_sparse_render_forward(1, 4, 8, 2, A, A, M, A, A, 1e-8, A, A, A, A,
                                                      A, 0, None) == _lib.EINVAL
    assert lib.dibr_b200_deftet_sparse_render_forward(1, 4, 8, 2, A, A, A, A, A, 1e-8, A, A, A, A,
                                                      A, 0, None) == _lib.EWORKSPACE
    assert lib.dibr_b200_deftet_sparse_render_backward(1, 4, 8, 2, 3, M, A, A, A, A, 1e-8, A, A,
                                                       None) == _lib.EINVAL
    assert lib.dibr_b200_texture_mapping_forward(1, 0, 3, 4, 4, M, A, 0, A, None) == _lib.EINVAL
    assert lib.dibr_b200_texture_mapping_forward(1, 0, 3, 4, 4, A, A, 0, A, None) == 0
    assert lib.dibr_b200_mask_iou_backward(1, 16, A, A, A, A, M, A, None) == _lib.EINVAL


def test_misaligned_views_are_copied_before_the_abi():
    """The Python layers hand the C ABI a 16-byte aligned copy of a tensor view at a storage offset."""
    from kaolin_b200.render.mesh import _host
    buf = torch.zeros(1 + 4 * 3 * 2)
    t = buf[1:].view(4, 3, 2)
    assert t.is_contiguous() and t.data_ptr() % 16 == 4
    c = _host.aligned(t)
    assert c.data_ptr() % 16 == 0 and torch.equal(c, t) and c.is_contiguous()
    a = buf[4:].view(-1)
    assert a.data_ptr() % 16 == 0 and _host.aligned(a) is a            # aligned views are passed through
    assert _host.aligned(None) is None
    h = torch.zeros(9, dtype=torch.bfloat16)[1:]
    assert h.data_ptr() % 16 == 2 and _host.aligned(h).data_ptr() % 16 == 0


def test_python_signatures_match_reference():
    """rasterization.py:373-381, dibr.py:75-76,119-122."""
    sig = inspect.signature(rasterize)
    assert list(sig.parameters) == ["height", "width", "face_vertices_z", "face_vertices_image",
                                    "face_features", "valid_faces", "multiplier", "eps", "backend"]
    assert sig.parameters["backend"].default == "cuda" and sig.parameters["eps"].default is None
    sig = inspect.signature(dibr_soft_mask)
    assert [(k, v.default) for k, v in sig.parameters.items()][2:] == [
        ("sigmainv", 7000), ("boxlen", 0.02), ("knum", 30), ("multiplier", 1000.)]
    sig = inspect.signature(dibr_rasterization)
    assert list(sig.parameters) == ["height", "width", "face_vertices_z", "face_vertices_image",
                                    "face_features", "face_normals_z", "sigmainv", "boxlen", "knum",
                                    "multiplier", "eps", "rast_backend"]
    for op in ("packed_rasterize_forward_cuda", "rasterize_backward_cuda",
               "dibr_soft_mask_forward_cuda", "dibr_soft_mask_backward_cuda"):
        assert callable(getattr(_C.render.mesh, op))          # bindings.cpp:111-115


def test_no_cpu_fallback():
    fvz = torch.zeros(1, 4, 3)
    fvi = torch.zeros(1, 4, 3, 2)
    ff = torch.zeros(1, 4, 3, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        rasterize(8, 8, fvz, fvi, ff)
    with pytest.raises(RuntimeError, match="CUDA"):
        dibr_rasterization(8, 8, fvz, fvi, ff, torch.zeros(1, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        dibr_soft_mask(fvi, torch.zeros(1, 8, 8, dtype=torch.long))
    with pytest.raises(RuntimeError):
        _C.render.mesh.rasterize_backward_cuda(torch.zeros(1, 8, 8, 2), torch.zeros(1, 8, 8, 2),
                                               torch.zeros(1, 8, 8, dtype=torch.long),
                                               torch.zeros(1, 8, 8, 3), fvi, ff, 1e-8)
    with pytest.raises(ValueError):
        rasterize(8, 8, fvz, fvi, ff, backend="nvdiffrast")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "kaolin_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "oracle/" not in src.replace("tests/", ""), f


def test_hit_cache_sizing_policy():
    """Every tile is cached when that fits in 4 GB (BASELINE configs[1]/[2]: a third of the tiles
    touch the silhouette at 256^2 - caching 1/8 of them halved the throughput), else as many as fit."""
    from kaolin_b200.render.mesh import _host
    lib = _lib.lib()
    assert _host.cache_tiles_for(8, 256, 256, 30) == 8 * 16 * 16                 # c2: all tiles
    c3 = _host.cache_tiles_for(64, 512, 512, 30)
    assert 0.5 * 64 * 1024 < c3 <= 64 * 1024                                      # c3: more than half
    c4 = _host.cache_tiles_for(32, 1024, 1024, 30)
    assert 0.25 * 32 * 4096 < c4 < 32 * 4096                                      # c4: the 4 GB cap
    base = lib.dibr_b200_workspace_bytes(32, 32 * 20480, 1024, 1024)
    full = lib.dibr_b200_workspace_bytes_cached(32, 32 * 20480, 1024, 1024, 30, c4)
    assert base < full <= base + _host.CACHE_MAX_BYTES + (1 << 20)
    assert _host.cache_tiles_for(1, 16, 16, 30) == 1
