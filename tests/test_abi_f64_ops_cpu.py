"""Host-side argument checks of the float64 operator entry points (include/dibr_b200.h): every error is
returned before any CUDA call, so these run without a GPU on fake device pointers."""
import ctypes

import pytest
import torch

from kaolin_b200 import _lib

A = ctypes.c_void_p(4096)          # aligned fake device pointer
M = ctypes.c_void_p(4096 + 8)      # 8 bytes off the 16-byte alignment
B, F, H, W, DIM, K = 1, 4, 8, 8, 1, 30


def packed_fwd(h=H, mult=1000.0, ws_bytes=0, **p):
    a = {k: p.get(k, A) for k in ("z", "xy", "bb", "ff", "first", "feat", "idx", "w")}
    return _lib.lib().dibr_b200_packed_rasterize_forward_f64(
        B, F, h, W, DIM, a["z"], a["xy"], a["bb"], a["ff"], a["first"], mult, 1e-8, a["feat"], a["idx"], a["w"],
        A, ws_bytes, None)


def raster_bwd(h=H, **p):
    a = {k: p.get(k, A) for k in ("g", "idx", "w", "xy", "ff", "gxy", "gff")}
    return _lib.lib().dibr_b200_rasterize_backward_f64(B, F, h, W, DIM, a["g"], a["idx"], a["w"], a["xy"], a["ff"],
                                                       1e-8, a["gxy"], a["gff"], None)


def soft_fwd(h=H, mult=1000.0, ws_bytes=0, **p):
    a = {k: p.get(k, A) for k in ("xy", "bb", "idx", "soft", "prob", "cidx", "ctype")}
    return _lib.lib().dibr_b200_soft_mask_forward_f64(B, F, h, W, K, a["xy"], a["bb"], a["idx"], 7000.0, mult,
                                                      a["soft"], a["prob"], a["cidx"], a["ctype"], A, ws_bytes, None)


def soft_bwd(h=H, mult=1000.0, **p):
    a = {k: p.get(k, A) for k in ("g", "soft", "idx", "prob", "cidx", "ctype", "xy", "gxy")}
    return _lib.lib().dibr_b200_soft_mask_backward_f64(B, F, h, W, K, a["g"], a["soft"], a["idx"], a["prob"],
                                                       a["cidx"], a["ctype"], a["xy"], 7000.0, mult, a["gxy"], None)


ENTRY = {
    "packed_rasterize_forward": (packed_fwd, ("z", "xy", "bb", "ff", "first", "feat", "idx", "w")),
    "rasterize_backward": (raster_bwd, ("g", "idx", "w", "xy", "ff", "gxy", "gff")),
    "soft_mask_forward": (soft_fwd, ("xy", "bb", "idx", "soft", "prob", "cidx", "ctype")),
    "soft_mask_backward": (soft_bwd, ("g", "soft", "idx", "prob", "cidx", "ctype", "xy", "gxy")),
}
REQUIRED = {  # the K-lists of the soft-mask forward are optional as a set
    "soft_mask_forward": ("xy", "bb", "idx", "soft"),
}


@pytest.mark.parametrize("op", sorted(ENTRY))
def test_null_and_misaligned_pointers(op):
    fn, ptrs = ENTRY[op]
    for name in REQUIRED.get(op, ptrs):
        assert fn(**{name: None}) == _lib.EINVAL, name
    for name in ptrs:
        assert fn(**{name: M}) == _lib.EINVAL, name


@pytest.mark.parametrize("op", ["packed_rasterize_forward", "soft_mask_forward", "soft_mask_backward"])
def test_non_positive_multiplier(op):
    fn, _ = ENTRY[op]
    for mult in (0.0, -1000.0):
        assert fn(mult=mult) == _lib.EINVAL, mult


def test_k_lists_all_or_none():
    assert soft_fwd(prob=None, cidx=None, ctype=None) == _lib.EWORKSPACE      # none: reaches the workspace
    for missing in ("prob", "cidx", "ctype"):
        assert soft_fwd(**{missing: None}) == _lib.EINVAL, missing
    assert soft_fwd(prob=None, cidx=None) == _lib.EINVAL


@pytest.mark.parametrize("op", sorted(ENTRY))
def test_image_size_limit(op):
    fn, ptrs = ENTRY[op]
    assert fn(h=16385) == _lib.ESIZE
    # 16384 passes the size check: the call stops at the next host-side check instead
    if op.endswith("forward"):
        assert fn(h=16384) == _lib.EWORKSPACE
    else:
        assert fn(h=16384, **{ptrs[0]: M}) == _lib.EINVAL


def test_workspace_one_byte_short():
    lib = _lib.lib()
    n = lib.dibr_b200_workspace_bytes_f64(B, F, H, W)
    assert n > 0
    assert packed_fwd(ws_bytes=n - 1) == _lib.EWORKSPACE
    n = lib.dibr_b200_workspace_bytes_f64(B, B * F, H, W)
    assert soft_fwd(ws_bytes=n - 1) == _lib.EWORKSPACE


def test_binding_rejects_cpu_double_tensors_as_off_gpu():
    from integration import build_binding
    m = build_binding.load()
    assert m is not None, "integration/_build/kaolin_b200_binding.so is missing: run __graft_entry__.build()"
    d = dict(dtype=torch.float64)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.packed_rasterize_forward_cuda(8, 8, torch.zeros(4, 3, **d), torch.zeros(4, 3, 2, **d),
                                        torch.zeros(4, 4, **d), torch.zeros(4, 3, 2, **d), torch.tensor([0, 4]),
                                        1000., 1e-8)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.rasterize_backward_cuda(torch.zeros(1, 8, 8, 2, **d), torch.zeros(1, 8, 8, 2, **d),
                                  torch.zeros(1, 8, 8, dtype=torch.long), torch.zeros(1, 8, 8, 3, **d),
                                  torch.zeros(1, 4, 3, 2, **d), torch.zeros(1, 4, 3, 2, **d), 1e-8)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.dibr_soft_mask_forward_cuda(torch.zeros(1, 4, 3, 2, **d), torch.zeros(1, 4, 4, **d),
                                      torch.zeros(1, 8, 8, dtype=torch.long), 7000., 30, 1000.)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.dibr_soft_mask_backward_cuda(torch.zeros(1, 8, 8, **d), torch.zeros(1, 8, 8, **d),
                                       torch.zeros(1, 8, 8, dtype=torch.long), torch.zeros(1, 8, 8, 30, **d),
                                       torch.zeros(1, 8, 8, 30, dtype=torch.long),
                                       torch.zeros(1, 8, 8, 30, dtype=torch.uint8), torch.zeros(1, 4, 3, 2, **d),
                                       7000., 1000.)
