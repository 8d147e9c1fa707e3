"""Host-side plumbing shared by the autograd wrappers: argument checks in the
style of the reference's C++ wrappers (rasterization.cpp:70-85,
dibr_soft_mask.cpp:63-82), workspace allocation, and the ctypes calls."""
import ctypes

import torch

from ... import _lib


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def aligned(t):
    """``t`` itself, or a copy when its data pointer is not a multiple of _lib.ALIGNMENT bytes.

    The C ABI rejects such pointers (the kernels use 16-byte vector and cp.async accesses); a
    contiguous view at a storage offset, such as an upstream gradient ``buf[1:].view(...)`` that
    autograd passes through unchanged, gets there otherwise."""
    if t is None or t.data_ptr() % _lib.ALIGNMENT == 0:
        return t
    return t.clone(memory_format=torch.contiguous_format)


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


FEATURE_DTYPES = (torch.float32, torch.bfloat16)   # storage of face_features / interpolated features


def check_feature_dtype(func, name, t):
    if t is not None and t.dtype not in FEATURE_DTYPES:
        raise RuntimeError(f"\"{func}\" not implemented for '{str(t.dtype).replace('torch.', '')}' "
                           f"({name}: kaolin_b200 stores features as float32 or bfloat16)")


def check_tensors(func, named, dtype=torch.float32):
    """All tensors on the same CUDA device with the expected dtype (no CPU path)."""
    dev = None
    for name, t in named:
        if t is None:
            continue
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{func}: {name} must be a torch.Tensor")
        if not t.is_cuda:
            raise RuntimeError(f"{func}: expected {name} to be a CUDA tensor "
                               "(kaolin_b200 has no CPU path)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"{func}: expected all tensors on {dev}, {name} is on {t.device}")
        if dtype is not None and t.is_floating_point() and t.dtype != dtype:
            raise RuntimeError(f"\"{func}\" not implemented for '{str(t.dtype).replace('torch.', '')}' "
                               "(kaolin_b200 supports float32 and float64)")
    return dev


def check_size(func, name, t, shape):
    if tuple(t.shape) != tuple(shape):
        raise RuntimeError(f"{func}: expected {name} of size {list(shape)}, got {list(t.shape)}")


# Screen tiles that get a soft-mask hit-cache block (forward scratch of the enumerate / evaluate
# kernels AND the backward's input).  Every tile when that fits in CACHE_MAX_BYTES - at 256^2 a third
# of the 16x16 tiles touch the silhouette, at 1024^2 a tenth, and the host cannot know the number
# without a device sync - else as many as fit; tiles beyond the cache take the single-kernel path
# and are recomputed in backward: same results, several times slower.  Both knobs are module
# attributes (a caller with many live forward graphs can lower CACHE_MAX_BYTES); callers that need
# no gradient do not keep the workspace alive (render/mesh/dibr.py).
CACHE_TILE_FRACTION = 1.0
CACHE_MIN_TILES = 64
CACHE_MAX_BYTES = 4 << 30


def cache_tiles_for(batch, height, width, knum):
    """How many 16x16 tiles get a soft-mask hit-cache block (3072*knum + 17.4 KB each)."""
    tiles = batch * ((height + 15) // 16) * ((width + 15) // 16)
    want = max(CACHE_MIN_TILES, int(tiles * CACHE_TILE_FRACTION))
    return min(tiles, want, max(1, CACHE_MAX_BYTES // (3072 * knum + 17500)))


_ws_bytes = {}     # (batch, faces, H, W, knum, cache policy) -> bytes: a pure function of the shape


def workspace(batch, total_faces, height, width, device, knum=0):
    key = (batch, total_faces, height, width, knum, CACHE_TILE_FRACTION, CACHE_MAX_BYTES)
    n = _ws_bytes.get(key)
    if n is None:
        if knum > 0:
            want = cache_tiles_for(batch, height, width, knum)
            n = _lib.lib().dibr_b200_workspace_bytes_cached(batch, total_faces, height, width, knum, want)
        else:
            n = _lib.lib().dibr_b200_workspace_bytes(batch, total_faces, height, width)
        if len(_ws_bytes) < 4096:
            _ws_bytes[key] = n
    if n == 0:
        raise RuntimeError("kaolin_b200: unsupported problem size "
                           f"(batch={batch}, faces={total_faces}, image={height}x{width})")
    return torch.empty(n, dtype=torch.uint8, device=device)


def forward(mode, height, width, fvz, fvi, ff, fnz, valid_u8, multiplier, eps,
            sigmainv, boxlen_m, knum, face_idx_in=None):
    """Calls dibr_b200_forward; returns (feat, face_idx, weights, soft, workspace)."""
    fvz, fvi, ff, fnz, valid_u8, face_idx_in = map(aligned, (fvz, fvi, ff, fnz, valid_u8, face_idx_in))
    dev = fvi.device
    B, F = fvi.shape[0], fvi.shape[1]
    D = 0 if ff is None else ff.shape[-1]
    raster = bool(mode & _lib.RASTER)
    soft_on = bool(mode & _lib.SOFT_MASK)
    bf16 = ff is not None and ff.dtype == torch.bfloat16
    feat = torch.empty((B, height, width, D), dtype=torch.bfloat16 if bf16 else torch.float32,
                       device=dev) if raster else None
    wts = torch.empty((B, height, width, 3), dtype=torch.float32, device=dev) if raster else None
    idx = torch.empty((B, height, width), dtype=torch.int64, device=dev) if raster else face_idx_in
    soft = torch.empty((B, height, width), dtype=torch.float32, device=dev) if soft_on else None
    if B == 0:       # an empty view shard (batch < world size): empty images, nothing to launch
        return feat, idx, wts, soft, None
    ws = workspace(B, B * F, height, width, dev, knum if soft_on else 0)
    with torch.cuda.device(dev):
        fn = _lib.lib().dibr_b200_forward_bf16 if bf16 else _lib.lib().dibr_b200_forward
        st = fn(
            B, F, height, width, D, ptr(fvz), ptr(fvi), ptr(ff), ptr(fnz), ptr(valid_u8),
            float(multiplier), float(eps), mode, float(sigmainv), float(boxlen_m), int(knum),
            ptr(feat), ptr(idx), ptr(wts), ptr(soft), ptr(ws), ws.numel(), stream_ptr(dev))
    _lib.check(st, "dibr_b200_forward")
    return feat, idx, wts, soft, ws



def _backward_call(B, F, height, width, D, g_feat, g_soft, face_idx, wts, soft, fvi, ff, multiplier, eps,
                   sigmainv, boxlen_m, knum, g_fvi, g_ff, ws, ws_bytes, flags, dev, views=None):
    bf16 = ff is not None and ff.dtype == torch.bfloat16
    if g_feat is not None and ff is not None and g_feat.dtype != ff.dtype:
        raise RuntimeError(f"dibr_b200_backward: grad_features is {g_feat.dtype}, face_features is {ff.dtype}")
    if views is not None:
        with torch.cuda.device(dev):
            st = _lib.lib().dibr_b200_backward_views(
                B, F, height, width, D, ptr(g_feat), ptr(g_soft), ptr(face_idx), ptr(wts), ptr(soft),
                ptr(fvi), ptr(ff), int(bf16), float(multiplier), float(eps), float(sigmainv), float(boxlen_m),
                int(knum), ptr(g_fvi), ptr(g_ff), ptr(ws), ws_bytes, int(flags), int(views[0]), int(views[1]),
                stream_ptr(dev))
        _lib.check(st, "dibr_b200_backward_views")
        return
    with torch.cuda.device(dev):
        fn = _lib.lib().dibr_b200_backward_bf16 if bf16 else _lib.lib().dibr_b200_backward
        st = fn(
            B, F, height, width, D, ptr(g_feat), ptr(g_soft), ptr(face_idx), ptr(wts), ptr(soft),
            ptr(fvi), ptr(ff), float(multiplier), float(eps), float(sigmainv), float(boxlen_m),
            int(knum), ptr(g_fvi), ptr(g_ff), ptr(ws), ws_bytes, int(flags), stream_ptr(dev))
    _lib.check(st, "dibr_b200_backward")


def backward(height, width, g_feat, g_soft, face_idx, wts, soft, fvi, ff, multiplier, eps,
             sigmainv, boxlen_m, knum, ws, bins_valid, feature_grad_hook=None, views=None, out=None):
    """Calls dibr_b200_backward; returns (grad_face_vertices_image, grad_face_features fp32).

    ``views=(v0, v1)`` restricts the call to those views of the batch (dibr_b200_backward_views: all
    tensors stay the full-batch ones, only rows v0..v1-1 of the gradients are written) and ``out=
    (g_fvi, g_ff)`` supplies the full-batch gradient buffers to write into - together they let a
    caller pipeline view chunks (kaolin_b200.multi_gpu.pipelined_backward_all_gather); being outputs,
    they are never copied and must be aligned (DIBR_B200_ALIGNMENT).

    ``feature_grad_hook`` (per call — there is no process-global state): called as
    ``hook(g_ff)`` between the two branches of a fused backward.  grad_face_features is
    final after the rasterize branch, so e.g. its all-gather can travel while the
    soft-mask branch runs (kaolin_b200.multi_gpu.OverlappedGradAllGather)."""
    g_feat, g_soft, face_idx, wts, soft, fvi, ff = map(aligned, (g_feat, g_soft, face_idx, wts, soft, fvi, ff))
    dev = fvi.device
    B, F = fvi.shape[0], fvi.shape[1]
    D = 0 if ff is None else ff.shape[-1]
    if B * F == 0 and out is None:       # empty mesh: empty gradients, nothing to launch
        return torch.zeros_like(fvi), (torch.zeros(ff.shape, dtype=torch.float32, device=dev) if ff is not None else None)
    if out is not None:
        g_fvi, g_ff = out
    else:
        g_fvi = torch.empty_like(fvi)
        # grad_face_features is accumulated (atomics) in fp32 whatever the storage type
        g_ff = torch.empty(ff.shape, dtype=torch.float32, device=dev) if ff is not None else None
    # The workspace carries forward's bins / hit cache (soft-mask branch, bins_valid) and the
    # per-face records of the row-walk rasterize backward; without forward state a fresh
    # minimum-size one serves both.
    if ws is None:
        ws = workspace(B, B * F, height, width, dev)
        bins_valid = False
    ws_bytes = ws.numel()
    flags = _lib.BINS_VALID if bins_valid else 0
    hook = feature_grad_hook
    if hook is not None and g_feat is not None and g_soft is not None and D > 0:
        # two calls: rasterize branch (g_ff final -> hook), then the soft-mask branch added on top
        _backward_call(B, F, height, width, D, g_feat, None, face_idx, wts, None, fvi, ff, multiplier, eps,
                       sigmainv, boxlen_m, knum, g_fvi, g_ff, ws, ws_bytes, 0, dev, views)
        hook(g_ff)
        _backward_call(B, F, height, width, D, None, g_soft, face_idx, wts, soft, fvi, ff, multiplier, eps,
                       sigmainv, boxlen_m, knum, g_fvi, None, ws, ws_bytes, flags | _lib.ACCUMULATE, dev, views)
    else:
        _backward_call(B, F, height, width, D, g_feat, g_soft, face_idx, wts, soft, fvi, ff, multiplier, eps,
                       sigmainv, boxlen_m, knum, g_fvi, g_ff, ws, ws_bytes, flags, dev, views)
    return g_fvi, g_ff


# ---------------------------------------------------------------------------
# float64 instantiation (dibr_b200_forward_f64 / dibr_b200_backward_f64)
def forward_f64(mode, height, width, fvz, fvi, ff, fnz, valid_u8, multiplier, eps, sigmainv, boxlen_m, knum,
                face_idx_in=None):
    """-> (feat f64, face_idx, weights f64, soft f64, workspace); boxlen_m is a Python float (double)."""
    fvz, fvi, ff, fnz, valid_u8, face_idx_in = map(aligned, (fvz, fvi, ff, fnz, valid_u8, face_idx_in))
    dev = fvi.device
    B, F = fvi.shape[0], fvi.shape[1]
    D = 0 if ff is None else ff.shape[-1]
    raster = bool(mode & _lib.RASTER)
    soft_on = bool(mode & _lib.SOFT_MASK)
    f64 = torch.float64
    feat = torch.empty((B, height, width, D), dtype=f64, device=dev) if raster else None
    wts = torch.empty((B, height, width, 3), dtype=f64, device=dev) if raster else None
    idx = torch.empty((B, height, width), dtype=torch.int64, device=dev) if raster else face_idx_in
    soft = torch.empty((B, height, width), dtype=f64, device=dev) if soft_on else None
    if B == 0:
        return feat, idx, wts, soft, None
    n = _lib.lib().dibr_b200_workspace_bytes_f64(B, B * F, height, width)
    if n == 0:
        raise RuntimeError("kaolin_b200: unsupported problem size")
    ws = torch.empty(n, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        st = _lib.lib().dibr_b200_forward_f64(
            B, F, height, width, D, ptr(fvz), ptr(fvi), ptr(ff), ptr(fnz), ptr(valid_u8), float(multiplier),
            float(eps), mode, float(sigmainv), float(boxlen_m), int(knum), ptr(feat), ptr(idx), ptr(wts), ptr(soft),
            ptr(ws), ws.numel(), stream_ptr(dev))
    _lib.check(st, "dibr_b200_forward_f64")
    return feat, idx, wts, soft, ws


def backward_f64(height, width, g_feat, g_soft, face_idx, wts, soft, fvi, ff, multiplier, eps, sigmainv, boxlen_m,
                 knum, ws):
    g_feat, g_soft, face_idx, wts, soft, fvi, ff = map(aligned, (g_feat, g_soft, face_idx, wts, soft, fvi, ff))
    dev = fvi.device
    B, F = fvi.shape[0], fvi.shape[1]
    D = 0 if ff is None else ff.shape[-1]
    if B * F == 0:
        return torch.zeros_like(fvi), (torch.zeros_like(ff) if ff is not None else None)
    g_fvi = torch.empty_like(fvi)
    g_ff = torch.empty_like(ff) if ff is not None else None
    flags = _lib.BINS_VALID if ws is not None else 0
    if ws is None:
        ws = torch.empty(_lib.lib().dibr_b200_workspace_bytes_f64(B, B * F, height, width), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        st = _lib.lib().dibr_b200_backward_f64(
            B, F, height, width, D, ptr(g_feat), ptr(g_soft), ptr(face_idx), ptr(wts), ptr(soft), ptr(fvi), ptr(ff),
            float(multiplier), float(eps), float(sigmainv), float(boxlen_m), int(knum), ptr(g_fvi), ptr(g_ff),
            ptr(ws), ws.numel(), int(flags), stream_ptr(dev))
    _lib.check(st, "dibr_b200_backward_f64")
    return g_fvi, g_ff
