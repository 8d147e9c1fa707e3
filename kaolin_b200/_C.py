"""``kaolin_b200._C.render.mesh`` — the four operators the reference registers in
kaolin/csrc/bindings.cpp:111-115, with identical names, argument order/meaning,
return structure and error behaviour, implemented by libdibr_b200.so.

This is what makes the library a drop-in *below* the reference's own Python
wrappers: ``kaolin.render.mesh.rasterization`` / ``.dibr`` run unmodified with
``kaolin._C`` replaced by this module (tests/test_reference_wrappers.py: arity / dispatch on CPU,
results on the GPU).
"""
import ctypes
import types

import torch

from . import _lib


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _aligned(*ts):
    """The tensors, each copied when its data pointer is not 16-byte aligned (include/dibr_b200.h:
    the C ABI rejects it; the reference's wrappers take contiguous views at any storage offset)."""
    from .render.mesh._host import aligned
    return [aligned(t) for t in ts]


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _scalar_type(func, t):
    """AT_DISPATCH_FLOATING_TYPES on the tensor the reference dispatches on (rasterization_cuda.cu:218/427,
    dibr_soft_mask_cuda.cu:205/376): float32 or float64."""
    if t.dtype not in (torch.float32, torch.float64):
        raise RuntimeError(f"\"{func}\" not implemented for '{str(t.dtype).replace('torch.', '')}' "
                           "(kaolin_b200 supports float32 and float64)")
    return t.dtype


def _check_all(func, named, float_dtype=torch.float32):
    """at::checkAllSameGPU + at::checkAllContiguous (rasterization.cpp:70-75); every floating tensor of the
    dispatch dtype, as the reference's data_ptr<scalar_t>() requires."""
    dev = None
    for name, t in named:
        if not t.is_cuda:
            raise RuntimeError(f"{func}: expected tensor for argument {name} to be on GPU "
                               "(kaolin_b200 has no CPU path)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"{func}: expected all tensors on the same GPU; {name} is on {t.device}")
        if not t.is_contiguous():
            raise RuntimeError(f"{func}: expected contiguous tensor for argument {name}")
        if t.is_floating_point() and t.dtype != float_dtype:
            if t.dtype in (torch.float32, torch.float64):
                raise RuntimeError(f"{func}: expected {name} to be {float_dtype}, got {t.dtype} "
                                   "(the reference's data_ptr<scalar_t>() refuses mixed float/double)")
            raise RuntimeError(f"\"{func}\" not implemented for '{str(t.dtype).replace('torch.', '')}' "
                               "(kaolin_b200 supports float32)")
    return dev


def _fp64_via_fp32(op):
    """The deftet operators serve double callers by casting: float64 inputs -> float32, the op,
    floating-point outputs -> float64 (fp32 rounding applies)."""
    import functools

    @functools.wraps(op)
    def wrapped(*args):
        if not any(isinstance(a, torch.Tensor) and a.dtype == torch.float64 for a in args):
            return op(*args)
        out = op(*[a.to(torch.float32) if isinstance(a, torch.Tensor) and a.dtype == torch.float64 else a
                   for a in args])
        cast = lambda t: t.to(torch.float64) if isinstance(t, torch.Tensor) and t.dtype == torch.float32 else t
        return [cast(t) for t in out] if isinstance(out, (list, tuple)) else cast(out)
    return wrapped


def _check_size(func, name, t, shape):
    if tuple(t.shape) != tuple(shape):
        raise RuntimeError(f"{func}: expected tensor of size {list(shape)} for argument {name}, "
                           f"got {list(t.shape)}")


def _workspace(batch, total_faces, height, width, dev, dtype=torch.float32):
    query = _lib.lib().dibr_b200_workspace_bytes_f64 if dtype == torch.float64 else _lib.lib().dibr_b200_workspace_bytes
    n = query(batch, total_faces, height, width)
    if n == 0:
        raise RuntimeError("kaolin_b200: unsupported problem size")
    return torch.empty(n, dtype=torch.uint8, device=dev)


def packed_rasterize_forward_cuda(height, width, face_vertices_z, face_vertices_image,
                                  face_bboxes, face_features, first_idx_face_per_mesh,
                                  multiplier, eps):
    """rasterization.cpp:49-104 -> [interpolated_features, selected_face_idx, output_weights]."""
    fn = "packed_rasterize_forward_cuda"
    dt = _scalar_type(fn, face_vertices_z)
    dev = _check_all(fn, [("face_vertices_z", face_vertices_z),
                          ("face_vertices_image", face_vertices_image),
                          ("face_bboxes", face_bboxes), ("face_features", face_features),
                          ("first_idx_face_per_mesh", first_idx_face_per_mesh)], dt)
    num_faces = face_vertices_z.shape[0]
    batch_size = first_idx_face_per_mesh.shape[0] - 1
    feat_dim = face_features.shape[2]
    _check_size(fn, "face_vertices_z", face_vertices_z, (num_faces, 3))
    _check_size(fn, "face_vertices_image", face_vertices_image, (num_faces, 3, 2))
    _check_size(fn, "face_bboxes", face_bboxes, (num_faces, 4))
    _check_size(fn, "face_features", face_features, (num_faces, 3, feat_dim))
    _check_size(fn, "first_idx_face_per_mesh", first_idx_face_per_mesh, (batch_size + 1,))
    if first_idx_face_per_mesh.dtype != torch.int64:
        raise RuntimeError(f"{fn}: first_idx_face_per_mesh must be a LongTensor")
    face_vertices_z, face_vertices_image, face_bboxes, face_features, first_idx_face_per_mesh = _aligned(
        face_vertices_z, face_vertices_image, face_bboxes, face_features, first_idx_face_per_mesh)
    idx = torch.empty((batch_size, height, width), dtype=torch.int64, device=dev)
    w = torch.empty((batch_size, height, width, 3), dtype=dt, device=dev)
    out = torch.empty((batch_size, height, width, feat_dim), dtype=dt, device=dev)
    ws = _workspace(batch_size, num_faces, height, width, dev, dt)
    op = _lib.lib().dibr_b200_packed_rasterize_forward_f64 if dt == torch.float64 else \
        _lib.lib().dibr_b200_packed_rasterize_forward
    with torch.cuda.device(dev):
        st = op(
            batch_size, num_faces, height, width, feat_dim, _ptr(face_vertices_z),
            _ptr(face_vertices_image), _ptr(face_bboxes), _ptr(face_features),
            _ptr(first_idx_face_per_mesh), float(multiplier), float(eps),
            _ptr(out), _ptr(idx), _ptr(w), _ptr(ws), ws.numel(), _stream(dev))
    _lib.check(st, fn)
    return [out, idx, w]


def rasterize_backward_cuda(grad_interpolated_features, interpolated_features, selected_face_idx,
                            output_weights, face_vertices_image, face_features, eps):
    """rasterization.cpp:106-168 -> [grad_face_vertices_image, grad_face_features]."""
    fn = "rasterize_backward_cuda"
    dt = _scalar_type(fn, grad_interpolated_features)
    dev = _check_all(fn, [("grad_interpolated_features", grad_interpolated_features),
                          ("interpolated_features", interpolated_features),
                          ("selected_face_idx", selected_face_idx),
                          ("output_weights", output_weights),
                          ("face_vertices_image", face_vertices_image),
                          ("face_features", face_features)], dt)
    B, H, W, D = grad_interpolated_features.shape
    F = face_vertices_image.shape[1]
    _check_size(fn, "interpolated_features", interpolated_features, (B, H, W, D))
    _check_size(fn, "selected_face_idx", selected_face_idx, (B, H, W))
    _check_size(fn, "output_weights", output_weights, (B, H, W, 3))
    _check_size(fn, "face_vertices_image", face_vertices_image, (B, F, 3, 2))
    _check_size(fn, "face_features", face_features, (B, F, 3, D))
    grad_interpolated_features, selected_face_idx, output_weights, face_vertices_image, face_features = _aligned(
        grad_interpolated_features, selected_face_idx, output_weights, face_vertices_image, face_features)
    g_xy = torch.empty_like(face_vertices_image)
    g_ff = torch.empty_like(face_features)
    op = _lib.lib().dibr_b200_rasterize_backward_f64 if dt == torch.float64 else _lib.lib().dibr_b200_rasterize_backward
    with torch.cuda.device(dev):
        st = op(
            B, F, H, W, D, _ptr(grad_interpolated_features), _ptr(selected_face_idx),
            _ptr(output_weights), _ptr(face_vertices_image), _ptr(face_features), float(eps),
            _ptr(g_xy), _ptr(g_ff), _stream(dev))
    _lib.check(st, fn)
    return [g_xy, g_ff]


def dibr_soft_mask_forward_cuda(face_vertices_image, face_large_bboxes, selected_face_idx,
                                sigmainv, knum, multiplier):
    """dibr_soft_mask.cpp:48-108 -> [soft_mask, close_face_prob, close_face_idx, close_face_dist_type]."""
    fn = "dibr_soft_mask_forward_cuda"
    dt = _scalar_type(fn, face_vertices_image)
    dev = _check_all(fn, [("face_vertices_image", face_vertices_image),
                          ("face_bboxes", face_large_bboxes),
                          ("selected_face_idx", selected_face_idx)], dt)
    B, F = face_vertices_image.shape[0], face_vertices_image.shape[1]
    H, W = selected_face_idx.shape[1], selected_face_idx.shape[2]
    _check_size(fn, "face_vertices_image", face_vertices_image, (B, F, 3, 2))
    _check_size(fn, "face_bboxes", face_large_bboxes, (B, F, 4))
    _check_size(fn, "selected_face_idx", selected_face_idx, (B, H, W))
    face_vertices_image, face_large_bboxes, selected_face_idx = _aligned(
        face_vertices_image, face_large_bboxes, selected_face_idx)
    soft = torch.empty((B, H, W), dtype=dt, device=dev)
    prob = torch.empty((B, H, W, knum), dtype=dt, device=dev)
    cidx = torch.empty((B, H, W, knum), dtype=torch.int64, device=dev)
    ctype = torch.empty((B, H, W, knum), dtype=torch.uint8, device=dev)
    ws = _workspace(B, B * F, H, W, dev, dt)
    op = _lib.lib().dibr_b200_soft_mask_forward_f64 if dt == torch.float64 else _lib.lib().dibr_b200_soft_mask_forward
    with torch.cuda.device(dev):
        st = op(
            B, F, H, W, int(knum), _ptr(face_vertices_image), _ptr(face_large_bboxes),
            _ptr(selected_face_idx), float(sigmainv), float(multiplier),
            _ptr(soft), _ptr(prob), _ptr(cidx), _ptr(ctype), _ptr(ws), ws.numel(), _stream(dev))
    _lib.check(st, fn)
    return [soft, prob, cidx, ctype]


def dibr_soft_mask_backward_cuda(grad_soft_mask, soft_mask, selected_face_idx, close_face_prob,
                                 close_face_idx, close_face_dist_type, face_vertices_image,
                                 sigmainv, multiplier):
    """dibr_soft_mask.cpp:110-183 -> grad_face_vertices_image."""
    fn = "dibr_soft_mask_backward_cuda"
    dt = _scalar_type(fn, face_vertices_image)
    dev = _check_all(fn, [("grad_soft_mask", grad_soft_mask), ("soft_mask", soft_mask),
                          ("close_face_idx", close_face_idx),
                          ("close_face_dist_type", close_face_dist_type),
                          ("close_face_prob", close_face_prob),
                          ("face_vertices_image", face_vertices_image)], dt)
    B, F = face_vertices_image.shape[0], face_vertices_image.shape[1]
    H, W = selected_face_idx.shape[1], selected_face_idx.shape[2]
    K = close_face_idx.shape[-1]
    _check_size(fn, "grad_soft_mask", grad_soft_mask, (B, H, W))
    _check_size(fn, "soft_mask", soft_mask, (B, H, W))
    _check_size(fn, "selected_face_idx", selected_face_idx, (B, H, W))
    _check_size(fn, "close_face_prob", close_face_prob, (B, H, W, K))
    _check_size(fn, "close_face_idx", close_face_idx, (B, H, W, K))
    _check_size(fn, "close_face_dist_type", close_face_dist_type, (B, H, W, K))
    _check_size(fn, "face_vertices_image", face_vertices_image, (B, F, 3, 2))
    grad_soft_mask, soft_mask, close_face_prob, close_face_idx, close_face_dist_type, face_vertices_image = _aligned(
        grad_soft_mask, soft_mask, close_face_prob, close_face_idx, close_face_dist_type, face_vertices_image)
    g = torch.empty_like(face_vertices_image)
    sel, = _aligned(selected_face_idx.contiguous())
    op = _lib.lib().dibr_b200_soft_mask_backward_f64 if dt == torch.float64 else _lib.lib().dibr_b200_soft_mask_backward
    with torch.cuda.device(dev):
        st = op(
            B, F, H, W, K, _ptr(grad_soft_mask), _ptr(soft_mask), _ptr(sel), _ptr(close_face_prob),
            _ptr(close_face_idx), _ptr(close_face_dist_type), _ptr(face_vertices_image),
            float(sigmainv), float(multiplier), _ptr(g), _stream(dev))
    _lib.check(st, fn)
    return g


@_fp64_via_fp32
def deftet_sparse_render_forward_cuda(face_vertices_z, face_vertices_image, face_bboxes, pixel_coords,
                                      pixel_depth_ranges, knum, eps):
    """deftet.cpp:48-113 -> [selected_face_idx, pixel_depths, w0_arr, w1_arr], each (B, P, knum)."""
    fn = "deftet_sparse_render_forward_cuda"
    dev = _check_all(fn, [("face_vertices_z", face_vertices_z), ("face_vertices_image", face_vertices_image),
                          ("face_bboxes", face_bboxes), ("pixel_coords", pixel_coords),
                          ("pixel_depth_ranges", pixel_depth_ranges)])
    B, F = face_vertices_z.shape[0], face_vertices_z.shape[1]
    P = pixel_coords.shape[1]
    _check_size(fn, "face_vertices_z", face_vertices_z, (B, F, 3))
    _check_size(fn, "face_vertices_image", face_vertices_image, (B, F, 3, 2))
    _check_size(fn, "face_bboxes", face_bboxes, (B, F, 4))
    _check_size(fn, "pixel_coords", pixel_coords, (B, P, 2))
    _check_size(fn, "pixel_depth_ranges", pixel_depth_ranges, (B, P, 2))
    face_vertices_z, face_vertices_image, face_bboxes, pixel_coords, pixel_depth_ranges = _aligned(
        face_vertices_z, face_vertices_image, face_bboxes, pixel_coords, pixel_depth_ranges)
    idx = torch.empty((B, P, knum), dtype=torch.int64, device=dev)
    depth = torch.empty((B, P, knum), dtype=torch.float32, device=dev)
    w0 = torch.empty((B, P, knum), dtype=torch.float32, device=dev)
    w1 = torch.empty((B, P, knum), dtype=torch.float32, device=dev)
    n = _lib.lib().dibr_b200_deftet_workspace_bytes(B, F)
    ws = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        st = _lib.lib().dibr_b200_deftet_sparse_render_forward(
            B, F, P, int(knum), _ptr(face_vertices_z), _ptr(face_vertices_image), _ptr(face_bboxes),
            _ptr(pixel_coords), _ptr(pixel_depth_ranges), float(eps), _ptr(idx), _ptr(depth), _ptr(w0), _ptr(w1),
            _ptr(ws), ws.numel(), _stream(dev))
    _lib.check(st, fn)
    return [idx, depth, w0, w1]


@_fp64_via_fp32
def deftet_sparse_render_backward_cuda(grad_interpolated_features, face_idx, weights, face_vertices_image,
                                       face_features, eps):
    """deftet.cpp:115-170 -> [grad_face_vertices_image, grad_face_features]."""
    fn = "deftet_sparse_render_backward_cuda"
    dev = _check_all(fn, [("grad_interpolated_features", grad_interpolated_features), ("face_idx", face_idx),
                          ("weights", weights), ("face_vertices_image", face_vertices_image),
                          ("face_features", face_features)])
    B, P, K, D = grad_interpolated_features.shape
    F = face_vertices_image.shape[1]
    _check_size(fn, "face_idx", face_idx, (B, P, K))
    _check_size(fn, "weights", weights, (B, P, K, 3))
    _check_size(fn, "face_vertices_image", face_vertices_image, (B, F, 3, 2))
    _check_size(fn, "face_features", face_features, (B, F, 3, D))
    grad_interpolated_features, face_idx, weights, face_vertices_image, face_features = _aligned(
        grad_interpolated_features, face_idx, weights, face_vertices_image, face_features)
    g_xy = torch.empty_like(face_vertices_image)
    g_ff = torch.empty_like(face_features)
    with torch.cuda.device(dev):
        st = _lib.lib().dibr_b200_deftet_sparse_render_backward(
            B, F, P, K, D, _ptr(grad_interpolated_features), _ptr(face_idx), _ptr(weights),
            _ptr(face_vertices_image), _ptr(face_features), float(eps), _ptr(g_xy), _ptr(g_ff), _stream(dev))
    _lib.check(st, fn)
    return [g_xy, g_ff]


# kaolin._C.render.mesh.<op> namespace, as bindings.cpp:42,111-115 lays it out
render = types.SimpleNamespace(mesh=types.SimpleNamespace(
    packed_rasterize_forward_cuda=packed_rasterize_forward_cuda,
    rasterize_backward_cuda=rasterize_backward_cuda,
    dibr_soft_mask_forward_cuda=dibr_soft_mask_forward_cuda,
    dibr_soft_mask_backward_cuda=dibr_soft_mask_backward_cuda,
    deftet_sparse_render_forward_cuda=deftet_sparse_render_forward_cuda,
    deftet_sparse_render_backward_cuda=deftet_sparse_render_backward_cuda,
))
