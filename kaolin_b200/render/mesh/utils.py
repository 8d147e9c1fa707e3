"""``prepare_vertices`` and ``texture_mapping`` — drop-ins for kaolin/render/mesh/utils.py:22-79
and :129-175, the steps immediately before and after the rasterizer in every DIB-R caller
(SURVEY.md §8f rank 1 and 2).  One sm_100a kernel each way (kaolin_b200/csrc/mesh_pipeline.cu)
instead of the reference's chain of PyTorch kernels and its (B,V,3)/(B,V,2) intermediates.
Same signatures, argument meaning and return structure; CUDA tensors only (no CPU path).
"""
import ctypes

import torch
from torch.autograd import Function

from ... import _lib
from . import _host

__all__ = ["prepare_vertices", "texture_mapping"]


def _proj3(camera_proj):
    """camera_proj (3,1) -> host array of 3 floats (one tiny D2H if it lives on the GPU, as the
    reference's broadcast would read it on the device)."""
    vals = [float(x) for x in camera_proj.detach().reshape(-1).tolist()]
    if len(vals) != 3:
        raise RuntimeError("prepare_vertices: camera_proj must be of shape (3, 1)")
    return (ctypes.c_float * 3)(*vals)


class PrepareVerticesB200(Function):
    @staticmethod
    def forward(ctx, vertices, faces, camera_proj, camera_rot, camera_trans, camera_transform):
        v = _host.aligned(vertices.contiguous())
        f = _host.aligned(faces.contiguous())
        B, V = v.shape[0], v.shape[1]
        F = f.shape[0]
        T = None if camera_transform is None else _host.aligned(camera_transform.contiguous())
        R = None if camera_rot is None else _host.aligned(camera_rot.contiguous())
        t = None if camera_trans is None else _host.aligned(camera_trans.reshape(B, 3).contiguous())
        proj = _proj3(camera_proj)
        fvc = torch.empty((B, F, 3, 3), dtype=torch.float32, device=v.device)
        fvi = torch.empty((B, F, 3, 2), dtype=torch.float32, device=v.device)
        fn = torch.empty((B, F, 3), dtype=torch.float32, device=v.device)
        with torch.cuda.device(v.device):
            st = _lib.lib().dibr_b200_prepare_vertices_forward(
                B, V, F, _host.ptr(v), _host.ptr(f), _host.ptr(T), _host.ptr(R), _host.ptr(t), proj,
                _host.ptr(fvc), _host.ptr(fvi), _host.ptr(fn), _host.stream_ptr(v.device))
        _lib.check(st, "dibr_b200_prepare_vertices_forward")
        ctx.save_for_backward(v, f, T, R, t)
        ctx.proj = proj
        return fvc, fvi, fn

    @staticmethod
    def backward(ctx, g_fvc, g_fvi, g_fn):
        v, f, T, R, t = ctx.saved_tensors
        B, V = v.shape[0], v.shape[1]
        F = f.shape[0]
        c = lambda g: None if g is None else _host.aligned(g.contiguous())
        g_fvc, g_fvi, g_fn = c(g_fvc), c(g_fvi), c(g_fn)
        g_vc = torch.empty((B, V, 3), dtype=torch.float32, device=v.device)
        with torch.cuda.device(v.device):
            st = _lib.lib().dibr_b200_prepare_vertices_backward(
                B, V, F, _host.ptr(v), _host.ptr(f), _host.ptr(T), _host.ptr(R), _host.ptr(t), ctx.proj,
                _host.ptr(g_fvc), _host.ptr(g_fvi), _host.ptr(g_fn), _host.ptr(g_vc),
                _host.stream_ptr(v.device))
        _lib.check(st, "dibr_b200_prepare_vertices_backward")
        # the camera map is linear: back through it with library GEMMs ((B,V,3) x (3,3))
        g_v = g_T = g_R = g_t = None
        if T is not None:
            if ctx.needs_input_grad[0]:
                g_v = g_vc @ T[:, :3, :].transpose(1, 2)
            if ctx.needs_input_grad[5]:
                g_T = torch.cat([v.transpose(1, 2) @ g_vc, g_vc.sum(dim=1, keepdim=True)], dim=1)
        else:
            g_d = g_vc @ R                        # vc = (p - t) @ R^T
            if ctx.needs_input_grad[0]:
                g_v = g_d
            if ctx.needs_input_grad[3]:
                g_R = g_vc.transpose(1, 2) @ (v - t.view(B, 1, 3))
            if ctx.needs_input_grad[4]:
                g_t = -g_d.sum(dim=1)
        return g_v, None, None, g_R, g_t, g_T


def prepare_vertices(vertices, faces, camera_proj, camera_rot=None, camera_trans=None,
                     camera_transform=None):
    r"""Move and project vertices to the cameras, then index them with faces
    (kaolin.render.mesh.utils.prepare_vertices, utils.py:129-175).

    Returns ``(face_vertices_camera (B,F,3,3), face_vertices_image (B,F,3,2), face_normals (B,F,3))``.
    Gradients flow to ``vertices`` and to the camera transform / rotation / translation;
    ``camera_proj`` is treated as a constant.
    """
    if camera_transform is None:
        assert camera_trans is not None and camera_rot is not None, \
            "camera_transform or camera_trans and camera_rot must be defined"
    else:
        assert camera_trans is None and camera_rot is None, \
            "camera_trans and camera_rot must be None when camera_transform is defined"
    _host.check_tensors("prepare_vertices", [("vertices", vertices), ("faces", faces),
                                             ("camera_rot", camera_rot), ("camera_trans", camera_trans),
                                             ("camera_transform", camera_transform)])
    if vertices.dim() != 3 or vertices.shape[-1] != 3:
        raise RuntimeError("prepare_vertices: vertices must be of shape (batch_size, num_vertices, 3)")
    if faces.dim() != 2 or faces.shape[-1] != 3 or faces.dtype != torch.int64:
        raise NotImplementedError("prepare_vertices: faces must be a LongTensor of shape (num_faces, 3) "
                                  "(triangle meshes)")
    B = vertices.shape[0]
    if camera_transform is not None:
        _host.check_size("prepare_vertices", "camera_transform", camera_transform, (B, 4, 3))
    else:
        _host.check_size("prepare_vertices", "camera_rot", camera_rot, (B, 3, 3))
        if camera_trans.numel() != B * 3:
            raise RuntimeError("prepare_vertices: camera_trans must hold (batch_size, 3) values")
    return PrepareVerticesB200.apply(vertices, faces, camera_proj, camera_rot, camera_trans, camera_transform)


class TextureMappingB200(Function):
    @staticmethod
    def forward(ctx, texture_coordinates, texture_maps, nearest):
        uv = _host.aligned(texture_coordinates.contiguous())
        tex = _host.aligned(texture_maps.contiguous())
        B, C, Ht, Wt = tex.shape
        N = uv.numel() // (2 * B)
        out = torch.empty((B, N, C), dtype=torch.float32, device=uv.device)
        with torch.cuda.device(uv.device):
            st = _lib.lib().dibr_b200_texture_mapping_forward(
                B, N, C, Ht, Wt, _host.ptr(uv), _host.ptr(tex), int(nearest), _host.ptr(out),
                _host.stream_ptr(uv.device))
        _lib.check(st, "dibr_b200_texture_mapping_forward")
        ctx.save_for_backward(uv, tex)
        ctx.nearest = int(nearest)
        return out

    @staticmethod
    def backward(ctx, g_out):
        uv, tex = ctx.saved_tensors
        B, C, Ht, Wt = tex.shape
        N = uv.numel() // (2 * B)
        g_tex = torch.empty_like(tex) if ctx.needs_input_grad[1] else None
        g_uv = torch.empty_like(uv) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(uv.device):
            st = _lib.lib().dibr_b200_texture_mapping_backward(
                B, N, C, Ht, Wt, _host.ptr(uv), _host.ptr(tex), ctx.nearest, _host.ptr(_host.aligned(g_out.contiguous())),
                _host.ptr(g_tex), _host.ptr(g_uv), _host.stream_ptr(uv.device))
        _lib.check(st, "dibr_b200_texture_mapping_backward")
        return g_uv, g_tex, None


def texture_mapping(texture_coordinates, texture_maps, mode='nearest'):
    r"""Interpolates ``texture_maps`` (B,C,h',w') at dense (B,h,w,2) or sparse (B,N,2) OpenGL texture
    coordinates in [0,1] (kaolin.render.mesh.utils.texture_mapping, utils.py:22-79): clamp,
    y flip, ``grid_sample(align_corners=False, padding_mode='border')``.  ``mode``: 'nearest'
    or 'bilinear'.  Returns (B,h,w,C) or (B,N,C)."""
    if mode not in ('nearest', 'bilinear'):
        raise ValueError(f"texture_mapping: mode must be 'nearest' or 'bilinear', got '{mode}'")
    _host.check_tensors("texture_mapping", [("texture_coordinates", texture_coordinates),
                                            ("texture_maps", texture_maps)])
    if texture_maps.dim() != 4 or texture_coordinates.shape[-1] != 2 \
            or texture_coordinates.shape[0] != texture_maps.shape[0]:
        raise RuntimeError("texture_mapping: expected texture_coordinates (B,...,2) and texture_maps (B,C,h',w')")
    out = TextureMappingB200.apply(texture_coordinates, texture_maps, mode == 'nearest')
    return out.reshape(texture_coordinates.shape[0], *texture_coordinates.shape[1:-1], texture_maps.shape[1])
