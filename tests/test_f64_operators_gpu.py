"""The four DIB-R operators in float64 (``kaolin_b200._C.render.mesh`` and the INTEGRATION.md Option A
binding) against the reference's own <double> operator kernels, whose outputs on these inputs are stored
in tests/golden/ref_cuda_f64_ops.npz (tests/golden/make_ref_cuda_f64_ops_golden.py).

Inputs are perturbed off the fp32 grid (test_f64_gpu._scene), so a path that computed in fp32 and cast
back would fail.  Bars are those of tests/test_f64_gpu.py: face_idx and the K-list ids / dist types
identical, images and probabilities within 1e-12 / 1e-10 absolute, gradients within 1e-9 of their scale
(double atomics in both, in different orders)."""
import json
import os

import numpy as np
import pytest
import torch

from kaolin_b200 import _C as b200_C
from kaolin_b200 import _lib
from oracle import ref_cuda, ref_golden
from test_f64_gpu import D, _mask_iou, _scene

pytestmark = pytest.mark.gpu

DEV = "cuda"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cuda_f64_ops.npz")
OPS = b200_C.render.mesh
KNUMS = (5, 30, 40)          # truncation, the default, more than a warp


class Golden:
    """Reader of one golden file in the format oracle/ref_golden.py writes (record / save): whole-array
    digests, seeded row samples and each output's full-array max |ref|."""

    def __init__(self, path):
        self.path = path
        self._d = None

    def get(self, case, name, field):
        if self._d is None:
            with np.load(self.path) as z:
                self._d = {k: z[k] for k in z.files}
            self._d["meta"] = json.loads(str(self._d["meta"]))
        key = f"{case}/{name}"
        value = self._d["meta"].get(key, {}).get(field) if field in ("shape", "sha", "scale") \
            else self._d.get(f"{key}/{field}")
        if value is None:
            raise KeyError(f"{key}/{field} is not in {self.path}; regenerate it with "
                           "tests/golden/make_ref_cuda_f64_ops_golden.py")
        return value

    def assert_equal(self, case, name, ours):
        """Bit-exact over the whole array."""
        assert tuple(ours.shape) == tuple(self.get(case, name, "shape")), (case, name, "shape")
        assert ref_golden.digest(ours) == str(self.get(case, name, "sha")), (case, name, "differs from the reference")

    def max_abs_err(self, case, name, ours):
        """max |ours - ref| over the stored sample of rows."""
        ref = self.get(case, name, "val")
        idx = torch.from_numpy(self.get(case, name, "idx").astype(np.int64)).to(ours.device)
        assert tuple(ours.shape) == tuple(self.get(case, name, "shape")), (case, name, "shape")
        mine = ours.detach().reshape(-1, ref.shape[1])[idx].double().cpu().numpy()
        return float(np.abs(mine - ref).max()) if ref.size else 0.0

    def rel_err(self, case, name, ours):
        """max |ours - ref| over the sample / max |ref| over the whole array."""
        return self.max_abs_err(case, name, ours) / max(float(self.get(case, name, "scale")), 1e-300)


golden = Golden(GOLDEN)


def logic_inputs():
    """2 views, icosphere level 3, 96 x 128, D = 3."""
    fvz, fvi, fnz, ff = _scene(2, 3, 110)
    H, W = 96, 128
    gen = torch.Generator(device=DEV); gen.manual_seed(11)
    g_feat = torch.rand((2, H, W, 3), device=DEV, generator=gen, dtype=torch.float64)
    g_soft = torch.rand((2, H, W), device=DEV, generator=gen, dtype=torch.float64)
    return H, W, D(fvz), D(fvi), D(ff), D(fnz), g_feat, g_soft


def packed_inputs(shrink=False):
    """3 views at 67 x 93 with back faces culled (mesh sizes differ) and view 1 with every face invalid
    (first_idx repeats an entry).  shrink: a third of the faces get their tight box shrunk by 25 %."""
    fvz, fvi, fnz, ff = _scene(3, 3, 120)
    fnz[1] = -1.0
    H, W, m = 67, 93, 1000.
    valid = torch.from_numpy(fnz >= 0.).to(DEV)
    vidx = torch.where(valid)
    z, xy, f = D(fvz)[vidx], D(fvi)[vidx] * m, D(ff)[vidx]
    first = torch.zeros(4, dtype=torch.long, device=DEV)
    torch.cumsum(valid.sum(dim=1), dim=0, out=first[1:])
    bb = torch.cat((xy.min(dim=1)[0], xy.max(dim=1)[0]), dim=1)
    if shrink:
        lo, hi = bb[:, :2], bb[:, 2:]
        d = (hi - lo) * 0.125
        pick = (torch.arange(bb.shape[0], device=DEV) % 3 == 0).unsqueeze(1)
        bb = torch.where(pick, torch.cat((lo + d, hi - d), dim=1), bb)
    return H, W, z.contiguous(), xy.contiguous(), bb.contiguous(), f.contiguous(), first, m


def packed_forward(C, shrink=False):
    H, W, z, xy, bb, f, first, m = packed_inputs(shrink)
    out, sel, w = C.packed_rasterize_forward_cuda(H, W, z, xy, bb, f, first, m, 1e-8)
    return {"features": out, "selected_face_idx": sel, "weights": w}


def soft_inputs(C, per_face_margin=False, boxlen=0.02):
    """The logic scene's multiplied xy, face_idx (rasterized through C) and enlarged boxes; with
    per_face_margin each face's margin is boxlen * multiplier scaled by its own factor in [0.5, 2)."""
    H, W, fvz, fvi, ff, fnz, _, _ = logic_inputs()
    m = 1000.
    _, face_idx, _ = ref_cuda.rasterize_forward(H, W, fvz, fvi, ff, fnz >= 0., m, 1e-8, C=C)
    fvi_m = fvi * m
    margin = torch.full(fvi.shape[:2] + (1,), boxlen * m, device=DEV, dtype=torch.float64)
    if per_face_margin:
        gen = torch.Generator(device=DEV); gen.manual_seed(13)
        margin = margin * (0.5 + 1.5 * torch.rand(margin.shape, device=DEV, generator=gen, dtype=torch.float64))
    bb = torch.cat([fvi_m.min(dim=-2)[0] - margin, fvi_m.max(dim=-2)[0] + margin], dim=-1).contiguous()
    return face_idx, fvi_m, bb, m


def soft_forward(C, per_face_margin=False, boxlen=0.02, knum=30):
    face_idx, fvi_m, bb, m = soft_inputs(C, per_face_margin, boxlen)
    soft, prob, cidx, ctype = C.dibr_soft_mask_forward_cuda(fvi_m, bb, face_idx, 7000., knum, m)
    return {"face_idx": face_idx, "soft_mask": soft, "close_face_prob": prob, "close_face_idx": cidx,
            "close_face_dist_type": ctype}


def klist_backward(C, r, knum):
    _, fvi_m, _, m = soft_inputs(C, boxlen=0.2)
    gen = torch.Generator(device=DEV); gen.manual_seed(17 + knum)
    g = torch.rand(r["soft_mask"].shape, device=DEV, generator=gen, dtype=torch.float64)
    return C.dibr_soft_mask_backward_cuda(g, r["soft_mask"], r["face_idx"], r["close_face_prob"],
                                          r["close_face_idx"], r["close_face_dist_type"], fvi_m, 7000., m)


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


def test_reference_wrapper_logic_in_double():
    H, W, fvz, fvi, ff, fnz, g_feat, g_soft = logic_inputs()
    r = ref_cuda.dibr_forward_backward(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, C=OPS)
    for k in ("features", "weights", "soft_mask", "grad_fvi", "grad_ff"):
        assert r[k].dtype == torch.float64, k
    case = "logic"
    golden.assert_equal(case, "face_idx", r["face_idx"])
    assert (r["face_idx"] >= 0).any() and (r["soft_mask"] < 1).any()
    assert golden.max_abs_err(case, "features", r["features"]) <= 1e-12
    assert golden.max_abs_err(case, "weights", r["weights"]) <= 1e-12
    assert golden.max_abs_err(case, "soft_mask", r["soft_mask"]) <= 1e-10
    assert golden.rel_err(case, "grad_fvi", r["grad_fvi"]) <= 1e-9
    assert golden.rel_err(case, "grad_ff", r["grad_ff"]) <= 1e-9


def test_operators_equal_the_fused_double_api():
    from kaolin_b200.render.mesh import dibr_rasterization
    H, W, fvz, fvi, ff, fnz, g_feat, g_soft = logic_inputs()
    r = ref_cuda.dibr_forward_backward(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, C=OPS)
    t_fvi, t_ff = fvi.clone().requires_grad_(True), ff.clone().requires_grad_(True)
    feat, soft, idx = dibr_rasterization(H, W, fvz, t_fvi, t_ff, fnz)
    torch.autograd.backward([feat, soft], [g_feat, g_soft])
    assert torch.equal(idx, r["face_idx"]) and torch.equal(feat, r["features"]) and torch.equal(soft, r["soft_mask"])
    # the weights of the fused double entry point itself
    B, F = fvz.shape[:2]
    w = torch.empty((B, H, W, 3), dtype=torch.float64, device=DEV)
    out = torch.empty((B, H, W, 3), dtype=torch.float64, device=DEV)
    i64 = torch.empty((B, H, W), dtype=torch.int64, device=DEV)
    s64 = torch.empty((B, H, W), dtype=torch.float64, device=DEV)
    n = _lib.lib().dibr_b200_workspace_bytes_f64(B, B * F, H, W)
    ws = torch.empty(n, dtype=torch.uint8, device=DEV)
    p = lambda t: t.data_ptr()
    st = _lib.lib().dibr_b200_forward_f64(B, F, H, W, 3, p(fvz), p(fvi), p(ff), p(fnz), None, 1000., 1e-8,
                                          _lib.RASTER | _lib.SOFT_MASK, 7000., 0.02 * 1000., 30, p(out), p(i64),
                                          p(w), p(s64), p(ws), n, torch.cuda.current_stream().cuda_stream)
    _lib.check(st, "dibr_b200_forward_f64")
    assert torch.equal(w, r["weights"]) and torch.equal(out, r["features"])
    assert _rel(r["grad_fvi"], t_fvi.grad) <= 1e-12 and _rel(r["grad_ff"], t_ff.grad) <= 1e-12


def test_packed_ragged_batch():
    _, _, _, _, _, _, first, _ = packed_inputs()
    assert first[1] == first[2] and first[1] > 0
    r = packed_forward(OPS)
    golden.assert_equal("packed", "selected_face_idx", r["selected_face_idx"])
    assert (r["selected_face_idx"][1] == -1).all() and (r["selected_face_idx"][2] >= 0).any()
    assert golden.max_abs_err("packed", "features", r["features"]) <= 1e-12
    assert golden.max_abs_err("packed", "weights", r["weights"]) <= 1e-12


def test_caller_bboxes_are_honoured():
    shrunk = packed_forward(OPS, shrink=True)
    golden.assert_equal("packed_shrunk", "selected_face_idx", shrunk["selected_face_idx"])
    assert golden.max_abs_err("packed_shrunk", "features", shrunk["features"]) <= 1e-12
    assert golden.max_abs_err("packed_shrunk", "weights", shrunk["weights"]) <= 1e-12
    minmax = packed_forward(OPS)
    changed = int((shrunk["selected_face_idx"] != minmax["selected_face_idx"]).sum())
    print(f"\n[f64 ops] pixels whose face changes with the shrunk boxes: {changed}")
    assert changed > 0

    r = soft_forward(OPS, per_face_margin=True)
    golden.assert_equal("soft_margin", "face_idx", r["face_idx"])
    for k in ("close_face_idx", "close_face_dist_type"):
        golden.assert_equal("soft_margin", k, r[k])
    assert golden.max_abs_err("soft_margin", "close_face_prob", r["close_face_prob"]) <= 1e-12
    assert golden.max_abs_err("soft_margin", "soft_mask", r["soft_mask"]) <= 1e-10
    uniform = soft_forward(OPS)
    changed = int((r["soft_mask"] != uniform["soft_mask"]).sum())
    print(f"[f64 ops] pixels whose soft mask changes with per-face margins: {changed}")
    assert changed > 0


@pytest.mark.parametrize("knum", KNUMS)
def test_k_lists(knum):
    r = soft_forward(OPS, boxlen=0.2, knum=knum)
    case = f"klists/{knum}"
    golden.assert_equal(case, "face_idx", r["face_idx"])
    for k in ("close_face_idx", "close_face_dist_type"):
        golden.assert_equal(case, k, r[k])
    assert r["close_face_prob"].dtype == torch.float64
    filled = (r["close_face_idx"] >= 0).sum(dim=-1)
    if knum < 40:
        assert int(filled.max()) == knum          # boxlen 0.2: some lists are full
    assert golden.max_abs_err(case, "close_face_prob", r["close_face_prob"]) <= 1e-12
    assert golden.max_abs_err(case, "soft_mask", r["soft_mask"]) <= 1e-10
    g = klist_backward(OPS, r, knum)
    assert g.dtype == torch.float64
    assert golden.rel_err(case, "grad_fvi", g) <= 1e-9


@pytest.mark.parametrize("sigmainv,boxlen", [(7000, 0.02), (70, 0.2)])
def test_reference_fixtures_through_the_operators(golden_dir, sigmainv, boxlen):
    g = np.load(os.path.join(golden_dir, "dibr_simple.npz"))
    key = f"s{sigmainv}_b{boxlen}_"
    fvi = D(g["fvi"])
    face_idx = torch.from_numpy(g["face_idx"].astype(np.int64)).to(DEV)
    m = 1000.
    fvi_m = fvi * m
    bb = torch.cat([fvi_m.min(dim=-2)[0] - boxlen * m, fvi_m.max(dim=-2)[0] + boxlen * m], dim=-1).contiguous()
    soft, prob, cidx, ctype = OPS.dibr_soft_mask_forward_cuda(fvi_m.detach().contiguous(), bb.detach(), face_idx,
                                                              float(sigmainv), 30, m)
    assert torch.equal(cidx.cpu(), torch.from_numpy(g[key + "close_face_idx"].astype(np.int64)))
    assert torch.equal(ctype.cpu(), torch.from_numpy(g[key + "close_face_dist_type"]))
    assert float((prob.cpu() - torch.from_numpy(g[key + "close_face_prob"]).double()).abs().max()) <= 1e-4
    assert float((soft.cpu() - torch.from_numpy(g[key + "soft_mask"]).double()).abs().max()) <= 1e-4
    s_req = soft.clone().requires_grad_(True)
    _mask_iou(s_req, face_idx).backward()
    g_m = OPS.dibr_soft_mask_backward_cuda(s_req.grad.contiguous(), soft, face_idx, prob, cidx, ctype,
                                           fvi_m.detach().contiguous(), float(sigmainv), m)
    gt = torch.from_numpy(g[key + "grad_fvi"]).double()          # (the kernel's gradient is wrt the unscaled xy)
    assert torch.allclose(g_m.cpu(), gt, rtol=1e-4, atol=1e-4)


def _binding():
    from integration import build_binding
    m = build_binding.load()
    assert m is not None, "integration/_build/kaolin_b200_binding.so is missing: run __graft_entry__.build()"
    return m


def test_option_a_binding_in_double():
    m = _binding()
    H, W, fvz, fvi, ff, fnz, g_feat, g_soft = logic_inputs()
    a = ref_cuda.dibr_forward_backward(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, C=m)
    b = ref_cuda.dibr_forward_backward(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, C=OPS)
    for k in ("face_idx", "features", "weights", "soft_mask"):
        assert torch.equal(a[k], b[k]), k
    assert a["features"].dtype == torch.float64
    assert _rel(a["grad_fvi"], b["grad_fvi"]) <= 1e-12 and _rel(a["grad_ff"], b["grad_ff"]) <= 1e-12
    golden.assert_equal("logic", "face_idx", a["face_idx"])


def test_mixed_and_unsupported_dtypes_are_refused():
    m = _binding()
    H, W, z, xy, bb, f, first, mult = packed_inputs()
    for C in (OPS, m):
        with pytest.raises(RuntimeError):
            C.packed_rasterize_forward_cuda(H, W, z, xy.float(), bb, f, first, mult, 1e-8)
        with pytest.raises(RuntimeError):
            C.packed_rasterize_forward_cuda(H, W, z.float(), xy, bb.float(), f.float(), first, mult, 1e-8)
    face_idx, fvi_m, sbb, _ = soft_inputs(OPS)
    for C in (OPS, m):
        with pytest.raises(RuntimeError):
            C.dibr_soft_mask_forward_cuda(fvi_m, sbb.float(), face_idx, 7000., 30, 1000.)
    with pytest.raises(RuntimeError, match="not implemented for 'Half'"):
        m.packed_rasterize_forward_cuda(H, W, z.half(), xy.half(), bb.half(), f.half(), first, mult, 1e-8)
    with pytest.raises(RuntimeError, match="not implemented for 'Half'"):
        m.dibr_soft_mask_forward_cuda(fvi_m.half(), sbb.half(), face_idx, 7000., 30, 1000.)
