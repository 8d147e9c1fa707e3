"""float64 instantiation (dibr_b200_forward_f64 / dibr_b200_backward_f64) against the reference's own
<double> kernels (outputs stored in tests/golden/ref_cuda.npz, AT_DISPATCH_FLOATING_TYPES at rasterization_cuda.cu:218/427,
dibr_soft_mask_cuda.cu:205/376; the reference parametrizes its tests over torch.double at
test_dibr.py:37 and test_rasterization.py:33).

Bars: face_idx identical (the depth test and the inside test are the same comparisons on the same
double values); interpolated features / weights / soft mask within 1e-12 / 1e-10 absolute; gradients
within 1e-9 of the gradient's scale (double atomics in both, in different orders)."""
import numpy as np
import pytest
import torch

from kaolin_b200 import synthetic
from oracle import ref_golden

pytestmark = pytest.mark.gpu

DEV = "cuda"


def D(a, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV).double()
    return t.requires_grad_(True) if grad else t


def _scene(views, level, seed, feat_dim=3):
    fvz, fvi, fnz = synthetic.icosphere_views(views, level, seed=seed)
    ff = synthetic.random_features(views, fvz.shape[1], feat_dim, seed=seed + 1)
    # perturb in double so that the inputs are not representable in fp32 (a cast path would show)
    rng = np.random.default_rng(seed + 2)
    j = lambda a: a.astype(np.float64) + rng.uniform(-1e-9, 1e-9, a.shape)
    return j(fvz), j(fvi), fnz.astype(np.float64), j(ff)


F64_CASES = [(2, 3, 96, 128, 3), (1, 2, 64, 64, 1), (3, 4, 160, 120, 5)]


def f64_inputs(views, level, H, W, feat_dim):
    fvz, fvi, fnz, ff = _scene(views, level, 50 + level, feat_dim)
    gen = torch.Generator(device=DEV); gen.manual_seed(7)
    g_feat = torch.rand((views, H, W, feat_dim), device=DEV, generator=gen, dtype=torch.float64)
    g_soft = torch.rand((views, H, W), device=DEV, generator=gen, dtype=torch.float64)
    return H, W, fvz, fvi, fnz, ff, g_feat, g_soft


@pytest.mark.parametrize("views,level,H,W,feat_dim", F64_CASES)
def test_dibr_rasterization_double_matches_reference_double(views, level, H, W, feat_dim):
    from kaolin_b200.render.mesh import dibr_rasterization
    H, W, fvz, fvi, fnz, ff, g_feat, g_soft = f64_inputs(views, level, H, W, feat_dim)
    t_fvi, t_ff = D(fvi, True), D(ff, True)
    feat, soft, idx = dibr_rasterization(H, W, D(fvz), t_fvi, t_ff, D(fnz))
    assert feat.dtype == torch.float64 and soft.dtype == torch.float64 and idx.dtype == torch.int64
    torch.autograd.backward([feat, soft], [g_feat, g_soft])
    case = f"f64/{views}-{level}-{H}-{W}-{feat_dim}"
    ref_golden.assert_equal(case, "face_idx", idx)
    assert (idx >= 0).any() and (soft > 0).any()
    e_feat = ref_golden.max_abs_err(case, "features", feat)
    e_soft = ref_golden.max_abs_err(case, "soft_mask", soft)
    e_gff, e_gxy = ref_golden.rel_err(case, "grad_ff", t_ff.grad), ref_golden.rel_err(case, "grad_fvi", t_fvi.grad)
    print(f"\n[f64 {views}x{H}x{W}] feat {e_feat:.2e} soft {e_soft:.2e} grad_ff {e_gff:.2e} grad_fvi {e_gxy:.2e} (sampled)")
    assert e_feat <= 1e-12
    assert e_soft <= 1e-10
    assert e_gff <= 1e-12
    assert e_gxy <= 1e-9
    # and this is not the fp32 path cast back: fp32 results differ from the double ones by ~1e-7
    f32, s32, _ = dibr_rasterization(H, W, D(fvz).float(), D(fvi).float(), D(ff).float(), D(fnz).float())
    assert float((f32.double() - feat).abs().max()) > 1e-9


def alone_inputs():
    fvz, fvi, fnz, ff = _scene(2, 3, 71)
    return 80, 112, fvz, fvi, fnz, ff


def test_rasterize_and_soft_mask_alone_in_double():
    from kaolin_b200.render.mesh import rasterize, dibr_soft_mask
    H, W, fvz, fvi, fnz, ff = alone_inputs()
    case = "f64/alone"
    valid = torch.from_numpy(fnz >= 0.).to(DEV)
    t_fvi, t_ff = D(fvi, True), D(ff, True)
    (fa, fb), idx = rasterize(H, W, D(fvz), t_fvi, [t_ff[..., :2], t_ff[..., 2:]], valid_faces=valid)
    feat = torch.cat([fa, fb], dim=-1)
    ref_golden.assert_equal(case, "face_idx", idx)
    assert ref_golden.max_abs_err(case, "features", feat) <= 1e-12
    gen = torch.Generator(device=DEV); gen.manual_seed(9)
    g = torch.rand(feat.shape, device=DEV, generator=gen, dtype=torch.float64)
    feat.backward(g)
    assert ref_golden.rel_err(case, "grad_ff", t_ff.grad) <= 1e-12
    assert ref_golden.rel_err(case, "grad_fvi", t_fvi.grad) <= 1e-9

    s_fvi = D(fvi, True)
    soft = dibr_soft_mask(s_fvi, idx, sigmainv=7000, boxlen=0.02, knum=30, multiplier=1000.)
    assert soft.dtype == torch.float64
    assert ref_golden.max_abs_err(case, "soft_mask", soft) <= 1e-10
    gs = torch.rand(soft.shape, device=DEV, generator=gen, dtype=torch.float64)
    soft.backward(gs)
    assert ref_golden.rel_err(case, "grad_fvi_soft", s_fvi.grad) <= 1e-9


def test_double_gradcheck_of_the_linear_branch():
    """interpolated features are linear in face_features: autograd.gradcheck in double is exact."""
    from kaolin_b200.render.mesh import rasterize
    fvz, fvi, fnz, ff = _scene(1, 1, 90, feat_dim=2)
    t_ff = D(ff, True)
    fn = lambda x: rasterize(24, 24, D(fvz), D(fvi), x)[0]
    assert torch.autograd.gradcheck(fn, (t_ff,), eps=1e-6, atol=1e-9, rtol=1e-7, nondet_tol=1e-12)


def test_double_soft_mask_gradient_by_central_differences():
    """dibr_soft_mask is smooth in the vertices away from the k-nearest cut: the analytic double
    gradient agrees with central differences of the double forward along a random direction."""
    from kaolin_b200.render.mesh import dibr_soft_mask, rasterize
    fvz, fvi, fnz, ff = _scene(1, 1, 95)
    H = W = 48
    _, idx = rasterize(H, W, D(fvz), D(fvi), D(ff))
    t = D(fvi, True)
    gen = torch.Generator(device=DEV); gen.manual_seed(3)
    wgt = torch.rand((1, H, W), device=DEV, generator=gen, dtype=torch.float64)
    knum = fvi.shape[1]                       # every face kept: no truncation discontinuity
    loss = (dibr_soft_mask(t, idx, 7000, 0.5, knum, 1000.) * wgt).sum()
    loss.backward()
    d = torch.randn(t.shape, device=DEV, generator=gen, dtype=torch.float64)
    h = 1e-7
    f = lambda x: float((dibr_soft_mask(x, idx, 7000, 0.5, knum, 1000.) * wgt).sum())
    num = (f(t.detach() + h * d) - f(t.detach() - h * d)) / (2 * h)
    ana = float((t.grad * d).sum())
    print(f"\n[f64 soft mask] directional derivative analytic {ana:.10e} numeric {num:.10e}")
    assert abs(num - ana) <= 1e-5 * max(abs(ana), 1e-12)


def test_double_edge_cases():
    from kaolin_b200.render.mesh import dibr_rasterization
    z = lambda *s: torch.zeros(s, device=DEV, dtype=torch.float64).requires_grad_(True)
    fvi = z(1, 0, 3, 2)
    feat, soft, idx = dibr_rasterization(16, 16, z(1, 0, 3), fvi, z(1, 0, 3, 2), z(1, 0))
    assert feat.shape == (1, 16, 16, 2) and (idx == -1).all() and (soft == 0).all() and (feat == 0).all()
    (feat.sum() + soft.sum()).backward()
    assert fvi.grad.shape == fvi.shape
    # all faces culled by the normals
    fvz, fvi, fnz, ff = _scene(1, 1, 97)
    feat, soft, idx = dibr_rasterization(16, 16, D(fvz), D(fvi), D(ff), -torch.ones_like(D(fnz)))
    assert (idx == -1).all() and (feat == 0).all()


def _mask_iou(soft, face_idx):
    """kaolin/metrics/render.py:18-41 with the shifted target of test_dibr.py:182-186."""
    mask = (face_idx != -1).to(soft.dtype)
    shifted = torch.nn.functional.pad(mask, (0, 5))[..., 5:]
    B = soft.shape[0]
    mul = soft * shifted
    add = soft + shifted
    up = torch.sum(mul.reshape(B, -1), dim=1)
    down = torch.sum((add - mul).reshape(B, -1), dim=1)
    return 1.0 - torch.mean(up / (down + 1e-10))


@pytest.mark.parametrize("fixture", ["dibr_simple", "dibr_sphere"])
def test_double_on_the_reference_fixtures(golden_dir, fixture):
    """The reference runs its fixture tests in torch.double too (test_dibr.py:37, 109-191, 309-394) against
    the SAME stored values: double results agree with the float goldens to the goldens' own rounding
    (1e-4 here), and with the reference's double kernels to 1e-10 / 1e-9."""
    import os
    from kaolin_b200.render.mesh import rasterize, dibr_soft_mask
    g = np.load(os.path.join(golden_dir, fixture + ".npz"))
    key = "s7000_b0.02_"
    H, W = 35, 31
    fvi, fvz = D(g["fvi"]), D(g["fvz"])
    ff = torch.zeros(tuple(fvz.shape) + (1,), device=DEV, dtype=torch.float64)
    _, face_idx = rasterize(H, W, fvz, fvi, ff)
    if "face_idx" in g.files:
        assert torch.equal(face_idx.cpu(), torch.from_numpy(g["face_idx"].astype(np.int64)))
    t = fvi.clone().requires_grad_(True)
    soft = dibr_soft_mask(t, face_idx, 7000, 0.02, 30, 1000)
    assert soft.dtype == torch.float64
    gt_soft = torch.from_numpy(g[key + "soft_mask"]).to(DEV).double()
    assert float((soft - gt_soft).abs().max()) <= 1e-4
    _mask_iou(soft, face_idx).backward()
    if fixture == "dibr_simple":           # (the sphere's stored gradient is only good to 1e-1, test_dibr.py:392)
        gt_grad = torch.from_numpy(g[key + "grad_fvi"]).to(DEV).double()
        assert torch.allclose(t.grad, gt_grad, rtol=1e-4, atol=1e-4)
    case = "f64_fixture/" + fixture
    assert ref_golden.max_abs_err(case, "soft_mask", soft) <= 1e-10
    assert ref_golden.rel_err(case, "grad_fvi", t.grad) <= 1e-9
