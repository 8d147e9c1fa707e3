"""INTEGRATION.md Option B, checked: the reference's OWN Python wrappers
(kaolin/render/mesh/rasterization.py, dibr.py) run on top of ``kaolin_b200._C``.

* CPU part: the operator calls the reference modules make when ``rasterize`` / ``dibr_soft_mask`` /
  ``dibr_rasterization`` / ``deftet_sparse_render`` run (recorded from the reference into
  tests/golden/reference_wrapper_calls.json) must reach the ctypes shim with the right arity and
  argument order, i.e. fail with the shim's "no CPU path" RuntimeError — not with a TypeError.
* GPU part (`-m gpu`): the torch restatement of those wrappers
  (oracle/ref_cuda.py, line-for-line rasterization.py:290-346 / dibr.py:31-72) driven with
  ``C = kaolin_b200._C.render.mesh`` must reproduce the fused public API: operator boundary and
  fused path agree bit-for-bit on images, and on gradients up to atomics order."""
import numpy as np
import pytest
import torch

from oracle import ref_golden
from kaolin_b200 import _C as b200_C
from kaolin_b200 import synthetic


def test_reference_wrappers_reach_the_shim_with_the_right_arity(golden_dir):
    """Every operator call the reference's own wrappers make (rasterize, dibr_soft_mask, dibr_rasterization,
    deftet_sparse_render; recorded by tests/golden/make_wrapper_calls_golden.py) is accepted by the shim
    with that arity and those argument kinds and ends in its "no CPU path" error on CPU tensors."""
    import inspect
    import json
    import os
    with open(os.path.join(golden_dir, "reference_wrapper_calls.json")) as f:
        calls = json.load(f)
    assert {c["op"] for c in calls} == {"packed_rasterize_forward_cuda", "dibr_soft_mask_forward_cuda",
                                        "deftet_sparse_render_forward_cuda"}
    for c in calls:
        args = [torch.zeros(a["shape"], dtype=getattr(torch, a["dtype"])) if "shape" in a else a["value"]
                for a in c["args"]]
        with pytest.raises(RuntimeError, match="GPU|CUDA|no CPU path"):
            getattr(b200_C.render.mesh, c["op"])(*args)
    assert len(inspect.signature(b200_C.render.mesh.deftet_sparse_render_forward_cuda).parameters) == 7
    assert len(inspect.signature(b200_C.render.mesh.deftet_sparse_render_backward_cuda).parameters) == 6
    # backward operators: arity of the shim == arity of the reference's call sites
    sig = lambda f: len(inspect.signature(f).parameters)
    assert sig(b200_C.render.mesh.packed_rasterize_forward_cuda) == 9      # rasterization.py:329-339
    assert sig(b200_C.render.mesh.rasterize_backward_cuda) == 7            # rasterization.py:360-368
    assert sig(b200_C.render.mesh.dibr_soft_mask_forward_cuda) == 6        # dibr.py:40-48
    assert sig(b200_C.render.mesh.dibr_soft_mask_backward_cuda) == 9       # dibr.py:63-72


WRAPPER_CASES = {
    # name: (icosphere level, seed, H, W, dtype)
    "logic": (4, 21, 192, 160, torch.float32),
    "f64_callers": (3, 31, 96, 128, torch.float64),
    "binding": (4, 41, 160, 176, torch.float32),
}


def wrapper_inputs(name):
    level, seed, H, W, dt = WRAPPER_CASES[name]
    dev = "cuda"
    fvz, fvi, fnz = synthetic.icosphere_views(2, level, seed=seed)
    ff = synthetic.random_features(2, fvz.shape[1], 3, seed=seed + 1)
    T = lambda a: torch.from_numpy(a).to(dev).to(dt)
    gen = torch.Generator(device=dev); gen.manual_seed(seed + 2)
    g_feat = torch.rand((2, H, W, 3), device=dev, generator=gen, dtype=dt)
    g_soft = torch.rand((2, H, W), device=dev, generator=gen, dtype=dt)
    return H, W, T(fvz), T(fvi), T(ff), T(fnz), g_feat, g_soft


@pytest.mark.gpu
def test_wrapper_logic_on_b200_operators_equals_fused_api():
    from oracle import ref_cuda
    from kaolin_b200.render.mesh import dibr_rasterization
    H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft = wrapper_inputs("logic")
    r = ref_cuda.dibr_forward_backward(H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft, C=b200_C.render.mesh)
    t_fvi, t_ff = t_fvi.clone().requires_grad_(True), t_ff.clone().requires_grad_(True)
    feat, soft, idx = dibr_rasterization(H, W, t_fvz, t_fvi, t_ff, t_fnz)
    torch.autograd.backward([feat, soft], [g_feat, g_soft])
    assert torch.equal(idx, r["face_idx"]) and torch.equal(soft, r["soft_mask"]) and torch.equal(feat, r["features"])
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert rel(t_fvi.grad, r["grad_fvi"]) <= 1e-5 and rel(t_ff.grad, r["grad_ff"]) <= 1e-5
    # and both equal the reference's own operators
    ref_golden.assert_equal("wrappers/logic", "face_idx", r["face_idx"])
    assert ref_golden.max_abs_err("wrappers/logic", "soft_mask", r["soft_mask"]) <= 1e-5


@pytest.mark.gpu
def test_float64_operator_callers_are_served_in_fp32():
    """The reference dispatches double in its operators too (AT_DISPATCH_FLOATING_TYPES).  The public
    API has a real float64 instantiation (tests/test_f64_gpu.py); the packed ``_C`` OPERATOR shims serve
    double callers by casting (fp32 arithmetic, float64 outputs) - this pins that contract."""
    from oracle import ref_cuda
    H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft = wrapper_inputs("f64_callers")
    ours = ref_cuda.dibr_forward_backward(H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft, C=b200_C.render.mesh)
    for k in ("features", "weights", "soft_mask", "grad_fvi", "grad_ff"):
        assert ours[k].dtype == torch.float64, k
    assert ours["face_idx"].dtype == torch.int64
    # against the reference's <double> kernels: fp32-level agreement
    case = "wrappers/f64_callers"
    ref_idx = ref_golden.full(case, "face_idx").astype(np.int64)
    same = ours["face_idx"].cpu().numpy() == ref_idx
    agree = float(same.mean())
    print(f"\nfp64 operator callers: face_idx agreement with the reference's double kernels {agree:.6f}")
    assert agree >= 0.999
    for k in ("features", "soft_mask"):
        mine, ref = ref_golden.sampled(case, k, ours[k])
        at = same.reshape(-1)[ref_golden.get(case, k, "idx")]
        assert np.abs(mine - ref)[at].max() <= 1e-4, k
    assert ref_golden.rel_err(case, "grad_ff", ours["grad_ff"]) <= 1e-3


def _binding():
    """The binding build() made (a missing binding is an error, not a skip)."""
    from integration import build_binding
    m = build_binding.load()
    assert m is not None, "integration/_build/kaolin_b200_binding.so is missing: run __graft_entry__.build()"
    return m


def test_option_a_binding_loads_and_checks_like_the_reference():
    """INTEGRATION.md Option A compiled for real (integration/kaolin_binding.cpp): the pybind11 module
    exports the four operator names of bindings.cpp:111-115 and rejects CPU tensors through the same
    at::checkAllSameGPU the reference wrappers use (rasterization.cpp:70-72)."""
    m = _binding()
    for name in ("packed_rasterize_forward_cuda", "rasterize_backward_cuda", "dibr_soft_mask_forward_cuda",
                 "dibr_soft_mask_backward_cuda"):
        assert hasattr(m, name)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.packed_rasterize_forward_cuda(8, 8, torch.zeros(4, 3), torch.zeros(4, 3, 2), torch.zeros(4, 4),
                                        torch.zeros(4, 3, 2), torch.tensor([0, 4]), 1000., 1e-8)
    with pytest.raises(RuntimeError, match="expected it to be on GPU"):
        m.dibr_soft_mask_forward_cuda(torch.zeros(1, 4, 3, 2), torch.zeros(1, 4, 4),
                                      torch.zeros(1, 8, 8, dtype=torch.long), 7000., 30, 1000.)


@pytest.mark.gpu
def test_option_a_binding_results():
    """The reference's wrapper logic (oracle/ref_cuda.py) on top of the compiled Option A binding ==
    the same logic on top of the ctypes shim == the fused public API."""
    from oracle import ref_cuda
    m = _binding()
    H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft = wrapper_inputs("binding")
    a = ref_cuda.dibr_forward_backward(H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft, C=m)
    b = ref_cuda.dibr_forward_backward(H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft, C=b200_C.render.mesh)
    for k in ("face_idx", "soft_mask", "features", "weights"):
        assert torch.equal(a[k], b[k]), k
    rel = lambda x, y: float((x - y).abs().max() / y.abs().max())
    assert rel(a["grad_fvi"], b["grad_fvi"]) <= 1e-5 and rel(a["grad_ff"], b["grad_ff"]) <= 1e-5
    ref_golden.assert_equal("wrappers/binding", "face_idx", a["face_idx"])
    assert ref_golden.rel_err("wrappers/binding", "grad_fvi", a["grad_fvi"]) <= 1e-5
    assert ref_golden.rel_err("wrappers/binding", "grad_ff", a["grad_ff"]) <= 1e-5
