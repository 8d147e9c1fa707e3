"""Parity at the FULL BASELINE.json sizes against the reference's own CUDA kernels: the exact workload
bench.py times (c4_shard: 32 views x 20 480 faces x 1024^2, rank 0's seeds), configs[2] at B = 64 and
configs[4] at B = 8 views of the 1.3 M-triangle mesh.  The reference's outputs on these inputs are
stored in tests/golden/ref_cuda.npz (tests/golden/make_ref_cuda_golden.py; ~4.4 s per view at c5):
face_idx as a digest of the whole array, the rest at a fixed sample of pixels and faces.  Bars:
face_idx bit-exact; features / soft mask within 1e-5; gradients within 1e-5 of the reference CUDA
kernels (both sides accumulate with fp32 atomics)."""
import os
import sys

import pytest
import torch

from oracle import ref_golden
from kaolin_b200.render.mesh import dibr_rasterization

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402  (make_scene: the generator of the timed workload)

pytestmark = pytest.mark.gpu
DEV = "cuda"
GRAD_TOL = 1e-5     # north_star: "within 1e-5 fp32"


FULL = {
    # name: (bench workload, reference view chunk)
    "c4_shard_32x20480f_1024_as_timed": ("c4_shard", 8),
    "c3_full_64x20480f_512": ("c3", 16),
    "c5_full_8x1310720f_2048": ("c5", 2),
}


def full_inputs(name):
    B, F, H, W, D, fvz, fvi, fnz, ff = bench.make_scene(FULL[name][0], 0)
    T = lambda a: torch.from_numpy(a).to(DEV)
    gen = torch.Generator(device=DEV); gen.manual_seed(4321)
    g_feat = torch.rand((B, H, W, D), device=DEV, generator=gen)
    g_soft = torch.rand((B, H, W), device=DEV, generator=gen)
    return H, W, T(fvz), T(fvi), T(ff), T(fnz), g_feat, g_soft


@pytest.mark.parametrize("name", list(FULL))
def test_full_size_vs_reference_cuda(name):
    H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft = full_inputs(name)
    t_fvi.requires_grad_(True); t_ff.requires_grad_(True)
    feat, soft, idx = dibr_rasterization(H, W, t_fvz, t_fvi, t_ff, t_fnz,
                                         bench.SIGMAINV, bench.BOXLEN, bench.KNUM)
    torch.autograd.backward([feat, soft], [g_feat, g_soft])
    cov = (idx >= 0).float().mean().item()
    assert 0.2 < cov < 0.9
    case = "full/" + name
    ref_golden.assert_equal(case, "face_idx", idx)
    mine, ref = ref_golden.sampled(case, "soft_mask", soft)
    worst = {"feat": ref_golden.max_abs_err(case, "features", feat),
             "soft": ref_golden.max_abs_err(case, "soft_mask", soft),
             "g_fvi": ref_golden.assert_grad_close(case, "grad_fvi", t_fvi.grad, GRAD_TOL),
             "g_ff": ref_golden.assert_grad_close(case, "grad_ff", t_ff.grad, GRAD_TOL),
             "soft_bit_equal": float((mine == ref).mean())}
    print(f"\n[{name}] covered {cov:.3f}; face_idx exact on all {idx.shape[0]} views; " +
          ", ".join(f"{k} {v:.3e}" for k, v in worst.items()) + " (sampled)")
    assert worst["feat"] <= 1e-5 and worst["soft"] <= 1e-5
    assert worst["soft_bit_equal"] > 0.9999
