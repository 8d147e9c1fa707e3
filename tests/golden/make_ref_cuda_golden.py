"""Regenerates tests/golden/ref_cuda.npz: the outputs of the reference's own CUDA kernels (oracle/_ref, built
by oracle/build_ref.py) on the inputs of every test that compares with them.  Needs a CUDA device and
oracle/_ref; the tests themselves need neither.

    python tests/golden/make_ref_cuda_golden.py [OUT.npz]

Inputs come from the tests' own input functions, so a case here and its test see the same tensors.
What is kept of each output is described in oracle/ref_golden.py.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import ref_cuda, ref_golden  # noqa: E402
import test_f64_gpu  # noqa: E402
import test_fullsize_gpu  # noqa: E402
import test_parity_gpu  # noqa: E402
import test_reference_wrappers  # noqa: E402

DEV = "cuda"


def put(store, case, r, exact=("face_idx",), full=(), names=("features", "soft_mask", "grad_fvi", "grad_ff"),
        scale_rows=1):
    """exact: digest only; full: the whole array; names: rows (a sample when large)."""
    for name in exact:
        ref_golden.record(store, case, name, r[name], exact=True)
    for name in full:
        ref_golden.record(store, case, name, r[name], full=True)
    for name in names:
        ref_golden.record(store, case, name, r[name], "grad" if name.startswith("grad") else "image",
                          scale_rows=scale_rows)
    print(case, flush=True)


def main(out):
    assert ref_cuda.available(), "oracle/_ref/kaolin_ref_C.so is missing: run oracle/build_ref.py first"
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    store = {}

    tp = test_parity_gpu
    for name in tp.SCENES:
        H, W, fvz, fvi, fnz, ff, g_feat, g_soft = tp.fused_inputs(name)
        put(store, "fused/" + name,
            ref_cuda.dibr_forward_backward(H, W, T(fvz), T(fvi), T(ff), T(fnz), T(g_feat), T(g_soft)))
    for name in tp.CONFIG_CASES:
        # the BASELINE sizes have no CPU-oracle test of their own: a larger sample
        put(store, "config/" + name, ref_cuda.dibr_forward_backward(*tp.config_inputs(name)), scale_rows=2)
        torch.cuda.empty_cache()
    for D in (3, 5):
        H, W, t_fvz, t_fvi, ff16, t_fnz, g_feat16, g_soft = tp.bf16_inputs(D)
        r = ref_cuda.dibr_forward_backward(H, W, t_fvz, t_fvi, ff16.float(), t_fnz, g_feat16.float(), g_soft)
        r["features_bf16"] = r["features"].to(torch.bfloat16)
        put(store, f"bf16/D{D}", r, exact=("face_idx", "soft_mask", "features_bf16"), names=("grad_fvi", "grad_ff"))

    tf = test_fullsize_gpu
    for name, (_, chunk) in tf.FULL.items():
        H, W, t_fvz, t_fvi, t_ff, t_fnz, g_feat, g_soft = tf.full_inputs(name)
        parts = []
        for c0 in range(0, t_fvz.shape[0], chunk):
            c1 = min(t_fvz.shape[0], c0 + chunk)
            r = ref_cuda.dibr_forward_backward(H, W, t_fvz[c0:c1], t_fvi[c0:c1], t_ff[c0:c1], t_fnz[c0:c1],
                                               g_feat[c0:c1].contiguous(), g_soft[c0:c1].contiguous(),
                                               tf.bench.SIGMAINV, tf.bench.BOXLEN, tf.bench.KNUM)
            parts.append({k: r[k].cpu() for k in ("face_idx", "features", "soft_mask", "grad_fvi", "grad_ff")})
            del r
            torch.cuda.empty_cache()
        put(store, "full/" + name, {k: torch.cat([p[k] for p in parts]) for k in parts[0]}, scale_rows=2)
        del parts, g_feat, g_soft
        torch.cuda.empty_cache()

    t64 = test_f64_gpu
    D64 = t64.D
    for case in t64.F64_CASES:
        H, W, fvz, fvi, fnz, ff, g_feat, g_soft = t64.f64_inputs(*case)
        put(store, "f64/" + "-".join(map(str, case)),
            ref_cuda.dibr_forward_backward(H, W, D64(fvz), D64(fvi), D64(ff), D64(fnz), g_feat, g_soft))
    H, W, fvz, fvi, fnz, ff = t64.alone_inputs()
    valid = torch.from_numpy(fnz >= 0.).to(DEV)
    r_feat, r_idx, r_w = ref_cuda.rasterize_forward(H, W, D64(fvz), D64(fvi), D64(ff), valid)
    gen = torch.Generator(device=DEV); gen.manual_seed(9)
    g = torch.rand(r_feat.shape, device=DEV, generator=gen, dtype=torch.float64)
    gxy, gff = ref_cuda.rasterize_backward(g, r_feat, r_idx, r_w, D64(fvi), D64(ff))
    r_soft, fvi_m, prob, cidx, ctype = ref_cuda.soft_mask_forward(D64(fvi), r_idx)
    gs = torch.rand(r_soft.shape, device=DEV, generator=gen, dtype=torch.float64)
    r_g = ref_cuda.soft_mask_backward(gs, r_soft, r_idx, prob, cidx, ctype, fvi_m)
    put(store, "f64/alone", {"face_idx": r_idx, "features": r_feat, "grad_fvi": gxy, "grad_ff": gff,
                             "soft_mask": r_soft, "grad_fvi_soft": r_g},
        names=("features", "grad_fvi", "grad_ff", "soft_mask", "grad_fvi_soft"))
    for fixture in ("dibr_simple", "dibr_sphere"):
        gz = np.load(os.path.join(HERE, fixture + ".npz"))
        fvi, fvz = D64(gz["fvi"]), D64(gz["fvz"])
        _, face_idx, _ = ref_cuda.rasterize_forward(35, 31, fvz, fvi, torch.zeros(tuple(fvz.shape) + (1,),
                                                                                  device=DEV, dtype=torch.float64))
        r_soft, fvi_m, prob, cidx, ctype = ref_cuda.soft_mask_forward(fvi, face_idx, 7000, 0.02, 30, 1000.)
        s_req = r_soft.clone().requires_grad_(True)
        t64._mask_iou(s_req, face_idx).backward()
        r_g = ref_cuda.soft_mask_backward(s_req.grad, r_soft, face_idx, prob, cidx, ctype, fvi_m, 7000, 1000.)
        put(store, "f64_fixture/" + fixture, {"soft_mask": r_soft, "grad_fvi": r_g}, exact=(),
            names=("soft_mask", "grad_fvi"))

    tw = test_reference_wrappers
    put(store, "wrappers/logic", ref_cuda.dibr_forward_backward(*tw.wrapper_inputs("logic")), names=("soft_mask",))
    put(store, "wrappers/f64_callers", ref_cuda.dibr_forward_backward(*tw.wrapper_inputs("f64_callers")),
        exact=(), full=("face_idx",), names=("features", "soft_mask", "grad_ff"))
    put(store, "wrappers/binding", ref_cuda.dibr_forward_backward(*tw.wrapper_inputs("binding")),
        names=("grad_fvi", "grad_ff"))

    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    ref_golden.save(out, store)
    print(f"wrote {out}: {os.path.getsize(out)} bytes, {len(store)} arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else ref_golden.PATH)
