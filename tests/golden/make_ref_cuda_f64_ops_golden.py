"""Writes tests/golden/ref_cuda_f64_ops.npz: the outputs of the reference's <double> operator kernels
(oracle/_ref, built by oracle/build_ref.py) on the inputs of tests/test_f64_operators_gpu.py.  Needs a
CUDA device and oracle/_ref; the tests themselves need neither.

    python tests/golden/make_ref_cuda_f64_ops_golden.py [OUT.npz]

Inputs come from the test file's own input functions.  Every case keeps B*H*W >= 512: the reference's
rasterize backward launches B*H*W/512 blocks, rounded down.  What is kept of each output is described
in oracle/ref_golden.py; tests/test_f64_operators_gpu.py reads it with its own loader.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import ref_cuda, ref_golden  # noqa: E402
import test_f64_operators_gpu as t  # noqa: E402


def put(store, case, r, exact=(), names=()):
    for name in exact:
        ref_golden.record(store, case, name, r[name], exact=True)
    for name in names:
        ref_golden.record(store, case, name, r[name], "grad" if name.startswith("grad") else "image")
    print(case, flush=True)


def main(out):
    assert ref_cuda.available(), "oracle/_ref/kaolin_ref_C.so is missing: run oracle/build_ref.py first"
    ref = ref_cuda.module()
    store = {}
    put(store, "logic", ref_cuda.dibr_forward_backward(*t.logic_inputs()), exact=("face_idx",),
        names=("features", "weights", "soft_mask", "grad_fvi", "grad_ff"))
    for case, shrink in (("packed", False), ("packed_shrunk", True)):
        put(store, case, t.packed_forward(ref, shrink), exact=("selected_face_idx",), names=("features", "weights"))
    lists = ("face_idx", "close_face_idx", "close_face_dist_type")
    put(store, "soft_margin", t.soft_forward(ref, per_face_margin=True), exact=lists,
        names=("close_face_prob", "soft_mask"))
    for knum in t.KNUMS:
        r = t.soft_forward(ref, boxlen=0.2, knum=knum)
        r["grad_fvi"] = t.klist_backward(ref, r, knum)
        put(store, f"klists/{knum}", r, exact=lists, names=("close_face_prob", "soft_mask", "grad_fvi"))
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    ref_golden.save(out, store)
    print(f"wrote {out}: {os.path.getsize(out)} bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else t.GOLDEN)
