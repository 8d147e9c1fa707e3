"""Regenerates tests/golden/reference_wrapper_calls.json from the reference (needs its source tree; see
oracle/ref_import.py).

The reference's own Python wrappers (rasterize, dibr_soft_mask, dibr_rasterization, deftet_sparse_render)
are imported in place with ``kaolin._C`` replaced by a recorder: every operator call they make is stored
as (operator name, positional arguments: tensor shape and dtype, or the Python scalar).
tests/test_reference_wrappers.py replays these calls against ``kaolin_b200._C``.
"""
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from kaolin_b200 import synthetic  # noqa: E402
from oracle import ref_import  # noqa: E402

OUT = os.path.join(HERE, "reference_wrapper_calls.json")


class _Stop(Exception):
    pass


class _Recorder:
    def __init__(self):
        self.calls = []
        self.render = self
        self.mesh = self

    def __getattr__(self, op):
        def call(*args, **kwargs):
            assert not kwargs, (op, kwargs)
            self.calls.append({"op": op, "args": [
                {"shape": list(a.shape), "dtype": str(a.dtype).replace("torch.", "")} if torch.is_tensor(a)
                else {"value": a} for a in args]})
            raise _Stop
        return call


def main():
    rec = _Recorder()
    ref_import.setup(rec)
    rast = ref_import.module("kaolin.render.mesh.rasterization")
    dibr = ref_import.module("kaolin.render.mesh.dibr")
    deftet = ref_import.module("kaolin.render.mesh.deftet")
    fvz, fvi, fnz = synthetic.icosphere_views(1, 1, seed=1)
    ff = synthetic.random_features(1, fvz.shape[1], 3, seed=2)
    t = torch.from_numpy
    for call in (lambda: rast.rasterize(32, 32, t(fvz), t(fvi), t(ff), backend="cuda"),
                 lambda: dibr.dibr_soft_mask(t(fvi), torch.full((1, 32, 32), -1, dtype=torch.long)),
                 lambda: dibr.dibr_rasterization(32, 32, t(fvz), t(fvi), t(ff), t(fnz)),
                 lambda: deftet.deftet_sparse_render(torch.zeros(1, 5, 2), torch.zeros(1, 5, 2), t(fvz), t(fvi),
                                                     t(ff), knum=4)):
        try:
            call()
        except _Stop:
            pass
        else:
            raise AssertionError("the wrapper returned without calling an operator")
    with open(OUT, "w") as f:
        json.dump(rec.calls, f, indent=1)
        f.write("\n")
    print(f"wrote {OUT}: {len(rec.calls)} calls")


if __name__ == "__main__":
    main()
