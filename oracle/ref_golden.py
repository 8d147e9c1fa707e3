"""TEST INFRASTRUCTURE — stored outputs of the reference's own CUDA kernels (tests/golden/ref_cuda.npz).

tests/golden/make_ref_cuda_golden.py runs oracle/_ref on the inputs of every test that compares with the
reference CUDA path and stores, per output of each case:

* ``sha``   — SHA-256 of the whole array (dtype, shape, bytes): outputs that must match bit for bit;
* ``idx`` / ``val`` — rows (pixels of an image, faces of a gradient): all of them when there are at most
  twice the sample size, else a sample seeded by the case and output name, three quarters of it drawn
  where the reference output is non-zero;
* ``scale`` — max |ref| over the whole array, so that sampled gradient errors are normalised exactly as
  the whole-array comparison normalised them;
* ``full``  — the whole array, for the few small outputs a test reads everywhere.

``shape``, ``sha`` and ``scale`` of every output travel together as one JSON member (``meta``).

The tests then compare against this file, so they need neither the reference nor oracle/_ref.
"""
import hashlib
import json
import os
import zlib

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_cuda.npz")
N_ROWS = {"image": 128, "grad": 64}      # sample size per output; the generator doubles it for some cases

_data = None


def _numpy(t):
    """torch tensor (any device, bf16 as its bit pattern) or array -> contiguous numpy array."""
    if hasattr(t, "detach"):
        import torch
        t = t.detach()
        if t.dtype == torch.bfloat16:
            t = t.view(torch.int16)
        t = t.cpu().numpy()
    return np.ascontiguousarray(t)


def digest(t):
    a = _numpy(t)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.data)
    return h.hexdigest()


# ---------------------------------------------------------------------------- generator side
def record(store, case, name, ref, kind=None, exact=False, full=False, scale_rows=1):
    """Add output ``name`` of ``case`` to ``store`` (a dict written by ``save``).  kind "image": sample the
    pixels of (B, H, W[, D]); "grad": the faces of (B, F, 3, k); None: no sample."""
    a = _numpy(ref)
    key = f"{case}/{name}"
    meta = store.setdefault("meta", {}).setdefault(key, {})
    meta["shape"] = list(a.shape)
    if exact:
        meta["sha"] = digest(a)
    if full:
        store[key + "/full"] = a.astype(np.int32) if a.dtype == np.int64 else a
    if kind is None:
        return
    lead = 3 if kind == "image" else 2
    rows = a.reshape(int(np.prod(a.shape[:lead])), -1)
    n = N_ROWS[kind] * scale_rows
    if rows.shape[0] <= 2 * n:
        idx = np.arange(rows.shape[0])
    else:
        rng = np.random.default_rng(zlib.crc32(key.encode()))
        nz = np.flatnonzero(np.any(rows != 0, axis=1))
        n_nz = min(3 * n // 4, nz.size)
        idx = np.unique(np.concatenate([nz[rng.choice(nz.size, n_nz, replace=False)],
                                        rng.choice(rows.shape[0], n - n_nz, replace=False)]))
    store[key + "/idx"] = idx.astype(np.int32)
    store[key + "/val"] = rows[idx]
    if a.dtype.kind == "f":
        meta["scale"] = float(np.abs(a).max()) if a.size else 0.0


def save(path, store):
    arrays = {k: v for k, v in store.items() if k != "meta"}
    np.savez_compressed(path, meta=np.array(json.dumps(store["meta"], sort_keys=True)), **arrays)


# ---------------------------------------------------------------------------- test side
def _load():
    global _data
    if _data is None:
        with np.load(PATH) as z:
            _data = {k: z[k] for k in z.files}
        _data["meta"] = json.loads(str(_data["meta"]))
    return _data


def get(case, name, field):
    d = _load()
    key = f"{case}/{name}"
    if field in ("shape", "sha", "scale"):
        value = d["meta"].get(key, {}).get(field)
    else:
        value = d.get(f"{key}/{field}")
    if value is None:
        raise KeyError(f"{key}/{field} is not in {PATH}; regenerate it with tests/golden/make_ref_cuda_golden.py")
    return value


def assert_equal(case, name, ours):
    """Bit-exact over the whole array."""
    assert tuple(_numpy(ours).shape) == tuple(get(case, name, "shape")), (case, name, "shape")
    assert digest(ours) == str(get(case, name, "sha")), (case, name, "differs from the reference")


def full(case, name):
    return get(case, name, "full")


def scale(case, name):
    return float(get(case, name, "scale"))


def sampled(case, name, ours):
    """(our rows, the reference's rows) at the stored sample, as numpy arrays of shape (n, row width)."""
    ref = get(case, name, "val")
    idx = get(case, name, "idx").astype(np.int64)
    assert tuple(ours.shape) == tuple(get(case, name, "shape")), (case, name, "shape")
    if hasattr(ours, "detach"):
        import torch
        rows = ours.detach().reshape(-1, ref.shape[1])
        mine = rows[torch.from_numpy(idx).to(rows.device)].float() if rows.dtype == torch.bfloat16 \
            else rows[torch.from_numpy(idx).to(rows.device)]
        return mine.cpu().numpy(), ref
    return np.asarray(ours).reshape(-1, ref.shape[1])[idx], ref


def max_abs_err(case, name, ours):
    mine, ref = sampled(case, name, ours)
    return float(np.abs(mine.astype(np.float64) - ref).max()) if ref.size else 0.0


def rel_err(case, name, ours):
    """max |ours - ref| over the sample / max |ref| over the whole array."""
    return max_abs_err(case, name, ours) / max(scale(case, name), 1e-300)


def assert_grad_close(case, name, ours, tol):
    """Max-normalised error <= tol AND element-wise allclose(rtol=tol, atol=tol * scale)."""
    mine, ref = sampled(case, name, ours)
    s = max(scale(case, name), 1e-30)
    e = float(np.abs(mine.astype(np.float64) - ref).max() / s) if ref.size else 0.0
    assert e <= tol, (case, name, e)
    assert np.allclose(mine, ref, rtol=tol, atol=tol * s), (case, name)
    return e
