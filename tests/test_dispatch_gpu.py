"""One case per kernel variant the launcher selects (kaolin_b200/csrc/dibr_b200.cu), at the shapes
that select it, against the CPU oracle.

dibr_b200_forward / _backward pick a kernel per call from the feature dim, ``width % 4``, the
feature storage type, faces per 32x32 tile, the grid size, ``knum`` and the number of bin levels.
Every case asserts which kernels ran (from the library's per-thread launch trace, so the calls go
through ``_host`` directly: autograd runs CUDA backwards on a thread of its own) before it compares
values, so a change to the selection fails here instead of moving a case to another kernel.

Bars: face_idx exact; weights bit-equal to the oracle; fp32 features within 1e-6; bf16 features
bit-equal to the oracle's fp32 result on the bf16-rounded inputs rounded once to bf16; soft mask
within 1e-6; gradients within 3e-5 of their scale against the double-accumulating oracle.
"""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from kaolin_b200 import _lib, synthetic
from kaolin_b200 import _C as b200_C
from kaolin_b200.render.mesh import _host, dibr_rasterization, dibr_soft_mask, rasterize

pytestmark = pytest.mark.gpu
DEV = "cuda"
GRAD_REL = 3e-5
M, EPS, SIGMAINV, BOXLEN = 1000., 1e-8, 7000., 0.02

ROWS = ("raster_bwd_rows_kernel", "raster_bwd_finalize_kernel")
WARP = "raster_bwd_kernel"
TILE, FWD2 = "dibr_tile_fwd_kernel", "dibr_fwd2_kernel<S=2>"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().float().cpu().numpy() if t.dtype == torch.bfloat16 else t.detach().cpu().numpy()


def rel_err(a, ref):
    return float(np.abs(np.asarray(a, np.float64) - ref).max() / max(np.abs(ref).max(), 1e-30))


def bits_equal(a, b):
    return np.array_equal(np.ascontiguousarray(a, np.float32).view(np.uint32),
                          np.ascontiguousarray(b, np.float32).view(np.uint32))


def traced_step(H, W, fvz, fvi, ff, fnz, g_feat, g_soft, mode=3, knum=30, boxlen=BOXLEN):
    """_host.forward + _host.backward (bins and hit cache reused) -> (outputs, kernel names)."""
    _lib.trace_begin()
    try:
        feat, idx, wts, soft, ws = _host.forward(mode, H, W, fvz, fvi, ff, fnz, None, M, EPS, SIGMAINV,
                                                 boxlen * M, knum)
        g_fvi, g_ff = _host.backward(H, W, g_feat, g_soft if mode & _lib.SOFT_MASK else None, idx, wts, soft,
                                     fvi, ff, M, EPS, SIGMAINV, boxlen * M, knum, ws, True)
    finally:
        names = [n for n, _ in _lib.trace_end(1024)]
    return (feat, idx, wts, soft, g_fvi, g_ff), names


def assert_raster_bwd_kernel(names, D, W):
    if D <= 4 and W % 4 == 0:
        assert all(k in names for k in ROWS) and WARP not in names, names
    else:
        assert WARP in names and not any(k in names for k in ROWS), names


def check_feat(feat, o_feat, bf16):
    if bf16:
        want = torch.from_numpy(np.ascontiguousarray(o_feat)).to(torch.bfloat16)
        got = feat.cpu()
        bad = int((got.view(torch.int16) != want.view(torch.int16)).sum())
        assert bad == 0, f"{bad} bf16 features differ from the rounded oracle"
        return 0.0
    err = float(np.abs(N(feat) - o_feat).max()) if feat.numel() else 0.0
    assert err <= 1e-6, err
    return err


# ---------------------------------------------------------------------------
# Raster matrix: fp32 / bf16 x D 1..5 x (W % 4 == 0, W % 4 != 0) on small scenes, H % 32 != 0
SMALL = {
    "ico": lambda: synthetic.icosphere_views(2, 3, seed=41),
    "soup": lambda: synthetic.triangle_soup(2, 300, seed=42, coverage=3.0),
}
MATRIX = [(s, ft, D, W) for s in SMALL for ft in ("fp32", "bf16") for D in (1, 2, 3, 4, 5) for W in (96, 93)
          if not (ft == "fp32" and D == 3)]


@pytest.mark.parametrize("scene,ft,D,W", MATRIX)
def test_raster_matrix_vs_oracle(scene, ft, D, W):
    H = 72
    fvz, fvi, fnz = SMALL[scene]()
    B, F = fvz.shape[:2]
    bf16 = ft == "bf16"
    dt = torch.bfloat16 if bf16 else torch.float32
    ff_t = T(synthetic.random_features(B, F, D, seed=D)).to(dt)
    ff = N(ff_t)                                          # the bf16-rounded values the kernel sees
    rng = np.random.default_rng(100 + D)
    g_feat_t = T(rng.uniform(size=(B, H, W, D)).astype(np.float32)).to(dt)
    # forward with the soft mask; backward through the features only: the soft-mask branch does not
    # depend on D, W % 4 or the feature type (the full-size, size-ceiling and knum cases cover it)
    (feat, idx, wts, soft, g_fvi, g_ff), names = traced_step(H, W, T(fvz), T(fvi), ff_t, T(fnz), g_feat_t, None)
    assert TILE in names and FWD2 not in names, names
    assert_raster_bwd_kernel(names, D, W)
    assert feat.dtype == dt and g_ff.dtype == torch.float32

    o_feat, o_soft, o_idx, o_w = oracle.dibr_rasterization(H, W, fvz, fvi, ff, fnz, return_weights=True)
    assert (o_idx >= 0).mean() > 0.05
    assert np.array_equal(N(idx), o_idx)
    assert bits_equal(N(wts), o_w)
    e_feat = check_feat(feat, o_feat, bf16)
    np.testing.assert_allclose(N(soft), o_soft, rtol=0, atol=1e-6)
    o_gxy, o_gff = oracle.rasterize_backward(N(g_feat_t), o_idx, o_w, fvi, ff)
    e_xy, e_ff = rel_err(N(g_fvi), o_gxy), rel_err(N(g_ff), o_gff)
    print(f"\n[{scene} {ft} D={D} W={W}] feat {e_feat:.1e} grad_fvi {e_xy:.2e} grad_ff {e_ff:.2e}")
    assert e_xy <= GRAD_REL and e_ff <= GRAD_REL


# ---------------------------------------------------------------------------
# Full-size arms (dibr_fwd2_kernel<S=2>: <= 40 faces per 32x32 tile and >= 2048 such tiles in the
# batch), checked on row strips: the upstream gradients are zero outside the strips, so the strip
# oracle's gradients are the whole gradients.
FULL = {
    # name: (views, icosphere level, H, W, strips); H % 32 != 0 leaves a partial last band
    "2x1000x1024_20480f": (2, 5, 1000, 1024, [(24, 40), (492, 500), (992, 1000)]),
    "8x500x512_5120f": (8, 4, 500, 512, [(28, 36), (246, 250), (496, 500)]),
}


def zero_outside(t, strips):
    keep = torch.zeros(t.shape[1], dtype=torch.bool, device=t.device)
    for a, b in strips:
        keep[a:b] = True
    t[:, ~keep] = 0
    return t


def full_inputs(name, D, dt, seed=0):
    B, level, H, W, strips = FULL[name]
    fvz, fvi, fnz = synthetic.icosphere_views(B, level, seed=500 + seed)
    F = fvz.shape[1]
    ff_t = T(synthetic.random_features(B, F, D, seed=7)).to(dt)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(8)
    g_feat = zero_outside(torch.rand((B, H, W, D), device=DEV, generator=gen), strips).to(dt)
    g_soft = zero_outside(torch.rand((B, H, W), device=DEV, generator=gen), strips)
    return B, H, W, strips, fvz, fvi, fnz, ff_t, g_feat, g_soft


@pytest.mark.parametrize("name", list(FULL))
@pytest.mark.parametrize("ft,D,mode", [("fp32", 3, 3), ("fp32", 4, 3), ("bf16", 3, 3), ("bf16", 4, 3),
                                       ("bf16", 4, 1)])
def test_full_size_arms_on_strips(name, ft, D, mode):
    bf16 = ft == "bf16"
    B, H, W, strips, fvz, fvi, fnz, ff_t, g_feat, g_soft = full_inputs(name, D, torch.bfloat16 if bf16 else torch.float32)
    soft_on = bool(mode & _lib.SOFT_MASK)
    (feat, idx, wts, soft, g_fvi, g_ff), names = traced_step(H, W, T(fvz), T(fvi), ff_t, T(fnz), g_feat, g_soft, mode)
    assert FWD2 in names and TILE not in names, names
    assert_raster_bwd_kernel(names, D, W)
    assert ("soft_enum_kernel" in names) == soft_on, names

    ff = N(ff_t)
    rs = oracle.RowSample(H, W, fvz, fvi, ff, fnz, N(g_feat), N(g_soft), 0, 0, strips=strips,
                          sigmainv=SIGMAINV, boxlen=BOXLEN, knum=30, multiplier=M, eps=EPS)
    # each strip's backward overwrites the gradient arrays: sum them strip by strip
    want_xy, o_gff = 0., 0.
    for a, b in strips:
        rs.row0, rs.row1 = a, b
        r_xy, s_xy, r_ff = rs._run_strip()
        want_xy = want_xy + r_xy.astype(np.float64) + (s_xy if soft_on else 0.)
        o_gff = o_gff + r_ff.astype(np.float64)
    rows = np.concatenate([np.arange(a, b) for a, b in strips])
    assert np.array_equal(N(idx)[:, rows], rs.idx[:, rows])
    assert (rs.idx[:, rows] >= 0).any() and (rs.idx[:, rows] < 0).any()        # strips cross the silhouette
    assert bits_equal(N(wts)[:, rows], rs.w[:, rows])
    e_feat = check_feat(feat[:, torch.from_numpy(rows).to(DEV)], rs.out[:, rows], bf16)
    if soft_on:
        np.testing.assert_allclose(N(soft)[:, rows], rs.soft[:, rows], rtol=0, atol=1e-6)
    e_xy, e_ff = rel_err(N(g_fvi), want_xy), rel_err(N(g_ff), o_gff)
    print(f"\n[{name} {ft} D={D} mode={mode}] feat {e_feat:.1e} grad_fvi {e_xy:.2e} grad_ff {e_ff:.2e}")
    assert e_xy <= GRAD_REL and e_ff <= GRAD_REL


@pytest.mark.parametrize("ft", ["fp32", "bf16"])
def test_batch_equals_views_rendered_alone(ft):
    """View b of the 2-view batch (dibr_fwd2_kernel<S=2>) equals that view rendered alone (B = 1: the
    tile kernel): images bit-equal, gradients up to the order of float atomics."""
    dt = torch.bfloat16 if ft == "bf16" else torch.float32
    B, H, W, strips, fvz, fvi, fnz, ff_t, _, _ = full_inputs("2x1000x1024_20480f", 3, dt, seed=1)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(9)
    g_feat = torch.rand((B, H, W, 3), device=DEV, generator=gen).to(dt)
    g_soft = torch.rand((B, H, W), device=DEV, generator=gen)
    full, names = traced_step(H, W, T(fvz), T(fvi), ff_t, T(fnz), g_feat, g_soft)
    assert FWD2 in names and TILE not in names, names
    for b in range(B):
        one, names1 = traced_step(H, W, T(fvz[b:b + 1]), T(fvi[b:b + 1]), ff_t[b:b + 1].contiguous(),
                                  T(fnz[b:b + 1]), g_feat[b:b + 1].contiguous(), g_soft[b:b + 1].contiguous())
        assert TILE in names1 and FWD2 not in names1, names1
        for k in range(4):          # feat, face_idx, weights, soft mask
            assert torch.equal(full[k][b], one[k][0]), k
        e_xy = rel_err(N(full[4][b]), N(one[4][0]).astype(np.float64))
        e_ff = rel_err(N(full[5][b]), N(one[5][0]).astype(np.float64))
        print(f"\n[batch vs alone {ft} view {b}] grad_fvi {e_xy:.1e} grad_ff {e_ff:.1e}")
        assert e_xy <= 1e-6 and e_ff <= 1e-6


# ---------------------------------------------------------------------------
# Size ceiling: 16384 px per side (6 bin levels)
def ceiling_scene(B, D, level=3, seed=0):
    """Icosphere views plus faces larger than the image, with vertices off screen, behind the mesh."""
    fvz, fvi, fnz = synthetic.icosphere_views(B, level, seed=900 + seed)
    big_xy = np.array([[[-5.0, -5.0], [-5.0, 5.0], [-0.6, 0.3]],       # left wedge, taller than the image
                       [[-3.0, -1.1], [3.0, 1.2], [3.0, 1.19]],         # sliver across the whole image
                       [[2.0, 2.0], [3.0, 2.5], [2.5, 3.0]]], np.float32)  # entirely off screen
    big_z = np.full((3, 3), -20.0, np.float32)
    fvi = np.concatenate([fvi, np.broadcast_to(big_xy, (B,) + big_xy.shape)], 1)
    fvz = np.concatenate([fvz, np.broadcast_to(big_z, (B, 3, 3))], 1)
    fnz = np.concatenate([fnz, np.ones((B, 3), np.float32)], 1)
    ff = synthetic.random_features(B, fvz.shape[1], D, seed=seed)
    return np.ascontiguousarray(fvz), np.ascontiguousarray(fvi), np.ascontiguousarray(fnz), ff


def _shifted(a, row0, row_elems, ctype):
    """A pointer to where element 0 of the full image would be, for a buffer that holds the rows from
    row0 on: the oracle's row-range functions only touch the rows they are given."""
    return ctypes.cast(ctypes.c_void_p(a.ctypes.data - row0 * row_elems * a.itemsize), ctypes.POINTER(ctype))


def strip_oracle_one_view(H, W, fvz, fvi, ff, fnz, g_feat_rows, g_soft_rows, strips, knum=30):
    """DIB-R forward + backward of one view on row strips only, holding just the strips' rows."""
    L = oracle.lib()
    f32, i64, u8 = ctypes.c_float, ctypes.c_int64, ctypes.c_uint8
    ci, cf = ctypes.c_int, ctypes.c_float
    F, D = fvz.shape[1], ff.shape[-1]
    f_idx = np.nonzero(fnz[0] >= 0)[0]
    p_xy = np.ascontiguousarray(fvi[0, f_idx] * np.float32(M))
    p_z = np.ascontiguousarray(fvz[0, f_idx])
    p_ff = np.ascontiguousarray(ff[0, f_idx])
    p_bb = np.ascontiguousarray(np.concatenate([p_xy.min(1), p_xy.max(1)], 1))
    first = np.array([0, len(f_idx)], np.int64)
    fvi_m = np.ascontiguousarray(fvi * np.float32(M))
    bb_large = np.ascontiguousarray(oracle._large_bboxes(fvi_m, BOXLEN, M))
    P = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))
    out = {"idx": [], "w": [], "feat": [], "soft": []}
    gxy = np.zeros((1, F, 3, 2), np.float64)
    gff = np.zeros((1, F, 3, D), np.float64)
    k0 = 0
    for a, b in strips:
        n = b - a
        sel = np.empty((n, W), np.int64)
        w = np.empty((n, W, 3), np.float32)
        feat = np.empty((n, W, D), np.float32)
        L.oracle_rasterize_forward_rows(ci(1), ci(H), ci(W), ci(D), P(p_z, f32), P(p_xy, f32), P(p_bb, f32),
                                        P(p_ff, f32), P(first, i64), cf(M), cf(EPS), _shifted(sel, a, W, i64),
                                        _shifted(w, a, 3 * W, f32), _shifted(feat, a, D * W, f32), ci(a), ci(b))
        idx = np.where(sel >= 0, f_idx[np.maximum(sel, 0)], -1).astype(np.int64)
        soft = np.empty((n, W), np.float32)
        prob = np.empty((n, W, knum), np.float32)
        cidx = np.empty((n, W, knum), np.int64)
        ctype = np.empty((n, W, knum), np.uint8)
        L.oracle_soft_mask_forward_rows(ci(1), ci(H), ci(W), ci(F), ci(knum), P(fvi_m, f32), P(bb_large, f32),
                                        _shifted(idx, a, W, i64), cf(SIGMAINV), cf(M), _shifted(soft, a, W, f32),
                                        _shifted(prob, a, W * knum, f32), _shifted(cidx, a, W * knum, i64),
                                        _shifted(ctype, a, W * knum, u8), ci(a), ci(b))
        g = np.ascontiguousarray(g_feat_rows[k0:k0 + n])
        gs = np.ascontiguousarray(g_soft_rows[k0:k0 + n])
        k0 += n
        r_xy = np.empty((1, F, 3, 2), np.float32)
        r_ff = np.empty((1, F, 3, D), np.float32)
        L.oracle_rasterize_backward_rows(ci(1), ci(H), ci(W), ci(F), ci(D), _shifted(g, a, W * D, f32),
                                         _shifted(idx, a, W, i64), _shifted(w, a, 3 * W, f32), P(fvi, f32),
                                         P(ff, f32), cf(EPS), P(r_xy, f32), P(r_ff, f32), ci(a), ci(b))
        s_xy = np.empty((1, F, 3, 2), np.float32)
        L.oracle_soft_mask_backward_rows(ci(1), ci(H), ci(W), ci(F), ci(knum), _shifted(gs, a, W, f32),
                                         _shifted(soft, a, W, f32), _shifted(idx, a, W, i64),
                                         _shifted(prob, a, W * knum, f32), _shifted(cidx, a, W * knum, i64),
                                         _shifted(ctype, a, W * knum, u8), P(fvi_m, f32), cf(SIGMAINV), cf(M),
                                         P(s_xy, f32), ci(a), ci(b))
        gxy += r_xy.astype(np.float64) + s_xy
        gff += r_ff
        for k, v in (("idx", idx), ("w", w), ("feat", feat), ("soft", soft)):
            out[k].append(v)
    return {k: np.concatenate(v) for k, v in out.items()}, gxy, gff


CEILING_STRIPS = [(0, 16), (8184, 8200), (16376, 16384)]


@pytest.mark.parametrize("D", [3, 8])
def test_size_ceiling_16384_squared_on_strips(D):
    """1 x 16384^2: six bin levels.  D = 8 makes B*H*W*D = 2^31 feature elements (64-bit pixel
    offsets in every kernel that touches the features); its last rows are among the strips."""
    H = W = 16384
    need = H * W * (2 * 4 * D + 8 + 12 + 4 + 4) + (6 << 30)
    free = torch.cuda.mem_get_info()[0]
    print(f"\n[16384^2 D={D}] needs ~{need / 2**30:.1f} GiB of device memory, {free / 2**30:.1f} GiB free")
    if free < need:
        pytest.skip(f"needs ~{need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    fvz, fvi, fnz, ff = ceiling_scene(1, D)
    rows = np.concatenate([np.arange(a, b) for a, b in CEILING_STRIPS])
    rows_t = torch.from_numpy(rows).to(DEV)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(11)
    g_feat = torch.zeros((1, H, W, D), device=DEV)
    g_soft = torch.zeros((1, H, W), device=DEV)
    g_feat[0, rows_t] = torch.rand((len(rows), W, D), device=DEV, generator=gen)
    g_soft[0, rows_t] = torch.rand((len(rows), W), device=DEV, generator=gen)
    (feat, idx, wts, soft, g_fvi, g_ff), names = traced_step(H, W, T(fvz), T(fvi), T(ff), T(fnz), g_feat, g_soft)
    assert FWD2 in names, names
    assert_raster_bwd_kernel(names, D, W)
    pick = lambda t: N(t[0, rows_t])
    o, o_gxy, o_gff = strip_oracle_one_view(H, W, fvz, fvi, ff, fnz, N(g_feat[0, rows_t]), N(g_soft[0, rows_t]),
                                            CEILING_STRIPS)
    del g_feat
    assert (o["idx"] >= 0).any() and (o["idx"] < 0).any()
    assert np.array_equal(pick(idx), o["idx"])
    assert bits_equal(pick(wts), o["w"])
    e_feat = check_feat(feat[0, rows_t], o["feat"], False)
    np.testing.assert_allclose(pick(soft), o["soft"], rtol=0, atol=1e-6)
    e_xy, e_ff = rel_err(N(g_fvi), o_gxy), rel_err(N(g_ff), o_gff)
    print(f"[16384^2 D={D}] feat {e_feat:.1e} grad_fvi {e_xy:.2e} grad_ff {e_ff:.2e}")
    assert e_xy <= GRAD_REL and e_ff <= GRAD_REL


@pytest.mark.parametrize("B,H,W", [(2, 40, 16384), (1, 16384, 36)])
def test_size_ceiling_thin_images(B, H, W):
    """Images 16384 px long on one side, compared whole; 16384 x 36 has W % 4 != 0."""
    fvz, fvi, fnz, ff = ceiling_scene(B, 3, level=3, seed=B)
    rng = np.random.default_rng(12)
    g_feat = rng.uniform(size=(B, H, W, 3)).astype(np.float32)
    g_soft = rng.uniform(size=(B, H, W)).astype(np.float32)
    (feat, idx, wts, soft, g_fvi, g_ff), names = traced_step(H, W, T(fvz), T(fvi), T(ff), T(fnz), T(g_feat), T(g_soft))
    assert_raster_bwd_kernel(names, 3, W)
    o_feat, o_soft, o_idx, o_w = oracle.dibr_rasterization(H, W, fvz, fvi, ff, fnz, return_weights=True)
    assert (o_idx >= 0).any() and (o_idx < 0).any()
    assert np.array_equal(N(idx), o_idx)
    assert bits_equal(N(wts), o_w)
    e_feat = check_feat(feat, o_feat, False)
    np.testing.assert_allclose(N(soft), o_soft, rtol=0, atol=1e-6)
    o_gxy, o_gff, _, _ = oracle.dibr_rasterization_backward(g_feat, g_soft, o_idx, o_w, fvi, ff)
    e_xy, e_ff = rel_err(N(g_fvi), o_gxy), rel_err(N(g_ff), o_gff)
    print(f"\n[{B}x{H}x{W}] feat {e_feat:.1e} grad_fvi {e_xy:.2e} grad_ff {e_ff:.2e}")
    assert e_xy <= GRAD_REL and e_ff <= GRAD_REL


# ---------------------------------------------------------------------------
# knum on either side of kEnumK = 32: enumerate / evaluate kernels and hit-cache slots (<= 32)
# or the single-kernel path (> 32)
@pytest.mark.parametrize("cache", ["full", "empty"])
@pytest.mark.parametrize("knum", [32, 33])
def test_knum_boundary(knum, cache, monkeypatch):
    if cache == "empty":
        monkeypatch.setattr(_host, "CACHE_TILE_FRACTION", 0.0)
        monkeypatch.setattr(_host, "CACHE_MIN_TILES", 0)
    boxlen = 0.05
    fvz, fvi, fnz = synthetic.icosphere_views(1, 5, seed=61)
    H, W = 112, 120
    ff = synthetic.random_features(1, fvz.shape[1], 1, seed=62)
    rng = np.random.default_rng(63)
    g_soft = rng.uniform(size=(1, H, W)).astype(np.float32)
    (feat, idx, wts, soft, g_fvi, _), names = traced_step(H, W, T(fvz), T(fvi), T(ff), T(fnz), None, T(g_soft),
                                                          knum=knum, boxlen=boxlen)
    assert ("soft_enum_kernel" in names) == (knum <= 32 and cache == "full"), names
    o_feat, o_idx = oracle.rasterize(H, W, fvz, fvi, ff, fnz >= 0)
    assert np.array_equal(N(idx), o_idx)
    o_soft, _, o_cidx, _ = oracle.dibr_soft_mask(fvi, o_idx, SIGMAINV, boxlen, knum, M, return_lists=True)
    truncated = int((o_cidx[..., -1] >= 0).sum())         # pixels whose candidate list is full
    assert truncated > 100, truncated
    e_soft = float(np.abs(N(soft) - o_soft).max())
    o_g = oracle.dibr_soft_mask_backward(g_soft, fvi, o_idx, SIGMAINV, boxlen, knum, M)
    e_g = rel_err(N(g_fvi), o_g)
    print(f"\n[knum={knum} cache {cache}] {truncated} pixels truncated; soft {e_soft:.1e} grad_fvi {e_g:.2e}")
    assert e_soft <= 1e-6 and e_g <= GRAD_REL


# ---------------------------------------------------------------------------
# Tensors at a storage offset (contiguous views 4 / 2 bytes into a buffer): copied before the C ABI
def offset_view(t):
    """t's values as a contiguous view one element into a buffer (differentiable: the gradient of the
    view reaches t)."""
    v = torch.cat([t.new_zeros(1), t.reshape(-1)])[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


@pytest.mark.parametrize("ft", ["fp32", "bf16"])
def test_misaligned_inputs_and_upstream_gradients(ft):
    dt = torch.bfloat16 if ft == "bf16" else torch.float32
    fvz, fvi, fnz = synthetic.icosphere_views(2, 3, seed=71)
    B, F = fvz.shape[:2]
    H, W, D = 72, 96, 4                                            # the row-walk backward (cp.async)
    ff = T(synthetic.random_features(B, F, D, seed=72)).to(dt)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(73)
    g_feat = torch.rand((B, H, W, D), device=DEV, generator=gen).to(dt)
    g_soft = torch.rand((B, H, W), device=DEV, generator=gen)
    res = []
    for move in (lambda t: t, offset_view):
        t_fvi = T(fvi).requires_grad_(True)
        t_ff = ff.clone().requires_grad_(True)
        feat, soft, idx = dibr_rasterization(H, W, move(T(fvz)), move(t_fvi), move(t_ff), move(T(fnz)))
        torch.autograd.backward([feat, soft], [move(g_feat), move(g_soft)])
        f2, i2 = rasterize(H, W, move(T(fvz)), move(T(fvi)), move(ff))
        s2 = dibr_soft_mask(move(T(fvi)), move(i2))
        res.append((feat, soft, idx, f2, i2, s2, t_fvi.grad, t_ff.grad))
    for k in range(6):
        assert torch.equal(res[0][k], res[1][k]), k
    for k in (6, 7):
        assert rel_err(N(res[1][k]), N(res[0][k]).astype(np.float64)) <= 1e-6, k
    if ft == "fp32":     # the operator the reference's own wrappers call
        _, idx, wts, _, _ = _host.forward(_lib.RASTER, H, W, T(fvz), T(fvi), ff, None, None, M, EPS, 0., 0., 0)
        a = b200_C.render.mesh.rasterize_backward_cuda(g_feat, g_feat, idx, wts, T(fvi), ff, EPS)
        b = b200_C.render.mesh.rasterize_backward_cuda(offset_view(g_feat), g_feat, offset_view(idx),
                                                       offset_view(wts), offset_view(T(fvi)), offset_view(ff), EPS)
        for x, y in zip(a, b):
            assert rel_err(N(y), N(x).astype(np.float64)) <= 1e-6
