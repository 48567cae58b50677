"""Exact Euclidean distance transform and the Dice / Jaccard / Hausdorff / surface-distance agreement of masks.

CPU tests pin the oracle (oracle/surface_distance.py, a thin layer over scipy.ndimage and np.percentile) with known
answers, the percentile restatement against np.percentile bit for bit, the argument errors and the C ABI's error
returns.  ``-m gpu`` tests compare the kernels with scipy bit for bit at unit spacing, within 1e-15 at other spacings,
and check batching, slice stacks, repetition and graph replay."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import masked_metrics as omm
from oracle import morphology as omo
from oracle import surface_distance as osd

gpu = pytest.mark.gpu


def _random(shape, p, seed):
    return np.random.RandomState(seed).rand(*shape) < p


def _head(shape, seed):
    """A bright noisy ellipsoid in a dark noisy field with two darker spheres inside (the volumes of
    tests/test_morphology.py)."""
    rng = np.random.RandomState(seed)
    grids = np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij")
    inside = sum((g / 0.7) ** 2 for g in grids) < 1
    v = np.where(inside, rng.gamma(4.0, 100.0, size=shape), rng.gamma(1.0, 10.0, size=shape))
    for c in (0.25, -0.3):
        v[sum((g - c) ** 2 for g in grids) < 0.15 ** 2] = rng.gamma(1.0, 10.0)
    return v.astype(np.float32)


def _ball(shape, centre, radius):
    g = np.meshgrid(*[np.arange(s) - c for s, c in zip(shape, centre)], indexing="ij")
    return sum(a * a for a in g) <= radius * radius


def _cube(shape, lo, size):
    m = np.zeros(shape, bool)
    m[tuple(slice(a, a + size) for a in lo)] = True
    return m


# ------------------------------------------------------------------------------------------------- oracle (CPU)
def test_edt_known_answers():
    m = np.ones((7, 9, 11), bool)
    m[2, 3, 4] = False
    g = np.indices(m.shape)
    exact = np.sqrt((g[0] - 2) ** 2 + (g[1] - 3) ** 2 + (g[2] - 4) ** 2.0)
    assert np.array_equal(osd.distance_transform_edt(m), exact)
    aniso = np.sqrt(((g[0] - 2) * 2.0) ** 2 + ((g[1] - 3) * 0.5) ** 2 + ((g[2] - 4) * 1.25) ** 2)
    assert np.allclose(osd.distance_transform_edt(m, (2.0, 0.5, 1.25)), aniso, rtol=1e-15, atol=0)
    assert np.isinf(osd.distance_transform_edt(np.ones((4, 5), bool))).all()          # the departure from scipy
    assert np.isfinite(ndimage.distance_transform_edt(np.ones((4, 5), bool))).all()
    assert not osd.distance_transform_edt(np.zeros((3, 4, 5), bool)).any()
    stack = np.stack([m[2], np.ones_like(m[2])])
    got = osd.distance_transform_edt(stack, spatial_dims=2)
    assert np.array_equal(got[0], ndimage.distance_transform_edt(m[2])) and np.isinf(got[1]).all()


def test_agreement_known_answers():
    shape = (24, 26, 28)
    a = _cube(shape, (4, 5, 6), 10)
    for k in (1, 2, 3):
        b = _cube(shape, (4, 5, 6 + k), 10)
        r = osd.agreement(a, b)
        assert r["hausdorff"] == k and r["dice"] == 2 * (10 - k) / 20 and r["jaccard"] == (10 - k) / (10 + k)
        assert r["hausdorff_percentile"] <= k and r["average_surface_distance"] > 0
    same = osd.agreement(a, a, percentile=100)
    assert same["dice"] == same["jaccard"] == 1 and all(same[k] == 0 for k in osd.KEYS[2:])
    inner, outer = _ball(shape, (12, 13, 14), 5), _ball(shape, (12, 13, 14), 9)
    r = osd.agreement(inner, outer, percentile=0)
    assert 3 <= r["hausdorff_percentile"] <= r["hausdorff"] <= 5 and r["dice"] == 2 * inner.sum() / (inner.sum() + outer.sum())
    empty, full = np.zeros(shape, bool), np.ones(shape, bool)
    both = osd.agreement(empty, empty)
    assert all(math.isnan(both[k]) for k in osd.KEYS)
    for p, t in ((a, empty), (empty, a)):
        one = osd.agreement(p, t)
        assert one["dice"] == one["jaccard"] == 0 and all(one[k] == math.inf for k in osd.KEYS[2:])
    r = osd.agreement(full, full)                      # a full mask's surface is its outer layer
    assert r["dice"] == 1 and r["hausdorff"] == 0
    r = osd.agreement(full, a)
    assert r["hausdorff"] == ndimage.distance_transform_edt(~osd.surface(a))[osd.surface(full)].max()


def test_percentile_restatement_is_numpy_bit_for_bit():
    rng = np.random.RandomState(0)
    for n in (1, 2, 3, 21, 100, 100_000):
        v = rng.gamma(2.0, 3.0, size=n)
        v[:: 7] = np.round(v[:: 7])                    # ties
        for q in (95, 0, 100, 50, 99.9, 0.1, 33.3, 1e-9, 100 - 1e-9, 5):
            got, ref = osd.percentile_restated(v, q), np.percentile(v, q)
            assert got == ref or (math.isnan(got) and math.isnan(ref)), (n, q, got, ref)


def test_arguments_are_validated_before_the_device():
    from mpgan import transforms as T
    m = torch.ones(2, 8, 9, 10, dtype=torch.bool)
    for bad in (m.float(), m.to(torch.int32), m.numpy(), torch.zeros(3, 0, 4, dtype=torch.bool), m[0, 0, 0]):
        with pytest.raises(ValueError):
            T.distance_transform_edt(bad)
        with pytest.raises(ValueError):
            T.mask_agreement(bad, m)
        with pytest.raises(ValueError):
            T.mask_agreement(m, bad)
    for s in (0, -1.0, math.inf, math.nan, True, (1.0, 1.0), (1.0, 2.0, 0.0), (1, 1, 1, 1), "1", [1.0, None, 1.0]):
        with pytest.raises(ValueError):
            T.distance_transform_edt(m, sampling=s)
        with pytest.raises(ValueError):
            T.mask_agreement(m, m, sampling=s)
    for kw in (dict(spatial_dims=1), dict(spatial_dims=4), dict(spatial_dims=True)):
        with pytest.raises(ValueError):
            T.distance_transform_edt(m, **kw)
    for kw in (dict(percentile=-1), dict(percentile=100.5), dict(percentile=math.nan), dict(percentile=True),
               dict(percentile="95"), dict(connectivity=0), dict(connectivity=4), dict(connectivity=1.0),
               dict(spatial_dims=2, connectivity=3), dict(spatial_dims=5)):
        with pytest.raises(ValueError):
            T.mask_agreement(m, m, **kw)
    with pytest.raises(ValueError):
        T.mask_agreement(m, m[:, :, :, :9])
    with pytest.raises(ValueError):
        T.distance_transform_edt(m[0], sampling=(1.0, 1.0))                         # rank 3: three spacings
    for ok in (m, m.to(torch.uint8)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            T.distance_transform_edt(ok, sampling=(2.0, 1.0, 0.5))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            T.mask_agreement(ok, m, sampling=2.0, percentile=0, connectivity=3)


def test_c_abi_rejects_bad_arguments():
    from mpgan import _lib
    lib = _lib.load()
    need_d = lib.mpgan_distance_transform_workspace(2, 4, 5, 6)
    need_a = lib.mpgan_mask_agreement_workspace(2, 4, 5, 6)
    assert need_d >= 12 * 240 and need_a >= 30 * 240
    for fn in (lib.mpgan_distance_transform_workspace, lib.mpgan_mask_agreement_workspace):
        assert fn(0, 4, 5, 6) == 0 and fn(1, 2 ** 11, 2 ** 10, 2 ** 10) == 0 and fn(1, 4, 0, 6) == 0
    m, t, o, ws = 1 << 20, 1 << 24, 1 << 30, 1 << 32      # never dereferenced: the checks come first

    def edt(mask=m, rank=3, items=2, d=4, h=5, w=6, s=(1.0, 1.0, 1.0), out=o, wsp=ws, nbytes=need_d, **_):
        return lib.mpgan_distance_transform(mask, rank, items, d, h, w, *s, out, wsp, nbytes, None)

    def agree(mask=m, truth=t, rank=3, items=2, d=4, h=5, w=6, s=(1.0, 1.0, 1.0), conn=1, pct=95.0, out=o, wsp=ws,
              nbytes=need_a):
        return lib.mpgan_mask_agreement(mask, truth, rank, items, d, h, w, *s, conn, pct, out, wsp, nbytes, None)

    for kw in (dict(mask=None), dict(out=None), dict(wsp=None)):
        assert edt(**kw) == -1 and "null" in _lib.last_error()
        assert agree(**kw) == -1 and "null" in _lib.last_error()
    assert agree(truth=None) == -1 and "null" in _lib.last_error()
    cases = [(dict(rank=1), "rank"), (dict(rank=4), "rank"), (dict(rank=2), "d 4"), (dict(items=0), "size"),
             (dict(w=0), "size"), (dict(d=2 ** 11, h=2 ** 10, w=2 ** 10), "voxels"),
             (dict(s=(0.0, 1.0, 1.0)), "spacing"), (dict(s=(1.0, -2.0, 1.0)), "spacing"),
             (dict(s=(1.0, 1.0, math.inf)), "spacing"), (dict(s=(math.nan, 1.0, 1.0)), "spacing"),
             (dict(wsp=o - 8), "overlap"), (dict(wsp=m - 8), "overlap")]
    for kw, text in cases:
        assert edt(**kw) == -1 and text in _lib.last_error(), (kw, _lib.last_error())
        assert agree(**kw) == -1 and text in _lib.last_error(), (kw, _lib.last_error())
    assert edt(nbytes=need_d - 1) == -1 and "workspace" in _lib.last_error()
    assert edt(out=m + 100) == -1 and "overlap" in _lib.last_error()
    for kw, text in ((dict(nbytes=need_a - 1), "workspace"), (dict(conn=0), "connectivity"), (dict(conn=4), "connectivity"),
                     (dict(rank=2, d=1, conn=3), "connectivity"), (dict(pct=-0.5), "percentile"),
                     (dict(pct=100.5), "percentile"), (dict(pct=math.nan), "percentile"),
                     (dict(out=t + 8), "overlap"), (dict(wsp=t - 8), "overlap")):
        assert agree(**kw) == -1 and text in _lib.last_error(), (kw, _lib.last_error())


# ------------------------------------------------------------------------------------------------- CUDA kernels
def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _check_edt(mask, sampling=None, spatial_dims=None):
    from mpgan import transforms as T
    (tm,) = _cuda(mask)
    got = T.distance_transform_edt(tm, sampling, spatial_dims)
    assert got.dtype == torch.float64 and tuple(got.shape) == mask.shape
    got = got.cpu().numpy()
    ref = osd.distance_transform_edt(mask, sampling, spatial_dims)
    if sampling is None:
        bad = got != ref
        assert not bad.any(), f"{int(bad.sum())} of {ref.size} voxels differ, e.g. {got[bad][:3]} vs {ref[bad][:3]}"
    else:
        fin = np.isfinite(ref)
        assert np.array_equal(fin, np.isfinite(got))
        err = np.abs(got[fin] - ref[fin]) / np.maximum(ref[fin], 1e-300)
        assert err.max(initial=0) <= 1e-15, err.max()


@gpu
@pytest.mark.parametrize("rank", [2, 3])
def test_edt_matches_scipy_bit_for_bit(rank):
    shapes = [(3, 331, 257), (1, 1, 77), (2, 1000, 3)] if rank == 2 else [(37, 45, 53), (5, 130, 7), (2, 19, 1, 23)]
    for shape in shapes:
        for p in (0.02, 0.5, 0.9):                       # "in" probability: long and short distances
            _check_edt(_random(shape, p, int(100 * p)), spatial_dims=rank)
        _check_edt(np.ones(shape, bool), spatial_dims=rank)   # no "out" voxel: +inf
        _check_edt(np.zeros(shape, bool), spatial_dims=rank)
    head = omm.foreground_mask(_head((61, 70, 83), 3))
    _check_edt(head if rank == 3 else head[30], spatial_dims=rank)
    _check_edt(~head if rank == 3 else ~head[30], spatial_dims=rank)


@gpu
def test_edt_of_one_out_voxel_in_a_large_volume():
    from mpgan import transforms as T
    shape, at = (256, 512, 512), (3, 500, 7)
    m = torch.ones(shape, dtype=torch.bool, device="cuda")
    m[at] = False
    got = T.distance_transform_edt(m)
    g = [torch.arange(s, device="cuda", dtype=torch.float64) - a for s, a in zip(shape, at)]
    ref = torch.sqrt(((g[0] ** 2)[:, None, None] + (g[1] ** 2)[None, :, None]) + (g[2] ** 2)[None, None, :])
    assert torch.equal(got, ref)                       # integer squares: exact in any order; sqrt correctly rounded


@gpu
def test_edt_anisotropic_sampling():
    for shape, samp in (((37, 45, 53), (2.0, 0.7, 1.3)), ((37, 45, 53), 0.35), ((120, 97), (3.0, 0.5))):
        for p in (0.02, 0.6):
            _check_edt(_random(shape, p, 5), samp)
    head = omm.foreground_mask(_head((64, 64, 64), 4))
    _check_edt(head, (2.5, 1.0, 1.0))


def _check_agreement(p, t, sampling=None, percentile=95, connectivity=1, spatial_dims=None):
    from mpgan import transforms as T
    tp, tt = _cuda(p, t)
    got = T.mask_agreement(tp, tt, sampling, percentile, connectivity, spatial_dims)
    ref = osd.mask_agreement(p, t, sampling, percentile, connectivity, spatial_dims)
    exact = ("dice", "jaccard") + (("hausdorff", "hausdorff_percentile") if sampling is None else ())
    for k in osd.KEYS:
        g, r = got[k].cpu().numpy(), ref[k]
        assert got[k].dtype == torch.float64 and g.shape == r.shape, k
        if k in exact:
            assert np.array_equal(g, r, equal_nan=True), (k, g, r)
        else:
            fin = np.isfinite(r)
            assert np.array_equal(np.isnan(g), np.isnan(r)) and np.array_equal(g[~fin & ~np.isnan(r)], r[~fin & ~np.isnan(r)])
            tol = 1e-12 if k.endswith("surface_distance") else 1e-14
            assert np.all(np.abs(g[fin] - r[fin]) <= tol * np.abs(r[fin])), (k, g, r)
    return got


@gpu
@pytest.mark.parametrize("conn", [1, 2, 3])
def test_mask_agreement_matches_the_oracle_128(conn):
    x = _head((128, 128, 128), 5)
    head = omo.foreground_mask(x, True, True, conn)
    noisy = x * np.random.RandomState(6).gamma(20.0, 1 / 20.0, size=x.shape).astype(np.float32)
    head2 = omo.foreground_mask(noisy, True, True, conn)
    shifted = np.roll(head, (2, -3, 1), axis=(0, 1, 2))
    eroded = omo.binary_erosion(head, 3, conn)
    for other in (shifted, eroded, head2):
        for pct in (95, 0, 100):
            _check_agreement(other, head, percentile=pct, connectivity=conn)
    _check_agreement(shifted, head, sampling=(2.0, 1.0, 0.8), connectivity=conn)


@gpu
def test_slice_stacks_and_batches_equal_per_image_calls():
    from mpgan import transforms as T
    x = _head((40, 41, 43), 7)
    head = omo.foreground_mask(x, True, True)
    pairs = [(np.roll(head, s, axis=2), head) for s in (0, 1, 3)]
    pairs.append((np.zeros_like(head), head))                       # one empty
    pairs.append((np.zeros_like(head), np.zeros_like(head)))        # both empty
    pairs.append((omo.binary_dilation(head, 2), np.ones_like(head)))
    ps, ts = np.stack([p for p, _ in pairs]), np.stack([t for _, t in pairs])
    batch = _check_agreement(ps, ts, percentile=90)
    tps, tts = _cuda(ps, ts)
    for i in range(len(pairs)):
        one = T.mask_agreement(tps[i], tts[i], percentile=90)
        for k in osd.KEYS:
            assert torch.equal(one[k], batch[k][i]) or (one[k].isnan() and batch[k][i].isnan()), (i, k)
    assert batch["hausdorff"][3] == math.inf and batch["hausdorff"][4].isnan() and batch["dice"][3] == 0
    slices, slices_t = ps[:3].reshape(-1, 41, 43), ts[:3].reshape(-1, 41, 43)
    stack = _check_agreement(slices, slices_t, connectivity=2, spatial_dims=2)
    ts2, tt2 = _cuda(slices, slices_t)
    for i in (0, 17, 45, 119):
        one = T.mask_agreement(ts2[i], tt2[i], connectivity=2)
        for k in osd.KEYS:
            assert torch.equal(one[k], stack[k][i]) or (one[k].isnan() and stack[k][i].isnan()), (i, k)
    dist = T.distance_transform_edt(tps, spatial_dims=3)
    for i in (0, 3):
        assert torch.equal(dist[i], T.distance_transform_edt(tps[i]))


@gpu
def test_repetition_and_graph_replay_change_no_bit():
    from mpgan import transforms as T
    x = _head((2, 64, 72, 80), 9)
    masks = np.stack([omo.foreground_mask(x[i], True, True) for i in range(2)])
    p, t = np.roll(masks, 2, axis=3), masks
    tp, tt = _cuda(p, t)
    sp, st = tp.clone(), tt.clone()

    def run(a, b):
        r = T.mask_agreement(a, b, sampling=(1.0, 1.0, 1.0), percentile=95)
        return torch.stack([r[k] for k in osd.KEYS]), T.distance_transform_edt(b, sampling=(1.5, 1.0, 1.0))

    base = run(tp, tt)
    for _ in range(3):
        again = run(tp, tt)
        assert all(torch.equal(u, v) for u, v in zip(base, again))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = run(sp, st)
    for o in outs:
        o.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(outs, base))
    q = np.stack([omo.binary_erosion(masks[i], 2) for i in range(2)])
    sp.copy_(torch.from_numpy(q).cuda())
    g.replay()
    torch.cuda.synchronize()
    fresh = run(sp, st)
    assert all(torch.equal(u, v) for u, v in zip(outs, fresh))
    ref = osd.mask_agreement(q, t, percentile=95)
    assert np.array_equal(outs[0][2].cpu().numpy(), ref["hausdorff"])
