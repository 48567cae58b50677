"""Foreground-masked MAE, MSE, PSNR, SSIM and mutual information, and Otsu's foreground mask.

CPU tests pin the oracle (oracle/masked_metrics.py): the Otsu restatement against np.histogram and known answers, the
masked scores against the unmasked ones for an all-true mask and against explicit selections; they also check the
argument errors and the C ABI's error returns.  ``-m gpu`` tests compare the kernels with the oracle: Otsu thresholds
and masks bit for bit, masked counts and edges bit for bit with entropies to 1e-12, MAE / MSE / PSNR to 1e-9 and SSIM to
1e-7 (the tolerances of the unmasked tests)."""
import math
from ctypes import c_double

import numpy as np
import pytest
import torch

from oracle import masked_metrics as omm
from oracle import metrics as om
from oracle import mutual_info as omi
from oracle import transforms as ot

gpu = pytest.mark.gpu


def _volume(shape, seed, background=0.4):
    """Synthetic MRI-like volume: positive intensities with a large exactly-zero background."""
    rng = np.random.RandomState(seed)
    v = rng.gamma(2.0, 150.0, size=shape).astype(np.float32)
    v[rng.rand(*shape) < background] = 0.0
    return v


def _head(shape, seed):
    """A bright noisy ellipsoid (the head) in a dark noisy field of view, so that Otsu has a foreground to find."""
    rng = np.random.RandomState(seed)
    grids = np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij")
    inside = sum((g / 0.7) ** 2 for g in grids) < 1
    v = np.where(inside, rng.gamma(4.0, 100.0, size=shape), rng.gamma(1.0, 10.0, size=shape))
    return v.astype(np.float32)


def _display_pair(shape, seed, vol=_volume):
    """(generated, truth) on the display range 0..255 (integers): a noisy copy of the truth, and the truth."""
    v = vol(shape, seed)
    noise = np.random.RandomState(seed + 100).normal(1.0, 0.2, size=shape).astype(np.float32)
    return ot.to_display_range(v * noise), ot.to_display_range(v)


def _unit_pair(shape, seed):
    """(generated, truth) in [-1, 1], the generator's output range."""
    rng = np.random.RandomState(seed)
    truth = (rng.rand(*shape) * 2 - 1).astype(np.float32)
    return np.clip(truth + rng.normal(0, 0.3, shape), -1, 1).astype(np.float32), truth


def _random_mask(shape, seed, p=0.6):
    return np.random.RandomState(seed).rand(*shape) < p


# ------------------------------------------------------------------------------------------------- oracle (CPU)
def test_otsu_histogram_is_numpys():
    rng = np.random.RandomState(0)
    for t in range(300):
        scale = 10.0 ** rng.uniform(-3, 4)
        x = (rng.randn(500) * scale + rng.randn() * scale * rng.choice([0, 1, 100])).astype(np.float32)
        counts, e = omm.otsu_histogram(x, 256)
        ref_counts, ref_e = np.histogram(x, 256)
        assert ref_e.dtype == np.float32 and np.array_equal(e.view(np.uint32), ref_e.view(np.uint32)), t
        assert np.array_equal(counts, ref_counts), t
    x = _display_pair((20, 21, 22), 1)[1]
    assert np.array_equal(omm.otsu_histogram(x)[0], np.histogram(x, 256)[0])


def test_otsu_known_answers():
    # two levels: every split between them has the same variance, so the first one, bin 0, wins
    x = np.full((10, 12, 14), 10.0, np.float32)
    x[:, :5] = 200.0
    _, e = omm.otsu_histogram(x)
    t = omm.otsu_threshold(x)
    assert t == np.float32((e[0] + e[1]) / np.float32(2)) and 10.0 < t < 200.0
    assert np.array_equal(omm.foreground_mask(x), x == 200.0)
    # two separated modes: the threshold splits them exactly (the first split in the gap between them)
    rng = np.random.RandomState(2)
    y = np.concatenate([rng.normal(20, 3, 5000), rng.normal(120, 5, 3000)]).astype(np.float32)
    t = omm.otsu_threshold(y)
    assert y[y < 70].max() <= t < y[y > 70].min() and np.array_equal(omm.foreground_mask(y), y > 70)
    for c in (0.0, -3.5, 255.0):                                    # constant: the value itself, an empty mask
        assert omm.otsu_threshold(np.full((4, 5), c, np.float32)) == np.float32(c)
        assert not omm.foreground_mask(np.full((4, 5), c, np.float32)).any()
    for bad in (np.inf, -np.inf, np.nan):                           # non-finite extreme: NaN, an empty mask
        z = y.copy()
        z[7] = bad
        assert np.isnan(omm.otsu_threshold(z))
    t = omm.otsu_thresholds(np.stack([x[0], x[0] * 2, np.full_like(x[0], 5.0)]), spatial_dims=2)
    assert t.shape == (3,) and t[2] == 5.0 and t[1] > t[0]


def test_masked_oracles_with_an_all_true_mask_are_the_unmasked_ones():
    gen, truth = _display_pair((18, 19, 20), 3)
    m = np.ones(gen.shape, bool)
    d = gen.astype(np.float64) - truth
    assert omm.mean_absolute_error(gen, truth, m) == pytest.approx(np.abs(d).mean(), rel=1e-12)
    assert omm.mean_squared_error(gen, truth, m) == pytest.approx((d * d).mean(), rel=1e-12)
    assert omm.peak_signal_noise_ratio(truth, gen, m, data_range=255.0) == pytest.approx(
        om.peak_signal_noise_ratio(truth, gen, data_range=255.0), rel=1e-12)
    for kw in ({}, dict(gaussian_weights=True)):
        assert omm.structural_similarity(gen, truth, m, data_range=255.0, **kw) == pytest.approx(
            om.structural_similarity(gen, truth, data_range=255.0, **kw), rel=1e-12)
    c, e1, e2 = omm.joint_histogram(gen, truth, m, 100)
    rc, r1, r2 = omi.joint_histogram(gen, truth, 100)
    assert np.array_equal(c, rc) and np.array_equal(e1, r1) and np.array_equal(e2, r2)


def test_masked_ssim_is_the_mean_over_masked_centres():
    gen, truth = _unit_pair((15, 16, 17), 4)
    m = _random_mask(gen.shape, 5)
    for kw, win in (({}, 7), (dict(win_size=5), 5), (dict(gaussian_weights=True, sigma=1.0), 9)):
        _, s = om.structural_similarity(gen, truth, data_range=2.0, full=True, **kw)
        r = win // 2
        centres = [tuple(p) for p in np.argwhere(m) if all(r <= q < n - r for q, n in zip(p, m.shape))]
        ref = np.mean([s[p] for p in centres])
        assert omm.structural_similarity(gen, truth, m, data_range=2.0, **kw) == pytest.approx(ref, rel=1e-12)
    assert np.isnan(omm.structural_similarity(gen, truth, np.zeros_like(m), data_range=2.0))
    assert np.isnan(omm.mean_absolute_error(gen, truth, np.zeros_like(m)))


def test_arguments_are_validated_before_the_device():
    from mpgan import inference
    from mpgan import transforms as T
    x, y = torch.zeros(2, 16, 16, 16), torch.zeros(2, 16, 16, 16)
    good = torch.ones(2, 16, 16, 16, dtype=torch.bool)
    bad_masks = [good[:, :, :, :15], good.float(), good.to(torch.int32), good.numpy(),
                 torch.ones(2, 16, 16, 16, dtype=torch.bool, device="meta")]
    fns = [lambda m: T.mean_absolute_error(x, y, mask=m), lambda m: T.mean_squared_error(x, y, mask=m),
           lambda m: T.error_sums(x, y, mask=m), lambda m: T.peak_signal_noise_ratio(x, y, data_range=1.0, mask=m),
           lambda m: T.structural_similarity(x, y, data_range=1.0, mask=m),
           lambda m: T.joint_histogram(x, y, mask=m), lambda m: T.mutual_information(x, y, mask=m),
           lambda m: T.normalized_mutual_information(x, y, mask=m),
           lambda m: inference.evaluate(x, y, data_range=1.0, mi_bins=10, mask=m)]
    for fn in fns:
        for m in bad_masks:
            with pytest.raises(ValueError):
                fn(m)
        for m in (good, good.to(torch.uint8)):          # valid arguments on CPU tensors: the no-fallback error
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                fn(m)
    for kw in (dict(bins=1), dict(bins=257), dict(bins=2.0), dict(bins=True), dict(spatial_dims=1),
               dict(spatial_dims=4), dict(spatial_dims=True)):
        with pytest.raises(ValueError):
            T.otsu_threshold(x, **kw)
    for kw in (dict(bins=257), dict(threshold="1"), dict(threshold=True), dict(threshold=torch.zeros(3)),
               dict(threshold=torch.zeros(2, dtype=torch.float64)), dict(threshold=torch.zeros(2, device="meta"))):
        with pytest.raises(ValueError):
            T.foreground_mask(x, **kw)
    for fn in (T.otsu_threshold, T.foreground_mask):
        for bad in (x.double(), x.numpy(), torch.zeros(3, 0, 4)):
            with pytest.raises(ValueError):
                fn(bad)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.foreground_mask(x, threshold=torch.zeros(2))


def test_c_abi_rejects_bad_sizes():
    from mpgan import _lib
    lib = _lib.load()
    p = 256   # never dereferenced: the checks come first
    assert lib.mpgan_err_sums_masked(p, p, None, 10, p, None) == -1 and "null" in _lib.last_error()
    assert lib.mpgan_err_sums_masked(p, p, p, -1, p, None) == -1 and "size" in _lib.last_error()
    assert lib.mpgan_err_sums_masked(p, p, p, 0, p, None) == 0                      # nothing to do, no CUDA call
    taps = (c_double * 7)(*([1 / 7] * 7))

    def ssim(mask=p, count=p, rank=3, d=16, win=7):
        return lib.mpgan_ssim_sums_masked(p, p, mask, rank, 1, d, 16, 16, taps, win, 1.0, 1.0, 1.0, p, count, None)

    assert ssim(mask=None) == -1 and "null" in _lib.last_error()
    assert ssim(count=None) == -1 and "null" in _lib.last_error()
    assert ssim(rank=4) == -1 and ssim(d=6) == -1 and ssim(win=4) == -2
    need = lib.mpgan_mutual_info_workspace(3)

    def mi(mask=p, items=3, n=1000, bins=100, ws=need):
        return lib.mpgan_mutual_info_masked(p, p, mask, items, n, bins, p, None, p, p, ws, None)

    assert mi(mask=None) == -1 and "null" in _lib.last_error()
    assert mi(bins=129) == -1 and mi(items=0) == -1 and mi(n=0) == -1 and mi(n=2 ** 31) == -1
    assert mi(ws=need - 1) == -1 and "workspace" in _lib.last_error()
    wneed = lib.mpgan_otsu_threshold_workspace(3, 256)
    assert wneed >= 3 * 16 + 3 * 256 * 8 and lib.mpgan_otsu_threshold_workspace(0, 256) == 0

    def otsu(x=p, thr=p, ws_ptr=p, items=3, n=1000, bins=256, ws=wneed):
        return lib.mpgan_otsu_threshold(x, items, n, bins, thr, ws_ptr, ws, None)

    for kw in (dict(x=None), dict(thr=None), dict(ws_ptr=None)):
        assert otsu(**kw) == -1 and "null" in _lib.last_error()
    assert otsu(bins=1) == -1 and otsu(bins=257) == -1 and "bins" in _lib.last_error()
    assert otsu(items=0) == -1 and otsu(n=0) == -1 and otsu(n=2 ** 31) == -1
    assert otsu(ws=wneed - 1) == -1 and "workspace" in _lib.last_error()
    assert lib.mpgan_threshold_mask(p, p, 3, 100, None, None) == -1 and "null" in _lib.last_error()
    assert lib.mpgan_threshold_mask(p, p, 0, 100, p, None) == -1
    assert lib.mpgan_threshold_mask(p, p, 3, 0, p, None) == -1


# ------------------------------------------------------------------------------------------------- CUDA kernels
def _same(x, y):
    """Bit-identical tensors (NaN where NaN)."""
    x, y = x.detach().cpu().numpy().reshape(-1), y.detach().cpu().numpy().reshape(-1)
    return x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _check_otsu(x, spatial_dims=None):
    from mpgan import transforms as T
    (tx,) = _cuda(x)
    thr = T.otsu_threshold(tx, spatial_dims=spatial_dims)
    ref = omm.otsu_thresholds(x, spatial_dims)
    assert thr.dtype == torch.float32 and tuple(thr.shape) == ref.shape
    assert np.array_equal(thr.cpu().numpy().view(np.uint32), ref.view(np.uint32)), (thr, ref)
    if spatial_dims is None:
        m = T.foreground_mask(tx)
        assert m.dtype == torch.bool and np.array_equal(m.cpu().numpy(), omm.foreground_mask(x))
    return thr


@gpu
def test_otsu_threshold_and_mask_bit_exact():
    gen, truth = _display_pair((128, 128, 128), 1, _head)
    _check_otsu(truth)
    _check_otsu(gen)
    _check_otsu(_unit_pair((128, 128, 128), 2)[1])
    _check_otsu(_display_pair((61, 67, 13), 3, _head)[1])                       # ragged float4 body and tail
    _check_otsu(_display_pair((9, 1, 97, 101), 4, _head)[1])                    # (S, 1, H, W): one item per slice
    _check_otsu(_display_pair((9, 1, 97, 101), 4, _head)[1][:, 0], spatial_dims=2)
    x = _display_pair((5, 40, 41), 5, _head)[1]
    x[1] = 7.0                                                                  # a constant item
    x[2, 3, 4] = np.inf                                                         # a non-finite item
    x[3, 0, 0] = np.nan
    thr = _check_otsu(x, spatial_dims=2)
    assert thr[1] == 7.0 and torch.isnan(thr[2]) and torch.isnan(thr[3])


@gpu
def test_otsu_volume_larger_than_l2():
    from mpgan import transforms as T
    truth = _display_pair((256, 512, 512), 11)[1]
    (tx,) = _cuda(truth)
    thr = T.otsu_threshold(tx)
    ref = omm.otsu_threshold(truth)
    assert thr.cpu().numpy().view(np.uint32) == np.float32(ref).view(np.uint32)
    assert torch.equal(T.foreground_mask(tx), tx > thr)


def _assert_entropies(got, ref):
    """H1, H2, H12 and NMI to 1e-12 relative; MI = H1 + H2 - H12 is a difference, so its error is relative to them (the
    tolerances of the unmasked tests)."""
    got = [float(v) for v in got]
    for k in (0, 1, 2, 4):
        if np.isnan(ref[k]):
            assert np.isnan(got[k])
        else:
            assert abs(got[k] - ref[k]) <= 1e-12 * abs(ref[k]), (k, got[k], ref[k])
    assert abs(got[3] - ref[3]) <= 1e-12 * max(abs(ref[3]), ref[0] + ref[1]), (got[3], ref[3])


def _check_mi(a, b, m, bins=100, spatial_dims=None):
    """Masked joint histogram, edges and entropies of every item against the oracle: counts and edges bit for bit,
    entropies by ``_assert_entropies``.  Returns the device counts, edges, MI and NMI."""
    from mpgan import ops
    from mpgan import transforms as T
    ta, tb, tm = _cuda(a, b, m)
    counts, e1, e2 = T.joint_histogram(ta, tb, bins=bins, spatial_dims=spatial_dims, mask=tm)
    mi = T.mutual_information(ta, tb, bins=bins, spatial_dims=spatial_dims, mask=tm)
    nmi = T.normalized_mutual_information(ta, tb, bins=bins, spatial_dims=spatial_dims, mask=tm)
    nd = spatial_dims or min(a.ndim, 3)
    sp = a.shape[a.ndim - nd:]
    items, n = int(np.prod(a.shape[:a.ndim - nd])), int(np.prod(sp))
    c5 = torch.empty(items, bins, bins, dtype=torch.int64, device="cuda")
    out5 = torch.empty(items, 5, dtype=torch.float64, device="cuda")
    ops.mutual_info(ta, tb, items, n, bins, c5, None, out5, tm.view(torch.uint8))
    assert _same(mi.reshape(-1), out5[:, 3]) and _same(nmi.reshape(-1), out5[:, 4])
    ia, ib, im = (v.reshape((-1,) + sp) for v in (a, b, m))
    c = counts.cpu().numpy().reshape(-1, bins, bins)
    g1, g2 = e1.cpu().numpy().reshape(-1, bins + 1), e2.cpu().numpy().reshape(-1, bins + 1)
    h = out5.cpu().numpy()
    for i in range(ia.shape[0]):
        rc, r1, r2 = omm.joint_histogram(ia[i], ib[i], im[i], bins)
        assert np.array_equal(c[i], rc), i
        assert np.array_equal(g1[i].view(np.uint32), r1.view(np.uint32)), i
        assert np.array_equal(g2[i].view(np.uint32), r2.view(np.uint32)), i
        _assert_entropies(h[i], omi.entropies(rc))
    return counts, e1, e2, mi.cpu().numpy().reshape(-1), nmi.cpu().numpy().reshape(-1)


@gpu
def test_masked_mutual_information():
    from mpgan import transforms as T
    gen, truth = _display_pair((128, 128, 128), 6, _head)
    otsu = omm.foreground_mask(truth)
    assert 0.05 < otsu.mean() < 0.5                                            # the head, about 18 % of the field
    _check_mi(gen, truth, otsu)
    _check_mi(gen, truth, _random_mask(gen.shape, 7))
    one = np.zeros(gen.shape, bool)
    one[60, 61, 62] = True                                                     # one voxel: constant images, NMI 0 / 0
    counts, _, _, mi, nmi = _check_mi(gen, truth, one)
    assert int(counts.sum()) == 1 and mi[0] == 0 and np.isnan(nmi[0])
    _check_mi(*_unit_pair((61, 67, 13), 8), _random_mask((61, 67, 13), 9), bins=64)
    # a per-slice batch whose items start at every alignment, and a mask one byte off the images' alignment (scalar path)
    a, b = _unit_pair((7, 97, 101), 10)
    m = _random_mask(a.shape, 11)
    res = _check_mi(a, b, m, spatial_dims=2)
    ta, tb, tm = _cuda(a, b, m)
    flat = torch.empty(m.size + 1, dtype=torch.bool, device="cuda")
    flat[1:] = tm.reshape(-1)
    shifted = flat[1:].view(tm.shape)
    got = T.joint_histogram(ta, tb, spatial_dims=2, mask=shifted)
    assert all(torch.equal(u, v) for u, v in zip(got, res[:3]))
    for i in range(7):
        one = T.joint_histogram(ta[i], tb[i], mask=tm[i])
        assert torch.equal(one[0], res[0][i]) and torch.equal(one[1], res[1][i]) and torch.equal(one[2], res[2][i])


@gpu
def test_masked_errors_and_psnr():
    from mpgan import transforms as T
    for shape, seed in (((128, 128, 128), 12), ((61, 67, 13), 13), ((3, 1, 97, 101), 14)):
        gen, truth = _display_pair(shape, seed, _head)
        for m in (omm.foreground_mask(truth), _random_mask(shape, seed)):
            tg, tt, tm = _cuda(gen, truth, m)
            s1, s2, c = omm.err_sums(gen, truth, m)
            got = T.error_sums(tg, tt, mask=tm).tolist()
            assert got[2] == c and got[0] == pytest.approx(s1, rel=1e-9) and got[1] == pytest.approx(s2, rel=1e-9)
            assert T.mean_absolute_error(tg, tt, mask=tm) == pytest.approx(s1 / c, rel=1e-9)
            assert T.mean_squared_error(tg, tt, mask=tm) == pytest.approx(s2 / c, rel=1e-9)
            assert T.peak_signal_noise_ratio(tt, tg, data_range=255, mask=tm) == pytest.approx(
                omm.peak_signal_noise_ratio(truth, gen, m, data_range=255.0), rel=1e-9)


@gpu
@pytest.mark.parametrize("kw", [{}, dict(gaussian_weights=True)], ids=["uniform", "gaussian"])
def test_masked_ssim(kw):
    from mpgan import transforms as T
    gen, truth = _display_pair((64, 72, 80), 15, _head)                          # rank 3
    for m in (omm.foreground_mask(truth), _random_mask(gen.shape, 16)):
        tg, tt, tm = _cuda(gen, truth, m)
        got = float(T.structural_similarity(tg, tt, data_range=255, mask=tm, **kw))
        assert abs(got - omm.structural_similarity(gen, truth, m, data_range=255.0, **kw)) <= 1e-7
    a, b = _unit_pair((5, 97, 101), 17)                                          # rank 2, a batch of slices
    m = _random_mask(a.shape, 18, 0.3)
    ta, tb, tm = _cuda(a, b, m)
    got = T.structural_similarity(ta, tb, data_range=2.0, spatial_dims=2, mask=tm, **kw)
    assert tuple(got.shape) == (5,)
    for i in range(5):
        assert abs(float(got[i]) - omm.structural_similarity(a[i], b[i], m[i], data_range=2.0, **kw)) <= 1e-7
        one = T.structural_similarity(ta[i], tb[i], data_range=2.0, mask=tm[i], **kw)
        assert abs(float(one) - float(got[i])) <= 1e-12


@gpu
def test_all_true_mask_gives_the_unmasked_results():
    from mpgan import transforms as T
    gen, truth = _display_pair((3, 40, 41, 43), 19)
    tg, tt = _cuda(gen, truth)
    ones = torch.ones(tg.shape, dtype=torch.bool, device="cuda")
    plain, masked = T.joint_histogram(tg, tt), T.joint_histogram(tg, tt, mask=ones)
    assert all(torch.equal(u, v) for u, v in zip(plain, masked))
    assert _same(T.mutual_information(tg, tt), T.mutual_information(tg, tt, mask=ones))
    assert _same(T.normalized_mutual_information(tg, tt), T.normalized_mutual_information(tg, tt, mask=ones))
    s, sm = T.error_sums(tg, tt).tolist(), T.error_sums(tg, tt, mask=ones).tolist()
    assert sm[2] == gen.size and all(abs(u - v) <= 1e-12 * abs(u) for u, v in zip(s, sm[:2]))
    for kw in ({}, dict(gaussian_weights=True)):
        u = T.structural_similarity(tg, tt, data_range=255, **kw)
        v = T.structural_similarity(tg, tt, data_range=255, mask=ones.to(torch.uint8), **kw)
        assert torch.all((u - v).abs() <= 1e-12 * u.abs())


@gpu
def test_non_finite_outside_the_mask_and_empty_masks():
    from mpgan import transforms as T
    gen, truth = _unit_pair((4, 40, 44), 20)
    m = np.zeros(gen.shape, bool)
    m[:, 10:30, 12:34] = True
    bad = gen.copy()
    bad[:, 0, 0], bad[:, 39, 1], bad[:, 2, 43] = np.nan, np.inf, -np.inf       # outside the mask, beyond every window
    bad[0, 9, 20] = np.nan                                                    # next to the mask: read by SSIM windows
    m[3] = False                                                              # item 3: an empty mask
    tg, tt, tm = _cuda(bad, truth, m)
    counts, e1, e2 = T.joint_histogram(tg, tt, spatial_dims=2, mask=tm)
    mi = T.mutual_information(tg, tt, spatial_dims=2, mask=tm)
    ssim = T.structural_similarity(tg, tt, data_range=2.0, spatial_dims=2, mask=tm)
    for i in (1, 2):
        assert torch.isfinite(mi[i]) and torch.isfinite(ssim[i]) and torch.isfinite(e1[i]).all()
        # against the clean image: scipy's running-sum filter in the oracle would carry a NaN along its row into
        # windows that do not contain it; no window around a masked centre does
        assert abs(float(ssim[i]) - omm.structural_similarity(gen[i], truth[i], m[i], data_range=2.0)) <= 1e-7
        one = T.joint_histogram(tg[i], tt[i], mask=tm[i])
        assert torch.equal(one[0], counts[i]) and torch.equal(one[1], e1[i])
    assert torch.isfinite(mi[0]) and torch.isnan(ssim[0])                     # the window rule of SSIM
    assert torch.all(counts[3] == 0) and torch.isnan(e1[3]).all() and torch.isnan(e2[3]).all()
    assert torch.isnan(mi[3]) and torch.isnan(ssim[3])
    assert math.isfinite(T.mean_absolute_error(tg[1:3], tt[1:3], mask=tm[1:3]))
    none = torch.zeros_like(tm)
    assert math.isnan(T.mean_absolute_error(tg, tt, mask=none)) and math.isnan(T.mean_squared_error(tg, tt, mask=none))
    assert math.isnan(T.peak_signal_noise_ratio(tt, tg, data_range=2.0, mask=none))
    _check_mi(gen[1:3], truth[1:3], m[1:3], spatial_dims=2)


@gpu
def test_repetition_batching_and_graph_replay_change_no_bit():
    from mpgan import transforms as T
    gen, truth = _display_pair((4, 40, 41, 43), 21, _head)
    tg, tt = _cuda(gen, truth)
    tm = T.foreground_mask(tt)
    thr = T.otsu_threshold(tt)
    base = T.joint_histogram(tg, tt, mask=tm)
    base_mi = T.mutual_information(tg, tt, mask=tm)
    base_ssim = T.structural_similarity(tg, tt, data_range=255, mask=tm)
    for i in range(4):
        assert _same(T.otsu_threshold(tt[i]), thr[i]) and torch.equal(T.foreground_mask(tt[i]), tm[i])
        assert torch.equal(T.joint_histogram(tg[i], tt[i], mask=tm[i])[0], base[0][i])
        assert _same(T.mutual_information(tg[i], tt[i], mask=tm[i]), base_mi[i])
    for _ in range(3):
        assert _same(T.otsu_threshold(tt), thr) and torch.equal(T.foreground_mask(tt), tm)
        assert all(torch.equal(u, v) for u, v in zip(T.joint_histogram(tg, tt, mask=tm), base))
        assert _same(T.mutual_information(tg, tt, mask=tm), base_mi)
    sg, st = tg.clone(), tt.clone()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out_thr = T.otsu_threshold(st)
        out_m = T.foreground_mask(st)
        out = T.joint_histogram(sg, st, mask=out_m)
        out_mi = T.mutual_information(sg, st, mask=out_m)
        out_ssim = T.structural_similarity(sg, st, data_range=255, mask=out_m)
    for _ in range(2):
        for t in (out_thr, out_mi, out_ssim, *out):
            t.fill_(7)
        out_m.fill_(False)
        g.replay()
        torch.cuda.synchronize()
        assert _same(out_thr, thr) and torch.equal(out_m, tm) and _same(out_mi, base_mi)
        assert all(torch.equal(u, v) for u, v in zip(out, base))
        assert torch.all((out_ssim - base_ssim).abs() <= 1e-12)
    sg.copy_(torch.flip(tg, [0]))
    st.copy_(torch.flip(tt, [0]))
    g.replay()
    assert _same(out_thr, torch.flip(thr, [0])) and _same(out_mi, torch.flip(base_mi, [0]))


@gpu
def test_evaluate_with_a_foreground_mask_of_a_generator_output():
    import mpgan
    from mpgan import inference
    from mpgan import transforms as T
    torch.manual_seed(0)
    model = mpgan.GAN(1, 64, 64, precision="fp32").cuda().freeze()
    t1 = torch.from_numpy(_unit_pair((12, 1, 64, 64), 22)[1]).cuda()
    gen = inference.to_display_range(inference.infer_volume(model, t1))
    truth = inference.to_display_range(torch.from_numpy(_display_pair((12, 1, 64, 64), 23, _head)[1]).cuda())
    m = T.foreground_mask(truth)
    assert m.shape == truth.shape and 0 < m.float().mean() < 1
    plain = inference.evaluate(gen, truth, data_range=255, mi_bins=100)
    # mask=None is the unmasked path: MI / NMI are fixed-order sums (bit for bit); MAE, MSE, PSNR and SSIM end in fp64
    # atomics whose order varies run to run, so they agree to 1e-12 (the unmasked tests' tolerance)
    again = inference.evaluate(gen, truth, data_range=255, mi_bins=100, mask=None)
    assert again.keys() == plain.keys() and again["mi"] == plain["mi"] and again["nmi"] == plain["nmi"]
    assert all(abs(again[k] - plain[k]) <= 1e-12 * abs(plain[k]) for k in ("mae", "mse", "psnr"))
    assert abs(again["ssim"] - plain["ssim"]) <= 1e-12
    res = inference.evaluate(gen, truth, data_range=255, mi_bins=100, mask=m)
    assert res.keys() == plain.keys()
    g, t, mm = gen.cpu().numpy()[:, 0], truth.cpu().numpy()[:, 0], m.cpu().numpy()[:, 0]   # the stack is one volume
    assert res["mae"] == pytest.approx(omm.mean_absolute_error(g, t, mm), rel=1e-9)
    assert res["mse"] == pytest.approx(omm.mean_squared_error(g, t, mm), rel=1e-9)
    assert res["psnr"] == pytest.approx(omm.peak_signal_noise_ratio(t, g, mm, data_range=255.0), rel=1e-9)
    assert abs(res["ssim"] - omm.structural_similarity(g, t, mm, data_range=255.0)) <= 1e-7
    ref = omi.entropies(omm.joint_histogram(g, t, mm, 100)[0])
    assert abs(res["mi"] - ref[3]) <= 1e-12 * (ref[0] + ref[1]) and abs(res["nmi"] - ref[4]) <= 1e-12 * ref[4]
    assert inference.evaluate(gen, truth, mask=m).keys() == {"mae", "mse"}
