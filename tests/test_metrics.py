"""SSIM and PSNR of generated-vs-true volumes (scikit-image ``structural_similarity`` / ``peak_signal_noise_ratio``,
psnr_ssim_metric.py:88-95; SURVEY.md section 8f row N5).

CPU tests pin the numpy/scipy oracle (oracle/metrics.py) against the definition evaluated window by window and
against known answers, and check that every argument error is raised before the device is touched; ``-m gpu`` tests
compare ``mpgan_ssim_sums`` with the oracle to 1e-7 on the mean SSIM."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import metrics as om
from oracle import transforms as ot

gpu = pytest.mark.gpu
WINDOWS = [dict(gaussian_weights=g, use_sample_covariance=c) for g in (False, True) for c in (True, False)]


def _volume(shape, seed, background=0.4):
    """Synthetic MRI-like volume: positive intensities with a large exactly-zero background."""
    rng = np.random.RandomState(seed)
    v = rng.gamma(2.0, 150.0, size=shape).astype(np.float32)
    v[rng.rand(*shape) < background] = 0.0
    return v


def _display_pair(shape, seed):
    """(generated, truth) on the display range 0..255 (integers): the truth, and a noisy copy of it."""
    v = _volume(shape, seed)
    noise = np.random.RandomState(seed + 100).normal(1.0, 0.2, size=shape).astype(np.float32)
    return ot.to_display_range(v * noise), ot.to_display_range(v)


def _taps(win, gaussian_weights, sigma):
    if not gaussian_weights:
        return np.full(win, 1.0 / win)
    t = np.arange(win) - win // 2
    k = np.exp(-0.5 * t * t / sigma ** 2)
    return k / k.sum()


def _brute_force_ssim_map(x, y, R, win, gaussian_weights, sigma, use_sample_covariance, K1=0.01, K2=0.03):
    """S at every interior voxel from the window's own moments: plain means and ddof-1 / ddof-0 (co)variances for the
    uniform window; weighted population moments times NP / (NP - 1) for the Gaussian one, as scikit-image does."""
    x, y = x.astype(np.float64), y.astype(np.float64)
    nd, n_win = x.ndim, win ** x.ndim
    c1, c2 = (K1 * R) ** 2, (K2 * R) ** 2
    t = _taps(win, gaussian_weights, sigma)
    wts = t
    for _ in range(nd - 1):
        wts = np.multiply.outer(wts, t)
    out = np.empty(tuple(s - win + 1 for s in x.shape))
    for idx in np.ndindex(*out.shape):
        sl = tuple(slice(i, i + win) for i in idx)
        px, py = x[sl], y[sl]
        if gaussian_weights:
            mx, my = (wts * px).sum(), (wts * py).sum()
            norm = n_win / (n_win - 1) if use_sample_covariance else 1.0
            vx = norm * (wts * (px - mx) ** 2).sum()
            vy = norm * (wts * (py - my) ** 2).sum()
            vxy = norm * (wts * (px - mx) * (py - my)).sum()
        else:
            ddof = 1 if use_sample_covariance else 0
            mx, my = px.mean(), py.mean()
            vx, vy = px.var(ddof=ddof), py.var(ddof=ddof)
            vxy = ((px - mx) * (py - my)).sum() / (n_win - ddof)
        out[idx] = ((2 * mx * my + c1) * (2 * vxy + c2)) / ((mx * mx + my * my + c1) * (vx + vy + c2))
    return out


# ------------------------------------------------------------------------------------------------- oracle (CPU)
@pytest.mark.parametrize("shape,sigma", [((13, 17), 1.5), ((9, 10, 11), 0.8)])
@pytest.mark.parametrize("kw", WINDOWS)
def test_oracle_ssim_matches_the_windowed_definition(shape, sigma, kw):
    rng = np.random.RandomState(len(shape))
    x = rng.rand(*shape) * 4.0 - 1.0
    y = 0.6 * x + 0.4 * (rng.rand(*shape) * 2.0 - 1.0)
    win = om.ssim_win_size(None, kw["gaussian_weights"], sigma)
    assert win == (7 if not kw["gaussian_weights"] else 2 * int(3.5 * sigma + 0.5) + 1)
    mssim, s = om.structural_similarity(x, y, data_range=2.0, sigma=sigma, full=True, **kw)
    ref = _brute_force_ssim_map(x, y, 2.0, win, kw["gaussian_weights"], sigma, kw["use_sample_covariance"])
    pad = (win - 1) // 2
    np.testing.assert_allclose(s[(slice(pad, -pad),) * len(shape)], ref, rtol=0, atol=1e-12)
    assert abs(mssim - ref.mean()) <= 1e-12


def test_oracle_known_answers():
    x = _volume((12, 13, 14), 0)
    for gw in (False, True):
        assert om.structural_similarity(x, x.copy(), data_range=255.0, gaussian_weights=gw) == 1.0
    a, b, R = 3.0, 7.5, 255.0
    c1 = (0.01 * R) ** 2
    const = om.structural_similarity(np.full((9, 9, 9), a), np.full((9, 9, 9), b), data_range=R)
    assert abs(const - (2 * a * b + c1) / (a * a + b * b + c1)) <= 1e-12
    y = x.astype(np.float64) + 2.0
    assert om.peak_signal_noise_ratio(x, y, data_range=255.0) == pytest.approx(10 * np.log10(255.0 ** 2 / 4.0), rel=1e-12)
    assert om.peak_signal_noise_ratio(x, x, data_range=255.0) == float("inf")


def test_arguments_are_validated_before_the_device():
    from mpgan import inference
    from mpgan import transforms as T
    x, y = torch.zeros(4, 20, 20, 20), torch.zeros(4, 20, 20, 20)
    bad = [dict(), dict(data_range=0), dict(data_range=-1.0), dict(data_range=float("nan")),
           dict(data_range=1.0, win_size=8), dict(data_range=1.0, win_size=1), dict(data_range=1.0, win_size=17),
           dict(data_range=1.0, win_size=21), dict(data_range=1.0, spatial_dims=1), dict(data_range=1.0, spatial_dims=4),
           dict(data_range=1.0, gaussian_weights=True, sigma=2.2), dict(data_range=1.0, gaussian_weights=True, sigma=0.0),
           dict(data_range=1.0, gaussian_weights=True, win_size=7), dict(data_range=1.0, K1=-0.01)]
    for kw in bad:
        with pytest.raises(ValueError):
            T.structural_similarity(x, y, **kw)
    with pytest.raises(ValueError):                    # window larger than a spatial extent
        T.structural_similarity(torch.zeros(6, 20, 20), torch.zeros(6, 20, 20), data_range=1.0)
    with pytest.raises(ValueError):
        T.structural_similarity(torch.zeros(3, 1, 20, 9), torch.zeros(3, 1, 20, 9), data_range=1.0, gaussian_weights=True,
                                spatial_dims=2)
    with pytest.raises(ValueError):                    # shape mismatch
        T.structural_similarity(x, y[:, :, :, :19], data_range=1.0)
    with pytest.raises(ValueError):
        T.structural_similarity(torch.zeros(20), torch.zeros(20), data_range=1.0)
    for kw in (dict(), dict(data_range=0.0)):
        with pytest.raises(ValueError):
            T.peak_signal_noise_ratio(x, y, **kw)
    with pytest.raises(ValueError):
        T.peak_signal_noise_ratio(x, y[:1], data_range=1.0)
    with pytest.raises(ValueError):
        inference.evaluate(x, y, data_range=-255)
    # valid arguments on CPU tensors: the library's no-fallback error
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.structural_similarity(x, y, data_range=1.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.structural_similarity(x[:, 0], y[:, 0], data_range=1.0, spatial_dims=2, gaussian_weights=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.peak_signal_noise_ratio(x, y, data_range=1.0)


def test_c_abi_rejects_bad_windows_and_shapes():
    from mpgan import _lib
    lib = _lib.load()
    taps = (ctypes.c_double * 15)()
    p = 256   # never dereferenced: the checks come first

    def call(rank, items, d, h, w, win):
        return lib.mpgan_ssim_sums(p, p, rank, items, d, h, w, taps, win, 1.0, 1.0, 1.0, p, None)

    assert call(4, 1, 16, 16, 16, 7) == -1 and "rank" in _lib.last_error()
    assert call(3, 1, 16, 16, 16, 8) == -2 and "window" in _lib.last_error()
    assert call(3, 1, 16, 16, 16, 17) == -2
    assert call(3, 1, 6, 16, 16, 7) == -1 and "interior" in _lib.last_error()
    assert call(2, 1, 2, 16, 16, 7) == -1
    assert call(2, 0, 1, 16, 16, 7) == -1


# ------------------------------------------------------------------------------------------------- CUDA kernel
def _check_against_oracle(a, b, R, spatial_dims, kw, tol=1e-7):
    from mpgan import transforms as T
    got = T.structural_similarity(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda(), data_range=R,
                                  spatial_dims=spatial_dims, **kw)
    lead = a.shape[:a.ndim - spatial_dims]
    assert got.dtype == torch.float64 and got.is_cuda and tuple(got.shape) == lead
    got = got.cpu().numpy().reshape(-1)
    ia, ib = a.reshape((-1,) + a.shape[a.ndim - spatial_dims:]), b.reshape((-1,) + b.shape[b.ndim - spatial_dims:])
    for i in range(ia.shape[0]):
        ref = om.structural_similarity(ia[i], ib[i], data_range=R, **kw)
        assert abs(got[i] - ref) <= tol, (i, got[i], ref)
    return got


@gpu
@pytest.mark.parametrize("kw", WINDOWS)
def test_ssim_128_cube_display_range(kw):
    gen, truth = _display_pair((128, 128, 128), 1)
    _check_against_oracle(gen, truth, 255.0, 3, kw)


@gpu
@pytest.mark.parametrize("kw", WINDOWS)
def test_ssim_ragged_tiles(kw):
    gen, truth = _display_pair((61, 67, 13), 2)          # interior 55 x 61 x 7 (uniform), 51 x 57 x 3 (Gaussian)
    _check_against_oracle(gen, truth, 255.0, 3, kw)


@gpu
@pytest.mark.parametrize("kw", WINDOWS)
def test_ssim_2d_slice_batch_and_batching_is_invisible(kw):
    from mpgan import transforms as T
    rng = np.random.RandomState(3)
    truth = (rng.rand(5, 1, 300, 301) * 2 - 1).astype(np.float32)
    gen = np.clip(truth + rng.normal(0, 0.3, truth.shape), -1, 1).astype(np.float32)
    got = _check_against_oracle(gen, truth, 2.0, 2, kw)
    for i in range(5):
        one = T.structural_similarity(torch.from_numpy(gen[i, 0]).cuda(), torch.from_numpy(truth[i, 0]).cuda(),
                                      data_range=2.0, **kw)
        assert one.dim() == 0 and abs(float(one) - got[i]) <= 1e-12


@gpu
def test_ssim_3d_batching_is_invisible():
    from mpgan import transforms as T
    pairs = [_display_pair((24, 40, 50), s) for s in (4, 5, 6)]
    gen = torch.from_numpy(np.stack([p[0] for p in pairs])).cuda()
    truth = torch.from_numpy(np.stack([p[1] for p in pairs])).cuda()
    for gw in (False, True):
        batch = T.structural_similarity(gen, truth, data_range=255.0, gaussian_weights=gw)
        assert tuple(batch.shape) == (3,)
        for i in range(3):
            one = T.structural_similarity(gen[i], truth[i], data_range=255.0, gaussian_weights=gw)
            assert abs(float(one) - float(batch[i])) <= 1e-12


@gpu
def test_ssim_known_answers_on_device():
    from mpgan import transforms as T
    gen, _ = _display_pair((40, 50, 60), 7)
    x = torch.from_numpy(gen).cuda()
    for gw in (False, True):
        assert float(T.structural_similarity(x, x.clone(), data_range=255.0, gaussian_weights=gw)) == 1.0
        assert float(T.structural_similarity(x[0], x[0].clone(), data_range=255.0, gaussian_weights=gw)) == 1.0
    a, b, R = 3.0, 7.5, 255.0
    c1 = (0.01 * R) ** 2
    for shape, sd in (((20, 21, 22), 3), ((2, 30, 31), 2)):
        s = T.structural_similarity(torch.full(shape, a, device="cuda"), torch.full(shape, b, device="cuda"),
                                    data_range=R, spatial_dims=sd)
        assert torch.all((s - (2 * a * b + c1) / (a * a + b * b + c1)).abs() <= 1e-12)
    assert T.peak_signal_noise_ratio(x, x.clone(), data_range=255.0) == float("inf")


@gpu
def test_evaluate_psnr_and_ssim():
    from mpgan import inference, transforms as T
    gen, truth = _display_pair((20, 64, 64), 8)
    g = torch.from_numpy(gen).cuda().unsqueeze(1)              # (S, 1, H, W): a stack of slices
    t = torch.from_numpy(truth).cuda().unsqueeze(1)
    plain = inference.evaluate(g, t)
    assert set(plain) == {"mae", "mse"}
    s = T.error_sums(g, t).tolist()
    assert plain == {"mae": s[0] / g.numel(), "mse": s[1] / g.numel()}
    m = inference.evaluate(g, t, data_range=255)
    assert set(m) == {"mae", "mse", "psnr", "ssim"} and m["mae"] == plain["mae"] and m["mse"] == plain["mse"]
    assert m["psnr"] == pytest.approx(om.peak_signal_noise_ratio(truth, gen, data_range=255.0), rel=1e-9)
    assert m["psnr"] == pytest.approx(T.peak_signal_noise_ratio(t, g, data_range=255), rel=1e-12)
    assert abs(m["ssim"] - om.structural_similarity(gen, truth, data_range=255.0)) <= 1e-7   # the stacked volume
    vols = [_display_pair((16, 24, 28), s) for s in (9, 10)]     # (S, 1, D, H, W): mean of the volume SSIMs
    g5 = torch.from_numpy(np.stack([v[0] for v in vols])).cuda().unsqueeze(1)
    t5 = torch.from_numpy(np.stack([v[1] for v in vols])).cuda().unsqueeze(1)
    m5 = inference.evaluate(g5, t5, data_range=255)
    ref = np.mean([om.structural_similarity(v[0], v[1], data_range=255.0) for v in vols])
    assert abs(m5["ssim"] - ref) <= 1e-7


def _oracle_by_slabs(a, b, R, win, slab=32, **kw):
    """The oracle's mean SSIM of a large volume from overlapping d-slabs: each slab of slab + win - 1 planes holds the
    complete windows of `slab` output planes, so the interior values are the same as over the whole volume."""
    od = a.shape[0] - win + 1
    total = 0.0
    for z0 in range(0, od, slab):
        n = min(slab, od - z0)
        total += n * om.structural_similarity(a[z0:z0 + n + win - 1], b[z0:z0 + n + win - 1], data_range=R, **kw)
    return total / od


@gpu
@pytest.mark.parametrize("gaussian_weights", [False, True])
def test_ssim_volume_larger_than_l2(gaussian_weights):
    """BASELINE config 5's 256 x 512 x 512 volume: 536 MB of inputs, more than the B200's L2."""
    from mpgan import transforms as T
    gen, truth = _display_pair((256, 512, 512), 11)
    got = float(T.structural_similarity(torch.from_numpy(gen).cuda(), torch.from_numpy(truth).cuda(), data_range=255.0,
                                        gaussian_weights=gaussian_weights))
    win = om.ssim_win_size(None, gaussian_weights, 1.5)
    ref = _oracle_by_slabs(gen, truth, 255.0, win, gaussian_weights=gaussian_weights)
    assert abs(got - ref) <= 1e-7
