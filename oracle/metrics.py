"""TEST INFRASTRUCTURE (oracle): numpy/scipy restatement of the image-quality scores the reference evaluates its generator
with.  Only tests/ and tools/ may import this module.

Follows scikit-image ``structural_similarity`` / ``peak_signal_noise_ratio`` (call site
/root/reference/code/GAN/psnr_ssim_metric.py:88-95), restated from scikit-image 0.18's published algorithm with its
defaults: float64 images; the five moments x, y, x*x, y*y, x*y filtered by ``scipy.ndimage.uniform_filter(size=win_size)``
(default 7) or, with ``gaussian_weights``, ``gaussian_filter(sigma, truncate=3.5)`` (window 2 int(3.5 sigma + 0.5) + 1);
sample covariance scaled by NP / (NP - 1), NP = win_size ** ndim; C1 = (K1 R)^2, C2 = (K2 R)^2; the mean of the SSIM map
over the crop of (win_size - 1) // 2 on every side.  ``data_range`` is required: scikit-image's float-dtype default for
it changed between versions.  PSNR = 10 log10(R^2 / mse) with mse in float64.

Parity with scikit-image itself is unpinned (it is not installed here), as it is for MONAI in oracle/transforms.py;
what tests/test_metrics.py pins is this restatement against the definition evaluated window by window, and known
answers.
"""
import numpy as np


def ssim_win_size(win_size=None, gaussian_weights=False, sigma=1.5):
    """scikit-image's window: 7 by default, 2 int(3.5 sigma + 0.5) + 1 (gaussian_filter's support) with gaussian_weights."""
    if win_size is not None:
        return win_size
    return 2 * int(3.5 * sigma + 0.5) + 1 if gaussian_weights else 7


def structural_similarity(im1, im2, *, data_range, win_size=None, gaussian_weights=False, sigma=1.5,
                          use_sample_covariance=True, K1=0.01, K2=0.03, full=False):
    """Mean SSIM of one 2-D or 3-D image pair; ``full=True`` also returns the SSIM map (uncropped)."""
    from scipy.ndimage import gaussian_filter, uniform_filter
    x, y = np.asarray(im1, dtype=np.float64), np.asarray(im2, dtype=np.float64)
    win_size = ssim_win_size(win_size, gaussian_weights, sigma)
    if gaussian_weights:
        def filt(a):
            return gaussian_filter(a, sigma=sigma, truncate=3.5)
    else:
        def filt(a):
            return uniform_filter(a, size=win_size)
    n_win = win_size ** x.ndim
    cov_norm = n_win / (n_win - 1) if use_sample_covariance else 1.0
    ux, uy = filt(x), filt(y)
    uxx, uyy, uxy = filt(x * x), filt(y * y), filt(x * y)
    vx = cov_norm * (uxx - ux * ux)
    vy = cov_norm * (uyy - uy * uy)
    vxy = cov_norm * (uxy - ux * uy)
    c1, c2 = (K1 * data_range) ** 2, (K2 * data_range) ** 2
    s = ((2 * ux * uy + c1) * (2 * vxy + c2)) / ((ux ** 2 + uy ** 2 + c1) * (vx + vy + c2))
    pad = (win_size - 1) // 2
    mssim = float(s[(slice(pad, -pad),) * x.ndim].mean())
    return (mssim, s) if full else mssim


def peak_signal_noise_ratio(image_true, image_test, *, data_range):
    d = np.asarray(image_true, dtype=np.float64) - np.asarray(image_test, dtype=np.float64)
    mse = float(np.mean(d * d))
    return float("inf") if mse == 0 else float(10 * np.log10(data_range ** 2 / mse))
