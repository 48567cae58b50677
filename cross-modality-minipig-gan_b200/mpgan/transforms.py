"""Device-side intensity transforms and volume metrics (SURVEY.md section 8f, rows N1 / N2 / N5).

Mirrors the interface of the MONAI 0.4.0 transforms the reference applies either side of the generator:
``ScaleIntensityRangePercentiles(lower, upper, b_min, b_max, clip=False, relative=False)`` and its dictionary form
``ScaleIntensityRangePercentilesd(keys, ...)`` (/root/reference/code/GAN/GAN_final.py:386-394,
/root/reference/code/GAN/inferrence.py:152-161), plus torchmetrics' ``MeanAbsoluteError`` / ``MeanSquaredError``
(inferrence.py:170-176, metrics.py:213-218) and scikit-image's ``structural_similarity`` / ``peak_signal_noise_ratio``
(psnr_ssim_metric.py:88-95).  Inputs are CUDA fp32 tensors; everything runs in libmpgan_sm100
(exact radix-select order statistics, fp32 rescale in the reference's operation order) -- there is no CPU path.
"""
import ctypes
import math

import torch

from . import _lib
from .ops import check, ptr, _stream


def _require(x):
    if not (isinstance(x, torch.Tensor) and x.is_cuda):
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    return x.detach().contiguous().float()


def percentile_ranks(n, q):
    """np.percentile's linear interpolation: position q/100*(n-1) between two neighbouring order statistics."""
    pos = (q / 100.0) * (n - 1)
    lo = int(math.floor(pos))
    frac = pos - lo
    hi = lo if frac == 0 else min(lo + 1, n - 1)   # exact percentiles (0, 100, ...) need one order statistic only
    return lo, hi, frac


def order_statistics(x, ranks):
    """The ``ranks``-th smallest values (0-based, exact) of a CUDA fp32 tensor; returns a python list of floats."""
    x = _require(x)
    if x.numel() == 0:
        raise RuntimeError("order_statistics of an empty tensor")
    lib = _lib.require_device()
    out = []
    for i in range(0, len(ranks), 4):
        grp = [int(r) for r in ranks[i:i + 4]]
        if any(r < 0 or r >= x.numel() for r in grp):
            raise RuntimeError(f"rank out of range for {x.numel()} elements: {grp}")
        r_dev = torch.tensor(grp, dtype=torch.int64, device=x.device)
        o_dev = torch.empty(len(grp), dtype=torch.float32, device=x.device)
        nbytes = int(lib.mpgan_order_stats_workspace(len(grp)))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        if all(r in (0, x.numel() - 1) for r in grp):   # 0 / 100 percentiles: one min/max pass
            check(lib.mpgan_minmax(ptr(x), x.numel(), ptr(r_dev), len(grp), ptr(o_dev), ptr(ws), nbytes, _stream()),
                  "mpgan_minmax")
        else:
            check(lib.mpgan_order_stats(ptr(x), x.numel(), ptr(r_dev), len(grp), ptr(o_dev), ptr(ws), nbytes, _stream()),
                  "mpgan_order_stats")
        out += o_dev.tolist()
    return out


def percentiles(x, qs):
    """np.percentile(x, q) (linear interpolation, evaluated in float64, rounded to float32) for each q."""
    n = x.numel()
    spec = [percentile_ranks(n, q) for q in qs]
    ranks = sorted({r for lo, hi, _ in spec for r in (lo, hi)})
    vals = dict(zip(ranks, order_statistics(x, ranks)))
    res = []
    for lo, hi, frac in spec:
        v = vals[lo] + (vals[hi] - vals[lo]) * frac
        res.append(float(torch.tensor(v, dtype=torch.float64).float()))
    return res


def rescale_intensity(x, a_min, a_max, b_min, b_max, clip=None, round_half_even=False, out_dtype=torch.float32):
    """MONAI ScaleIntensityRange arithmetic in fp32; ``clip`` = (lo, hi) or None."""
    x = _require(x)
    lib = _lib.require_device()
    if out_dtype not in (torch.float32, torch.float16):
        raise RuntimeError("rescale_intensity writes float32 or float16")
    y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    lo, hi = clip if clip is not None else (0.0, 0.0)
    check(lib.mpgan_rescale_intensity(ptr(x), x.numel(), float(a_min), float(a_max), float(b_min), float(b_max),
                                      0 if clip is None else 1, float(lo), float(hi), 1 if round_half_even else 0,
                                      0 if out_dtype == torch.float32 else 2, ptr(y), _stream()),
          "mpgan_rescale_intensity")
    return y


class ScaleIntensityRangePercentiles:
    """monai.transforms.ScaleIntensityRangePercentiles (0.4.0) on a CUDA tensor."""

    def __init__(self, lower, upper, b_min, b_max, clip=False, relative=False):
        if not (0.0 <= lower <= 100.0 and 0.0 <= upper <= 100.0):
            raise ValueError("Percentiles must be in the range [0, 100]")
        self.lower, self.upper, self.b_min, self.b_max, self.clip, self.relative = lower, upper, b_min, b_max, clip, relative

    def __call__(self, img, round_half_even=False, out_dtype=torch.float32):
        a_min, a_max = percentiles(img, [self.lower, self.upper])
        b_min, b_max = self.b_min, self.b_max
        if self.relative:
            b_min = ((self.b_max - self.b_min) * (self.lower / 100.0)) + self.b_min
            b_max = ((self.b_max - self.b_min) * (self.upper / 100.0)) + self.b_min
        return rescale_intensity(img, a_min, a_max, b_min, b_max, clip=(self.b_min, self.b_max) if self.clip else None,
                                 round_half_even=round_half_even, out_dtype=out_dtype)


class ScaleIntensityRangePercentilesd:
    """Dictionary form (keys are transformed independently, like MONAI's MapTransform)."""

    def __init__(self, keys, lower, upper, b_min, b_max, clip=False, relative=False):
        self.keys = [keys] if isinstance(keys, str) else list(keys)
        self.scaler = ScaleIntensityRangePercentiles(lower, upper, b_min, b_max, clip, relative)

    def __call__(self, data):
        d = dict(data)
        for k in self.keys:
            d[k] = self.scaler(d[k])
        return d


def error_sums(a, b):
    """(sum |a-b|, sum (a-b)^2) as a device float64 pair."""
    a, b = _require(a), _require(b)
    if a.shape != b.shape:
        raise RuntimeError(f"shape mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    lib = _lib.require_device()
    out = torch.zeros(2, dtype=torch.float64, device=a.device)
    check(lib.mpgan_err_sums(ptr(a), ptr(b), a.numel(), ptr(out), _stream()), "mpgan_err_sums")
    return out


def mean_absolute_error(a, b):
    return float(error_sums(a, b)[0]) / max(a.numel(), 1)


def mean_squared_error(a, b):
    return float(error_sums(a, b)[1]) / max(a.numel(), 1)


def _check_data_range(data_range):
    if data_range is None:
        raise ValueError("data_range is required (scikit-image's inference of it from the dtype changed between versions)")
    if not (math.isfinite(data_range) and data_range > 0):
        raise ValueError(f"data_range must be positive and finite, got {data_range}")


def _psnr(mse, data_range):
    return math.inf if mse == 0 else 10.0 * math.log10(data_range ** 2 / mse)


def peak_signal_noise_ratio(image_true, image_test, *, data_range=None):
    """scikit-image ``peak_signal_noise_ratio``: 10 log10(data_range^2 / mse) over the whole tensors (mse from
    ``error_sums``: fp32 differences, squares summed in float64); ``inf`` for identical inputs.  Returns a python float."""
    _check_data_range(data_range)
    if tuple(image_true.shape) != tuple(image_test.shape):
        raise ValueError(f"shape mismatch {tuple(image_true.shape)} vs {tuple(image_test.shape)}")
    return _psnr(mean_squared_error(image_true, image_test), data_range)


_SSIM_MAX_WIN = 15   # largest window the kernel takes (Gaussian: sigma < 15 / 7)


def _ssim_window(win_size, gaussian_weights, sigma):
    """(window length, 1-D taps): scikit-image's uniform window (default 7), or with ``gaussian_weights`` the taps of
    scipy's ``gaussian_filter`` (truncate 3.5), whose length 2 int(3.5 sigma + 0.5) + 1 is then the window."""
    if gaussian_weights:
        if not sigma > 0:
            raise ValueError(f"sigma must be positive, got {sigma}")
        r = int(3.5 * sigma + 0.5)
        if win_size is not None and win_size != 2 * r + 1:
            raise ValueError(f"with gaussian_weights the window is 2 * int(3.5 * sigma + 0.5) + 1 = {2 * r + 1}, "
                             f"not win_size={win_size}")
        win_size = 2 * r + 1
    elif win_size is None:
        win_size = 7
    if win_size != int(win_size) or int(win_size) % 2 == 0 or not 3 <= win_size <= _SSIM_MAX_WIN:
        raise ValueError(f"window size must be odd and in 3..{_SSIM_MAX_WIN}, got {win_size}")
    win = int(win_size)
    if not gaussian_weights:
        return win, [1.0 / win] * win
    r = win // 2
    t = [math.exp(-0.5 / sigma ** 2 * (i - r) ** 2) for i in range(win)]
    s = sum(t)
    return win, [v / s for v in t]


def structural_similarity(im1, im2, *, data_range=None, spatial_dims=None, win_size=None, gaussian_weights=False,
                          sigma=1.5, use_sample_covariance=True, K1=0.01, K2=0.03):
    """scikit-image ``structural_similarity`` (0.18, psnr_ssim_metric.py:88-95) of CUDA tensors, one launch.

    The last ``spatial_dims`` (2 or 3; default ``min(im1.dim(), 3)``) dimensions are spatial, every leading dimension
    indexes independent images: ``(S, 1, H, W)`` with ``spatial_dims=2`` gives S per-slice values.  The window is
    uniform (``win_size``, default 7) or Gaussian (``gaussian_weights``: scipy's taps for ``sigma``, truncate 3.5); the
    result is the mean of the SSIM map over the voxels whose window lies inside the image.  ``data_range`` is required.
    Returns a float64 CUDA tensor of the leading shape (0-d for one image).  Arguments are validated (ValueError)
    before the device is touched."""
    _check_data_range(data_range)
    if K1 < 0 or K2 < 0:
        raise ValueError("K1 and K2 must be non-negative")
    shape = tuple(im1.shape)
    if shape != tuple(im2.shape):
        raise ValueError(f"shape mismatch {shape} vs {tuple(im2.shape)}")
    nd = min(len(shape), 3) if spatial_dims is None else spatial_dims
    if nd not in (2, 3) or len(shape) < nd:
        raise ValueError(f"spatial_dims must be 2 or 3 and at most the tensor rank, got {nd} for shape {shape}")
    win, taps = _ssim_window(win_size, gaussian_weights, sigma)
    lead, spatial = shape[:len(shape) - nd], shape[len(shape) - nd:]
    if any(s < win for s in spatial):
        raise ValueError(f"window size {win} exceeds the image extent {spatial}")
    a, b = _require(im1), _require(im2)
    lib = _lib.require_device()
    items = math.prod(lead)
    out = torch.zeros(items, dtype=torch.float64, device=a.device)
    if items:
        n_win = win ** nd
        cov_norm = n_win / (n_win - 1) if use_sample_covariance else 1.0
        d, h, w = (1,) + spatial if nd == 2 else spatial
        check(lib.mpgan_ssim_sums(ptr(a), ptr(b), nd, items, d, h, w, (ctypes.c_double * win)(*taps), win,
                                  (K1 * data_range) ** 2, (K2 * data_range) ** 2, cov_norm, ptr(out), _stream()),
              "mpgan_ssim_sums")
    return (out / math.prod(s - win + 1 for s in spatial)).reshape(lead)
