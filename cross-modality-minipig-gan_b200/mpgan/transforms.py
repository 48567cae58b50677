"""Device-side intensity transforms and volume metrics (SURVEY.md section 8f, rows N1 / N2 / N5).

Mirrors the interface of the MONAI 0.4.0 transforms the reference applies either side of the generator:
``ScaleIntensityRangePercentiles(lower, upper, b_min, b_max, clip=False, relative=False)`` and its dictionary form
``ScaleIntensityRangePercentilesd(keys, ...)`` (/root/reference/code/GAN/GAN_final.py:386-394,
/root/reference/code/GAN/inferrence.py:152-161), plus torchmetrics' ``MeanAbsoluteError`` / ``MeanSquaredError``
(inferrence.py:170-176, metrics.py:213-218) and scikit-image's ``structural_similarity`` / ``peak_signal_noise_ratio``
(psnr_ssim_metric.py:88-95), and the mutual information the reference reports (``joint_histogram``,
``mutual_information``, ``normalized_mutual_information``: scikit-image's definition).  Inputs are CUDA fp32 tensors;
everything runs in libmpgan_sm100 (exact radix-select order statistics, fp32 rescale in the reference's operation
order) -- there is no CPU path.

Every metric takes an optional ``mask=`` (bool or uint8, the images' shape): the score is then taken over the voxels
where it is non-zero only, and voxels outside it are never read into a sum, even when NaN or inf.  ``otsu_threshold`` /
``foreground_mask`` give the simplest such mask, Otsu's threshold of the true image.  Without ``mask=`` every metric
runs exactly as before.

``label``, ``largest_component``, ``fill_holes``, ``binary_erosion`` and ``binary_dilation`` are scipy.ndimage's
connected components and binary morphology on the device, bit for bit; ``foreground_mask(..., largest_component=True,
fill_holes=True)`` uses them to clean the Otsu mask into a head mask.

``ImageGeometry`` / ``resample`` move images between physical grids with ITK's linear interpolation, the step the
reference's ``ResampleT1T2d`` (code/GAN/transforms.py:79-213) applies before everything above.
"""
import ctypes
import math
import numbers

import numpy as np
import torch

from . import _lib, ops
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


def _mask_of(mask, shape, device):
    """``mask`` validated against images of ``shape`` on ``device`` (ValueError, before the device is touched), as the
    contiguous uint8 tensor the kernels read."""
    if not isinstance(mask, torch.Tensor):
        raise ValueError(f"mask must be a torch tensor, got {type(mask).__name__}")
    if mask.dtype not in (torch.bool, torch.uint8):
        raise ValueError(f"mask must be bool or uint8, got {mask.dtype}")
    if tuple(mask.shape) != tuple(shape):
        raise ValueError(f"mask shape {tuple(mask.shape)} differs from the images' {tuple(shape)}")
    if mask.device != device:
        raise ValueError(f"mask on {mask.device}, images on {device}")
    return mask.detach().contiguous().view(torch.uint8)


def error_sums(a, b, mask=None):
    """(sum |a-b|, sum (a-b)^2) as a device float64 pair; with ``mask``, (sum, sum, voxels) over the voxels in it."""
    m = None if mask is None else _mask_of(mask, a.shape, a.device)
    a, b = _require(a), _require(b)
    if a.shape != b.shape:
        raise RuntimeError(f"shape mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    lib = _lib.require_device()
    if m is not None:
        out = torch.zeros(3, dtype=torch.float64, device=a.device)
        check(lib.mpgan_err_sums_masked(ptr(a), ptr(b), ptr(m), a.numel(), ptr(out), _stream()), "mpgan_err_sums_masked")
        return out
    out = torch.zeros(2, dtype=torch.float64, device=a.device)
    check(lib.mpgan_err_sums(ptr(a), ptr(b), a.numel(), ptr(out), _stream()), "mpgan_err_sums")
    return out


def _masked_mean(s, k):
    """sum / voxels of a masked ``error_sums`` triple ``s``: NaN for an empty mask."""
    return s[k] / s[2] if s[2] else math.nan


def mean_absolute_error(a, b, mask=None):
    if mask is not None:
        return _masked_mean(error_sums(a, b, mask).tolist(), 0)
    return float(error_sums(a, b)[0]) / max(a.numel(), 1)


def mean_squared_error(a, b, mask=None):
    if mask is not None:
        return _masked_mean(error_sums(a, b, mask).tolist(), 1)
    return float(error_sums(a, b)[1]) / max(a.numel(), 1)


def _check_data_range(data_range):
    if data_range is None:
        raise ValueError("data_range is required (scikit-image's inference of it from the dtype changed between versions)")
    if not (math.isfinite(data_range) and data_range > 0):
        raise ValueError(f"data_range must be positive and finite, got {data_range}")


def _psnr(mse, data_range):
    return math.inf if mse == 0 else 10.0 * math.log10(data_range ** 2 / mse)


def peak_signal_noise_ratio(image_true, image_test, *, data_range=None, mask=None):
    """scikit-image ``peak_signal_noise_ratio``: 10 log10(data_range^2 / mse) over the whole tensors (mse from
    ``error_sums``: fp32 differences, squares summed in float64); ``inf`` for identical inputs.  With ``mask``, the mse
    of the voxels in the mask (NaN for an empty mask).  Returns a python float."""
    _check_data_range(data_range)
    if tuple(image_true.shape) != tuple(image_test.shape):
        raise ValueError(f"shape mismatch {tuple(image_true.shape)} vs {tuple(image_test.shape)}")
    return _psnr(mean_squared_error(image_true, image_test, mask), data_range)


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
                          sigma=1.5, use_sample_covariance=True, K1=0.01, K2=0.03, mask=None):
    """scikit-image ``structural_similarity`` (0.18, psnr_ssim_metric.py:88-95) of CUDA tensors, one launch.

    The last ``spatial_dims`` (2 or 3; default ``min(im1.dim(), 3)``) dimensions are spatial, every leading dimension
    indexes independent images: ``(S, 1, H, W)`` with ``spatial_dims=2`` gives S per-slice values.  The window is
    uniform (``win_size``, default 7) or Gaussian (``gaussian_weights``: scipy's taps for ``sigma``, truncate 3.5); the
    result is the mean of the SSIM map over the voxels whose window lies inside the image.  ``data_range`` is required.
    With ``mask`` (bool or uint8, the images' shape) the mean is over those of the voxels whose centre is in the mask
    (NaN for an image with none); the windows still read the voxels around them, so the map itself is unchanged.
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
    m = None if mask is None else _mask_of(mask, shape, im1.device)
    a, b = _require(im1), _require(im2)
    lib = _lib.require_device()
    items = math.prod(lead)
    out = torch.zeros(items, dtype=torch.float64, device=a.device)
    cnt = None if m is None else torch.zeros(items, dtype=torch.float64, device=a.device)
    if items:
        n_win = win ** nd
        cov_norm = n_win / (n_win - 1) if use_sample_covariance else 1.0
        d, h, w = (1,) + spatial if nd == 2 else spatial
        args = (nd, items, d, h, w, (ctypes.c_double * win)(*taps), win, (K1 * data_range) ** 2, (K2 * data_range) ** 2,
                cov_norm, ptr(out))
        if m is None:
            check(lib.mpgan_ssim_sums(ptr(a), ptr(b), *args, _stream()), "mpgan_ssim_sums")
        else:
            check(lib.mpgan_ssim_sums_masked(ptr(a), ptr(b), ptr(m), *args, ptr(cnt), _stream()),
                  "mpgan_ssim_sums_masked")
    if m is not None:
        return (out / cnt).reshape(lead)
    return (out / math.prod(s - win + 1 for s in spatial)).reshape(lead)


_MI_MAX_BINS = 128          # the kernel's shared-memory histogram: 128 x 128 uint32 = 64 KB
_MI_MAX_VOXELS = 2 ** 31 - 1


def _check_bins(bins):
    if isinstance(bins, bool) or not isinstance(bins, numbers.Integral) or not 2 <= bins <= _MI_MAX_BINS:
        raise ValueError(f"bins must be an integer in 2..{_MI_MAX_BINS}, got {bins!r}")
    return int(bins)


def _mutual_info(im1, im2, bins, spatial_dims, want_edges, mask=None):
    """Validated call of ``mpgan_mutual_info`` (``mpgan_mutual_info_masked`` with a mask): (counts, edges or None,
    out5)."""
    for im in (im1, im2):
        if not isinstance(im, torch.Tensor):
            raise ValueError(f"images must be torch tensors, got {type(im).__name__}")
        if im.dtype != torch.float32:
            raise ValueError(f"images must be float32, got {im.dtype}")
    shape = tuple(im1.shape)
    if shape != tuple(im2.shape):
        raise ValueError(f"shape mismatch {shape} vs {tuple(im2.shape)}")
    if im1.device != im2.device:
        raise ValueError(f"images on different devices: {im1.device} and {im2.device}")
    nd = min(len(shape), 3) if spatial_dims is None else spatial_dims
    if isinstance(nd, bool) or nd not in (2, 3) or len(shape) < nd:
        raise ValueError(f"spatial_dims must be 2 or 3 and at most the tensor rank, got {nd!r} for shape {shape}")
    bins = _check_bins(bins)
    lead, spatial = shape[:len(shape) - nd], shape[len(shape) - nd:]
    n = math.prod(spatial)
    if not 1 <= n <= _MI_MAX_VOXELS:
        raise ValueError(f"an image has 1 .. 2^31 - 1 voxels, got {spatial}")
    m = None if mask is None else _mask_of(mask, shape, im1.device)
    if not (im1.is_cuda and im2.is_cuda):
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    items = math.prod(lead)
    dev = im1.device
    counts = torch.empty(lead + (bins, bins), dtype=torch.int64, device=dev)
    edges = torch.empty(lead + (2, bins + 1), dtype=torch.float32, device=dev) if want_edges else None
    out5 = torch.empty(lead + (5,), dtype=torch.float64, device=dev)
    if items:
        ops.mutual_info(im1.detach().contiguous(), im2.detach().contiguous(), items, n, bins, counts, edges, out5, m)
    return counts, edges, out5


def joint_histogram(im1, im2, *, bins=100, spatial_dims=None, mask=None):
    """The joint histogram ``np.histogramdd([im1.ravel(), im2.ravel()], bins=bins)`` of CUDA fp32 images, computed on
    the device with numpy's fp32 edges and bins (include/mpgan.h states them).

    The last ``spatial_dims`` (2 or 3; default ``min(im1.dim(), 3)``) dimensions are spatial, every leading dimension
    indexes an independent pair, as in ``structural_similarity``.  Returns ``(counts, edges1, edges2)``: int64
    ``(*lead, bins, bins)`` with ``counts[..., i, j]`` the voxels whose im1 value is in bin i and im2 value in bin j,
    and the fp32 ``(*lead, bins + 1)`` edges of each image.  ``bins`` is an integer in 2..128.

    With ``mask`` (bool or uint8, the images' shape) each pair is ``np.histogramdd([im1[m], im2[m]], bins)``: the ranges
    come from the voxels in the mask only, and the others are never read into the histogram.

    numpy raises when an image's min or max is NaN or +-inf; here that pair instead gets NaN edges and all-zero counts
    (no host synchronisation is needed to report it), and the other pairs are unaffected.  So does a pair whose mask is
    empty.  Arguments are validated (ValueError) before the device is touched."""
    counts, edges, _ = _mutual_info(im1, im2, bins, spatial_dims, True, mask)
    return counts, edges[..., 0, :], edges[..., 1, :]


def mutual_information(im1, im2, *, bins=100, spatial_dims=None, mask=None):
    """Mutual information H1 + H2 - H12 in nats from the joint histogram of ``joint_histogram`` (same arguments): the
    entropies of the two marginals and of the joint distribution, p = count / voxels (in the mask), in fp64.  Returns a
    float64 CUDA tensor of the leading shape (0-d for one pair); NaN for a pair holding NaN or +-inf or with an empty
    mask."""
    return _mutual_info(im1, im2, bins, spatial_dims, False, mask)[2][..., 3]


def normalized_mutual_information(im1, im2, *, bins=100, spatial_dims=None, mask=None):
    """scikit-image's ``normalized_mutual_information(im1, im2, bins=bins)``, (H1 + H2) / H12, from the same
    histogram and entropies as ``mutual_information`` (same arguments and result shape).  1 for independent images, 2
    for images that determine each other's bin; NaN when both images are constant (0 / 0), hold NaN or +-inf, or have
    an empty mask."""
    return _mutual_info(im1, im2, bins, spatial_dims, False, mask)[2][..., 4]


_OTSU_MAX_BINS = 256


def _split_images(x, spatial_dims, what):
    """(lead shape, voxels per image) of a float32 tensor whose last ``spatial_dims`` dims are spatial (ValueError)."""
    if not isinstance(x, torch.Tensor):
        raise ValueError(f"{what} takes a torch tensor, got {type(x).__name__}")
    if x.dtype != torch.float32:
        raise ValueError(f"{what} takes float32, got {x.dtype}")
    shape = tuple(x.shape)
    nd = min(len(shape), 3) if spatial_dims is None else spatial_dims
    if isinstance(nd, bool) or nd not in (2, 3) or len(shape) < nd:
        raise ValueError(f"spatial_dims must be 2 or 3 and at most the tensor rank, got {nd!r} for shape {shape}")
    lead, n = shape[:len(shape) - nd], math.prod(shape[len(shape) - nd:])
    if not 1 <= n <= _MI_MAX_VOXELS:
        raise ValueError(f"an image has 1 .. 2^31 - 1 voxels, got {shape[len(shape) - nd:]}")
    return lead, n


def _check_otsu_bins(bins):
    if isinstance(bins, bool) or not isinstance(bins, numbers.Integral) or not 2 <= bins <= _OTSU_MAX_BINS:
        raise ValueError(f"bins must be an integer in 2..{_OTSU_MAX_BINS}, got {bins!r}")
    return int(bins)


def otsu_threshold(x, *, bins=256, spatial_dims=None):
    """Otsu's threshold of every image of a CUDA fp32 tensor: scikit-image's ``threshold_otsu(image, nbins=bins)``
    algorithm with the precision include/mpgan.h pins (no parity with a scikit-image version is claimed).  The last
    ``spatial_dims`` (2 or 3; default ``min(x.dim(), 3)``) dims are spatial, as in ``structural_similarity``.  Returns
    fp32 thresholds of the leading shape (0-d for one image): NaN for an image holding NaN or +-inf, the value itself
    for a constant image.  Arguments are validated (ValueError) before the device is touched."""
    lead, n = _split_images(x, spatial_dims, "otsu_threshold")
    bins = _check_otsu_bins(bins)
    if not x.is_cuda:
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    thr = torch.empty(lead, dtype=torch.float32, device=x.device)
    if thr.numel():
        ops.otsu_threshold(x.detach().contiguous(), thr.numel(), n, bins, thr)
    return thr


def foreground_mask(x, *, threshold=None, bins=256, largest_component=False, fill_holes=False, connectivity=1):
    """The bool mask ``x > threshold`` of a CUDA fp32 tensor, per image (the last ``min(x.dim(), 3)`` dims): the
    simplest foreground mask of an MRI volume, for the metrics' ``mask=``.  ``threshold``: None for
    ``otsu_threshold(x, bins=bins)``, a number, or a float32 tensor of the leading shape on x's device.  A NaN threshold
    gives an empty mask.

    The clean-up that turns it into a head mask runs after the threshold, in this order: ``largest_component`` keeps
    each image's largest connected component (drops noise specks and ghosting in the air), then ``fill_holes`` fills
    the background enclosed by the mask (dark bone and sinuses inside the head), both under the structure of
    ``connectivity`` (see ``label``).  Without either flag the mask is the threshold's alone.  Arguments are validated
    (ValueError) before the device is touched."""
    lead, n = _split_images(x, None, "foreground_mask")
    bins = _check_otsu_bins(bins)
    if isinstance(threshold, torch.Tensor):
        if threshold.dtype != torch.float32 or tuple(threshold.shape) != lead or threshold.device != x.device:
            raise ValueError(f"threshold tensor must be float32 of shape {lead} on {x.device}, got "
                             f"{threshold.dtype} {tuple(threshold.shape)} on {threshold.device}")
    elif threshold is not None and (isinstance(threshold, bool) or not isinstance(threshold, numbers.Real)):
        raise ValueError(f"threshold must be None, a number or a tensor, got {threshold!r}")
    for name, flag in (("largest_component", largest_component), ("fill_holes", fill_holes)):
        if not isinstance(flag, bool):
            raise ValueError(f"{name} must be True or False, got {flag!r}")
    _check_connectivity(connectivity, min(x.dim(), 3))
    if not x.is_cuda:
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    if threshold is None:
        thr = otsu_threshold(x, bins=bins)
    elif isinstance(threshold, torch.Tensor):
        thr = threshold.detach().contiguous()
    else:
        thr = torch.full(lead, float(threshold), dtype=torch.float32, device=x.device)
    out = torch.empty(x.shape, dtype=torch.bool, device=x.device)
    if out.numel():
        ops.threshold_mask(x.detach().contiguous(), thr, thr.numel(), n, out.view(torch.uint8))
        if largest_component:
            out = _mask_op("largest_component", out, connectivity, None)
        if fill_holes:
            out = _mask_op("fill_holes", out, connectivity, None)
    return out


_MORPH_OPS = {"erosion": 0, "dilation": 1}


def _check_connectivity(connectivity, rank):
    if isinstance(connectivity, bool) or not isinstance(connectivity, numbers.Integral) or not 1 <= connectivity <= rank:
        raise ValueError(f"connectivity must be an integer in 1..{rank} (the spatial rank), got {connectivity!r}")
    return int(connectivity)


def _split_mask(mask, spatial_dims, connectivity, what):
    """(lead shape, rank, (d, h, w), connectivity) of a bool / uint8 mask whose last ``spatial_dims`` dims are spatial
    (ValueError, before the device is touched)."""
    if not isinstance(mask, torch.Tensor):
        raise ValueError(f"{what} takes a torch tensor, got {type(mask).__name__}")
    if mask.dtype not in (torch.bool, torch.uint8):
        raise ValueError(f"{what} takes a bool or uint8 mask, got {mask.dtype}")
    shape = tuple(mask.shape)
    nd = min(len(shape), 3) if spatial_dims is None else spatial_dims
    if isinstance(nd, bool) or nd not in (2, 3) or len(shape) < nd:
        raise ValueError(f"spatial_dims must be 2 or 3 and at most the tensor rank, got {nd!r} for shape {shape}")
    lead, spatial = shape[:len(shape) - nd], shape[len(shape) - nd:]
    if not 1 <= math.prod(spatial) <= _MI_MAX_VOXELS:
        raise ValueError(f"an image has 1 .. 2^31 - 1 voxels, got {spatial}")
    return lead, nd, (1,) * (3 - nd) + spatial, _check_connectivity(connectivity, nd)


def _mask_op(name, mask, connectivity, spatial_dims, *extra):
    """Validated ``ops.mask_op``: the bool result of ``name`` for every image of ``mask``."""
    lead, rank, dhw, conn = _split_mask(mask, spatial_dims, connectivity, name)
    if not mask.is_cuda:
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    out = torch.empty(mask.shape, dtype=torch.bool, device=mask.device)
    items = math.prod(lead)
    if items:
        ops.mask_op(name, mask.detach().contiguous().view(torch.uint8), rank, items, dhw, conn, out.view(torch.uint8),
                    *extra)
    return out


def label(mask, *, connectivity=1, spatial_dims=None):
    """Connected components of every image of a CUDA bool / uint8 mask: ``scipy.ndimage.label(mask, structure)`` with
    ``structure = generate_binary_structure(rank, connectivity)``.  The last ``spatial_dims`` (2 or 3; default
    ``min(mask.dim(), 3)``) dims are spatial and every leading index is an independent image, as in ``otsu_threshold``;
    non-zero voxels are "in".  ``connectivity`` 1..rank: 4 or 8 neighbours at rank 2, 6, 18 or 26 at rank 3 (1, scipy's
    default, is face-connected).

    Returns ``(labels, count)``: int32 labels of the mask's shape, 0 in the background and 1..k numbering the components
    in raster order of their first voxel (scipy's numbering exactly), and the int32 count k per image, a CUDA tensor of
    the leading shape (0-d for one image) rather than scipy's python int, so the call never synchronises.  Arguments
    are validated (ValueError) before the device is touched."""
    lead, rank, dhw, conn = _split_mask(mask, spatial_dims, connectivity, "label")
    if not mask.is_cuda:
        raise RuntimeError("mpgan.transforms need CUDA tensors on a B200: there is no CPU fallback")
    labels = torch.empty(mask.shape, dtype=torch.int32, device=mask.device)
    count = torch.empty(lead, dtype=torch.int32, device=mask.device)
    if count.numel():
        ops.label(mask.detach().contiguous().view(torch.uint8), rank, count.numel(), dhw, conn, labels, count)
    return labels, count


def largest_component(mask, *, connectivity=1, spatial_dims=None):
    """The largest connected component of every image of a CUDA bool / uint8 mask (``label``'s images and structure),
    as a bool mask: MONAI's ``KeepLargestConnectedComponent`` step.  Of equal-sized components the one with the lowest
    label wins (``np.argmax(np.bincount(labels)[1:])``; MONAI's tie handling is not claimed).  An empty image stays
    empty."""
    return _mask_op("largest_component", mask, connectivity, spatial_dims)


def fill_holes(mask, *, connectivity=1, spatial_dims=None):
    """``scipy.ndimage.binary_fill_holes(mask, structure)`` of every image of a CUDA bool / uint8 mask (``label``'s
    images and structure), as a bool mask: the mask plus every background component that touches no face of the image.
    At rank 3 an image of depth 1 is all face, so nothing is filled: pass ``spatial_dims=2`` to fill slices."""
    return _mask_op("fill_holes", mask, connectivity, spatial_dims)


def _check_iterations(iterations):
    if isinstance(iterations, bool) or not isinstance(iterations, numbers.Integral) or iterations < 1:
        raise ValueError(f"iterations must be an integer >= 1, got {iterations!r}")
    return int(iterations)


def binary_erosion(mask, *, iterations=1, connectivity=1, spatial_dims=None):
    """``scipy.ndimage.binary_erosion(mask, structure, iterations, border_value=0)`` of every image of a CUDA bool /
    uint8 mask (``label``'s images and structure), as a bool mask: a voxel stays "in" when every voxel of the structure
    around it is, and outside the image counts as "out", so "in" voxels on the faces go.  ``iterations`` >= 1 (scipy's
    "until nothing changes", < 1, is not offered).  An opening is ``binary_dilation(binary_erosion(m))``."""
    return _mask_op("binary_morphology", mask, connectivity, spatial_dims, _MORPH_OPS["erosion"],
                    _check_iterations(iterations))


def binary_dilation(mask, *, iterations=1, connectivity=1, spatial_dims=None):
    """``scipy.ndimage.binary_dilation(mask, structure, iterations, border_value=0)`` of every image of a CUDA bool /
    uint8 mask (``label``'s images and structure), as a bool mask: a voxel is "in" when any voxel of the structure
    around it is.  ``iterations`` >= 1.  A closing is ``binary_erosion(binary_dilation(m))``."""
    return _mask_op("binary_morphology", mask, connectivity, spatial_dims, _MORPH_OPS["dilation"],
                    _check_iterations(iterations))


class ImageGeometry:
    """The physical grid of an image, as ITK describes it: ``size`` (voxels), ``spacing`` (positive), ``origin`` (the
    centre of voxel 0) and ``direction`` (a non-singular rank x rank matrix, identity when None), all in ITK's axis
    order (x, y[, z]).  The rank is ``len(size)`` (2 or 3).  A tensor holding an image on this grid is laid out
    ``[..., z, y, x]`` (``itk.GetArrayFromImage``'s order): ``.shape`` gives that layout.  Bad fields raise ValueError."""

    def __init__(self, size, spacing, origin, direction=None):
        rank = len(size)
        if rank not in (2, 3):
            raise ValueError(f"an image geometry has 2 or 3 axes, got size {tuple(size)}")
        if not all(isinstance(n, numbers.Integral) and not isinstance(n, bool) and n >= 1 for n in size):
            raise ValueError(f"size must be positive integers, got {tuple(size)}")
        if len(spacing) != rank or len(origin) != rank:
            raise ValueError(f"size, spacing and origin need {rank} entries each, got {len(spacing)} and {len(origin)}")
        spacing, origin = tuple(float(s) for s in spacing), tuple(float(o) for o in origin)
        if not all(math.isfinite(s) and s > 0 for s in spacing):
            raise ValueError(f"spacing must be positive and finite, got {spacing}")
        if not all(math.isfinite(o) for o in origin):
            raise ValueError(f"origin must be finite, got {origin}")
        d = np.eye(rank) if direction is None else np.array(direction, dtype=np.float64)
        if d.shape != (rank, rank) or not np.isfinite(d).all():
            raise ValueError(f"direction must be a finite {rank}x{rank} matrix, got {direction!r}")
        if abs(_det(d)) <= 1e-12 * float(np.prod(np.sqrt((d * d).sum(axis=1)))):
            raise ValueError(f"direction must be non-singular, got {d.tolist()}")
        self.size, self.spacing, self.origin = tuple(int(n) for n in size), spacing, origin
        self.direction = d
        self.rank = rank

    @property
    def shape(self):
        """Tensor shape of one image on this grid: ``(z, y, x)`` or ``(y, x)``."""
        return self.size[::-1]

    def index_to_physical(self):
        """fp64 ``D diag(S)``: physical point = origin + this matrix times the ITK index."""
        return self.direction * np.array(self.spacing)[None, :]

    def physical_to_index(self):
        """fp64 ``inverse(D diag(S))``: continuous index = this matrix times (point - origin).  The cofactor formula in
        a fixed operation order, so the kernel and oracle/resample.py see the same bits on every host."""
        return _inverse(self.index_to_physical())

    def __repr__(self):
        return (f"ImageGeometry(size={self.size}, spacing={self.spacing}, origin={self.origin}, "
                f"direction={self.direction.tolist()})")


def _det(a):
    if len(a) == 2:
        return a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]
    return (a[0, 0] * (a[1, 1] * a[2, 2] - a[1, 2] * a[2, 1]) - a[0, 1] * (a[1, 0] * a[2, 2] - a[1, 2] * a[2, 0])
            + a[0, 2] * (a[1, 0] * a[2, 1] - a[1, 1] * a[2, 0]))


def _inverse(a):
    a = [[float(v) for v in r] for r in a]   # python floats: IEEE fp64, one rounding per operation
    n = len(a)
    if n == 2:
        cof = [[a[1][1], -a[1][0]], [-a[0][1], a[0][0]]]
    else:
        cof = [[a[(i + 1) % 3][(j + 1) % 3] * a[(i + 2) % 3][(j + 2) % 3]
                - a[(i + 1) % 3][(j + 2) % 3] * a[(i + 2) % 3][(j + 1) % 3] for j in range(3)] for i in range(3)]
    det = sum(a[0][j] * cof[0][j] for j in range(n))
    inv = np.array([[cof[j][i] / det for j in range(n)] for i in range(n)], dtype=np.float64)
    if det == 0 or not np.isfinite(inv).all():
        raise ValueError(f"index-to-physical matrix {a} is singular")
    return inv


def reference_grid(size=128, fov_mm=256.0, rank=3):
    """The generator's training grid: ``size`` voxels per axis of ``fov_mm / size`` mm, identity direction, origin
    ``-fov_mm / 2`` on every axis.  The defaults (128^3 at 2 mm, origin -128 mm) restate SURVEY.md section 2's summary of
    ResampleT1T2d (code/GAN/transforms.py:140-147): "identity-direction 256 mm grid, origin -size/2"."""
    return ImageGeometry((size,) * rank, (fov_mm / size,) * rank, (-fov_mm / 2.0,) * rank)


_RESAMPLE_MAX_EXTENT = 1 << 22


def _lift3(m, o):
    """(3x3 matrix, 3 origin) of a rank-2 or rank-3 (matrix, origin): z row and column of the identity, z origin 0."""
    m3 = np.eye(3)
    m3[:len(o), :len(o)] = m
    return m3, list(o) + [0.0] * (3 - len(o))


def resample_map(source, target):
    """The 24 fp64 words ``mpgan_resample_linear`` reads: o_out, M_out (row-major), o_in, N_in (row-major), rank-3
    lifted (include/mpgan.h)."""
    m_out, o_out = _lift3(target.index_to_physical(), target.origin)
    n_in, o_in = _lift3(source.physical_to_index(), source.origin)
    return [float(v) for v in (*o_out, *m_out.ravel(), *o_in, *n_in.ravel())]


def resample(image, source, target, *, default_value=0.0):
    """Linear resampling of ``image`` from the ``source`` grid onto the ``target`` grid (ImageGeometry), as ITK 5.1's
    ResampleImageFilter with an IdentityTransform and a LinearInterpolateImageFunction computes it on float pixels:
    target voxels whose continuous source index c satisfies -0.5 <= c < n - 0.5 on every axis are interpolated, the
    others take ``default_value`` (ITK's DefaultPixelValue, 0).  include/mpgan.h states the fp64 arithmetic.  ITK is not
    available to this project's tests: the kernel is checked bit for bit against a numpy restatement of that arithmetic
    (oracle/resample.py), not against ITK, and bit-parity with ITK is not claimed.

    ``image``: ``(*lead, *source.shape)`` CUDA fp32; every leading index is an image of the same geometry, resampled in
    one launch.  Returns ``(*lead, *target.shape)`` fp32.  Arguments are validated (ValueError) before the device is
    touched."""
    if not (isinstance(source, ImageGeometry) and isinstance(target, ImageGeometry)):
        raise ValueError("source and target must be ImageGeometry instances")
    if source.rank != target.rank:
        raise ValueError(f"source rank {source.rank} and target rank {target.rank} differ")
    if not isinstance(image, torch.Tensor):
        raise ValueError(f"image must be a torch tensor, got {type(image).__name__}")
    if image.dtype != torch.float32:
        raise ValueError(f"image must be float32, got {image.dtype}")
    rank = source.rank
    if image.dim() < rank or tuple(image.shape[image.dim() - rank:]) != source.shape:
        raise ValueError(f"image shape {tuple(image.shape)} does not end in the source grid's {source.shape}")
    if max(source.size + target.size) > _RESAMPLE_MAX_EXTENT:
        raise ValueError(f"extents above 2^22: source {source.size}, target {target.size}")
    if not isinstance(default_value, numbers.Real):
        raise ValueError(f"default_value must be a real number, got {default_value!r}")
    if not image.is_cuda:
        raise RuntimeError("mpgan.transforms.resample needs CUDA tensors on a B200: there is no CPU fallback")
    lead = tuple(image.shape[:image.dim() - rank])
    items = math.prod(lead)
    out = torch.empty(lead + target.shape, dtype=torch.float32, device=image.device)
    if items:
        pad = (1,) * (3 - rank)
        ops.resample_linear(image.detach().contiguous(), items, rank, source.size + pad, target.size + pad,
                            resample_map(source, target), float(default_value), out)
    return out
