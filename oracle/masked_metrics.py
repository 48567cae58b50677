"""TEST INFRASTRUCTURE (oracle): numpy restatement of the foreground-masked metrics and of Otsu's threshold.  Only tests/
and tools/ may import this module.

A mask is a boolean array of the images' shape; voxels outside it never enter a score.  The masked scores are the
existing definitions restricted to the mask (include/mpgan.h pins them):
  * MAE, MSE: sum |a - b|, sum (a - b)^2 over the voxels in the mask (fp32 differences, fp64 sums), over their count;
  * PSNR: 10 log10(data_range^2 / masked MSE);
  * SSIM: the mean of oracle/metrics.py's SSIM map over the interior voxels whose centre is in the mask (the windows
    still read the unmasked neighbours);
  * joint histogram, MI, NMI: oracle/mutual_info.py applied to x[m], y[m].
An empty mask gives NaN scores.

``otsu_threshold`` restates scikit-image's ``threshold_otsu(image, nbins=256)`` algorithm with the precision the header
pins: np.histogram's fp32 edges and counts, fp32 centres, int64 class weights, sequential fp64 cumulative sums, and
np.argmax of the between-class variance.  scikit-image is not installed here and its versions differ in the precision
of these sums, so no parity with a scikit-image version is claimed.
"""
import numpy as np

from . import metrics as om
from . import mutual_info as omi

F32 = np.float32


def err_sums(a, b, m):
    """(sum |a-b|, sum (a-b)^2, voxels) over the mask, the differences in fp32 and the sums in fp64."""
    m = np.asarray(m, dtype=bool)
    d = (np.asarray(a, dtype=F32)[m] - np.asarray(b, dtype=F32)[m]).astype(np.float64)
    return float(np.abs(d).sum()), float((d * d).sum()), int(m.sum())


def mean_absolute_error(a, b, m):
    s1, _, c = err_sums(a, b, m)
    return s1 / c if c else float("nan")


def mean_squared_error(a, b, m):
    _, s2, c = err_sums(a, b, m)
    return s2 / c if c else float("nan")


def peak_signal_noise_ratio(image_true, image_test, m, *, data_range):
    mse = mean_squared_error(image_true, image_test, m)
    if np.isnan(mse):
        return float("nan")
    return float("inf") if mse == 0 else float(10 * np.log10(data_range ** 2 / mse))


def structural_similarity(im1, im2, m, *, data_range, **kw):
    """Mean of the SSIM map S over the interior voxels whose centre is in the mask: s[crop][m[crop]].mean()."""
    _, s = om.structural_similarity(im1, im2, data_range=data_range, full=True, **kw)
    pad = (om.ssim_win_size(kw.get("win_size"), kw.get("gaussian_weights", False), kw.get("sigma", 1.5)) - 1) // 2
    crop = (slice(pad, -pad),) * s.ndim
    sel = s[crop][np.asarray(m, dtype=bool)[crop]]
    return float(sel.mean()) if sel.size else float("nan")


def joint_histogram(x, y, m, bins=100):
    """np.histogramdd([x[m], y[m]], bins): (counts, edges1, edges2)."""
    m = np.asarray(m, dtype=bool)
    return omi.joint_histogram(np.asarray(x, dtype=F32)[m], np.asarray(y, dtype=F32)[m], bins)


def otsu_histogram(x, bins=256):
    """(int64 counts, fp32 edges) of np.histogram(x, bins) for a finite, non-constant fp32 image: the edges of
    oracle/mutual_info.histogram_edges and searchsorted bins with the last bin closed."""
    x = np.asarray(x, dtype=F32).ravel()
    e = omi.histogram_edges(x.min(), x.max(), bins)
    return np.histogram(x, bins=e)[0].astype(np.int64), e


def otsu_threshold(x, bins=256):
    """Otsu's threshold of one fp32 image (include/mpgan.h): NaN for a non-finite extreme, the value for a constant
    image, else the centre of the first split of largest between-class variance."""
    x = np.asarray(x, dtype=F32)
    lo, hi = x.min(), x.max()
    if not (np.isfinite(lo) and np.isfinite(hi)):
        return F32(np.nan)
    if lo == hi:
        return F32(lo)
    counts, e = otsu_histogram(x, bins)
    c = ((e[:-1] + e[1:]).astype(F32) / F32(2)).astype(F32)
    w1 = np.cumsum(counts)
    w2 = np.cumsum(counts[::-1])[::-1]
    hc = counts.astype(np.float64) * c.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        mean1 = np.cumsum(hc) / w1
        mean2 = (np.cumsum(hc[::-1]) / w2[::-1])[::-1]
        d = mean1[:-1] - mean2[1:]
        var = (w1[:-1] * w2[1:]).astype(np.float64) * (d * d)
    return c[int(np.argmax(var))]


def otsu_thresholds(x, spatial_dims=None):
    """otsu_threshold of every leading index (the last ``spatial_dims``, default min(ndim, 3), dims are spatial)."""
    x = np.asarray(x, dtype=F32)
    nd = spatial_dims or min(x.ndim, 3)
    lead = x.shape[:x.ndim - nd]
    flat = x.reshape((-1,) + x.shape[x.ndim - nd:])
    return np.array([otsu_threshold(v) for v in flat], dtype=F32).reshape(lead)


def foreground_mask(x, spatial_dims=None):
    """x > its Otsu threshold, per leading index."""
    x = np.asarray(x, dtype=F32)
    t = otsu_thresholds(x, spatial_dims)
    nd = spatial_dims or min(x.ndim, 3)
    return x > t.reshape(t.shape + (1,) * nd)
