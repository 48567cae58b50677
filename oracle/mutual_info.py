"""TEST INFRASTRUCTURE (oracle): numpy/scipy restatement of the mutual information of two images.  Only tests/ and
tools/ may import this module.

The definition is scikit-image's ``skimage.metrics.normalized_mutual_information(image0, image1, bins=100)``: the
joint histogram ``np.histogramdd([image0.ravel(), image1.ravel()], bins=bins)`` with autodetected ranges, and the
entropies of its marginals and of itself from ``scipy.stats.entropy`` (nats).  NMI = (H1 + H2) / H12; plain mutual
information MI = H1 + H2 - H12 comes from the same histogram.  scikit-image is not installed here, so what this module
restates is the numpy/scipy computation that function performs; parity with scikit-image itself is unpinned, and so is
parity with whichever tool wrote the reference's code/eval/*.xml mutual-information values.

``histogram_edges`` restates, in explicit fp32 steps, the edges ``np.histogramdd`` builds for one float32 image (numpy
2.x, NEP 50): that restatement is what include/mpgan.h pins and the kernel computes.
"""
import numpy as np

F32 = np.float32


def outer_range(x):
    """(lo, hi) as np.histogramdd autodetects them: min and max, widened by 0.5 each way in fp32 when equal.
    numpy raises on a range that is not finite; so does this."""
    x = np.asarray(x, dtype=F32)
    lo, hi = x.min(), x.max()
    if not (np.isfinite(lo) and np.isfinite(hi)):
        raise ValueError(f"autodetected range of [{lo}, {hi}] is not finite")
    if lo == hi:
        lo, hi = F32(lo - F32(0.5)), F32(hi + F32(0.5))
    return F32(lo), F32(hi)


def histogram_edges(lo, hi, bins):
    """The bins + 1 fp32 edges of np.linspace(lo, hi, bins + 1, dtype=float32), one rounding per step:
    step = fl(fl(hi - lo) / bins); e_i = fl(fl(i step) + lo) for 0 <= i < bins; e_bins = hi.  (e_0 is lo + 0, which
    turns a minimum of -0.0 into +0.0.)
    When step underflows to 0 (a subnormal range), numpy scales the other way round: e_i = fl(fl(fl(i / bins) delta) + lo)
    with delta = fl(hi - lo)."""
    lo, hi = F32(lo), F32(hi)
    delta = F32(hi - lo)
    step = F32(delta / F32(bins))
    i = np.arange(bins + 1, dtype=F32)
    with np.errstate(under="ignore"):
        y = (i / F32(bins)) * delta if step == 0 else i * step
    e = (y.astype(F32) + lo).astype(F32)
    e[bins] = hi
    return e


def joint_histogram(x, y, bins=100):
    """(counts int64 [bins, bins], edges1, edges2): np.histogramdd of the two flattened float32 images."""
    x, y = np.asarray(x, dtype=F32).ravel(), np.asarray(y, dtype=F32).ravel()
    counts, (e1, e2) = np.histogramdd([x, y], bins=bins)
    return counts.astype(np.int64), e1, e2


def entropies(counts):
    """(H1, H2, H12, MI, NMI) in nats from a joint count matrix: H1 from the row sums, H2 from the column sums, H12 from
    all of it (scipy.stats.entropy normalises each to probabilities).  NMI is NaN when H12 == 0, as numpy's 0 / 0."""
    from scipy.stats import entropy
    c = np.asarray(counts, dtype=np.float64)
    h1, h2, h12 = float(entropy(c.sum(axis=1))), float(entropy(c.sum(axis=0))), float(entropy(c.ravel()))
    with np.errstate(invalid="ignore", divide="ignore"):
        nmi = float(np.float64(h1 + h2) / np.float64(h12))
    return h1, h2, h12, h1 + h2 - h12, nmi


def mutual_information(x, y, bins=100):
    return entropies(joint_histogram(x, y, bins)[0])[3]


def normalized_mutual_information(x, y, bins=100):
    """scikit-image's ``normalized_mutual_information(x, y, bins=bins)``."""
    return entropies(joint_histogram(x, y, bins)[0])[4]
