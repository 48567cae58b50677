"""TEST INFRASTRUCTURE (oracle): the exact Euclidean distance transform of masks and the agreement of two masks, a thin
layer over scipy.ndimage and np.percentile.  Only tests/ and tools/ may import this module.

include/mpgan.h pins the semantics; restated here:
  * images: the last ``spatial_dims`` (2 or 3, default min(ndim, 3)) dims are spatial, every leading index is an
    independent image; non-zero is "in".  ``sampling``: None, one number, or one per spatial dim in array order.
  * distance_transform_edt: ``scipy.ndimage.distance_transform_edt(mask, sampling)`` per image, with one deliberate
    departure: an image without a 0 voxel is +inf everywhere (scipy returns meaningless finite values there).
  * surface(M) = M & ~binary_erosion(M, generate_binary_structure(rank, connectivity), border_value=0) (MONAI's
    get_mask_edges; its crop to the bounding box changes nothing).
  * D(A -> B) = edt(~surface(B), sampling)[surface(A)].
  * dice = 2 i / (a + b), jaccard = i / (a + b - i) of the int counts a = |P|, b = |T|, i = |P & T|: NaN when both
    masks are empty, 0 when exactly one is.
  * hausdorff = max(max D(P->T), max D(T->P)); hausdorff_percentile = max of the two np.percentile(D, percentile);
    average_surface_distance = mean D(P->T); symmetric_surface_distance = mean of D(P->T) and D(T->P) concatenated.
  * both masks empty: the four distance metrics are NaN; exactly one empty: +inf.
"""
import math

import numpy as np
from scipy import ndimage

KEYS = ("dice", "jaccard", "hausdorff", "hausdorff_percentile", "average_surface_distance",
        "symmetric_surface_distance")


def _images(mask, spatial_dims):
    m = np.asarray(mask).astype(bool)
    nd = spatial_dims or min(m.ndim, 3)
    return m.reshape((-1,) + m.shape[m.ndim - nd:]), m.shape[:m.ndim - nd], nd


def _sampling(sampling, nd):
    if sampling is None:
        return None
    return (float(sampling),) * nd if np.ndim(sampling) == 0 else tuple(float(s) for s in sampling)


def edt(im, sampling=None):
    """One image: scipy's transform, +inf everywhere when the image has no 0 voxel."""
    if im.all():
        return np.full(im.shape, np.inf)
    return ndimage.distance_transform_edt(im, sampling=_sampling(sampling, im.ndim))


def distance_transform_edt(mask, sampling=None, spatial_dims=None):
    ims, _, nd = _images(mask, spatial_dims)
    out = np.zeros(ims.shape, np.float64)
    for i, im in enumerate(ims):
        out[i] = edt(im, sampling)
    return out.reshape(np.shape(mask))


def surface(im, connectivity=1):
    return im & ~ndimage.binary_erosion(im, ndimage.generate_binary_structure(im.ndim, connectivity), border_value=0)


def surface_distances(pred, truth, sampling=None, connectivity=1):
    """(D(P -> T), D(T -> P)) of one image pair, each in raster order of its surface voxels."""
    sp, st = surface(pred, connectivity), surface(truth, connectivity)
    return edt(~st, sampling)[sp], edt(~sp, sampling)[st]


def percentile_restated(values, percentile):
    """np.percentile(values, percentile) (numpy 2.x, method "linear") restated as the kernel computes it."""
    v = np.sort(np.asarray(values, np.float64))
    n = len(v)
    q = np.float64(percentile) / np.float64(100)
    virtual = np.float64(n - 1) * q          # numpy's "linear" method: (n - 1) q, one rounding
    if virtual >= n - 1:
        lo = hi = n - 1
    elif virtual < 0:
        lo = hi = 0
    else:
        lo = int(math.floor(virtual))
        hi = lo + 1
    a, b = v[lo], v[hi]
    if lo == hi:
        return a
    t = virtual - np.float64(lo)
    diff = b - a
    return b - diff * (np.float64(1) - t) if t >= 0.5 else a + diff * t


def agreement(pred, truth, sampling=None, percentile=95, connectivity=1):
    """The six metrics of one image pair, as python floats."""
    pred, truth = np.asarray(pred, bool), np.asarray(truth, bool)
    a, b, i = int(pred.sum()), int(truth.sum()), int((pred & truth).sum())
    dice = 2 * i / (a + b) if a + b else math.nan
    jaccard = i / (a + b - i) if a + b - i else math.nan
    if a == 0 or b == 0:
        d = math.nan if a == b == 0 else math.inf
        return dict(zip(KEYS, (dice, jaccard, d, d, d, d)))
    pt, tp = surface_distances(pred, truth, sampling, connectivity)
    return dict(zip(KEYS, (dice, jaccard, float(max(pt.max(), tp.max())),
                           float(max(np.percentile(pt, percentile), np.percentile(tp, percentile))),
                           float(pt.mean()), float(np.concatenate([pt, tp]).mean()))))


def mask_agreement(pred, truth, sampling=None, percentile=95, connectivity=1, spatial_dims=None):
    """dict of float64 arrays of the leading shape."""
    ps, lead, _ = _images(pred, spatial_dims)
    ts, _, _ = _images(truth, spatial_dims)
    rows = [agreement(p, t, sampling, percentile, connectivity) for p, t in zip(ps, ts)]
    return {k: np.array([r[k] for r in rows], np.float64).reshape(lead) for k in KEYS}
