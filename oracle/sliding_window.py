"""TEST INFRASTRUCTURE (oracle): numpy fp64 restatement of sliding-window inference.  Only tests/ and tools/ may import
this module.

Follows MONAI 0.4.0 ``sliding_window_inference`` / ``_get_scan_interval`` / ``dense_patch_slices`` /
``compute_importance_map`` (the call the reference's minipig_inference.py:110-114 leaves commented out), with constant
padding only:
  - roi: an entry that is None or <= 0 takes the image extent (``fall_back_tuple``);
  - padding: diff = max(roi - S, 0), lo = diff // 2 before, diff - lo after, filled with ``cval``;
  - interval: roi if roi equals the padded extent P, else max(int(roi (1 - overlap)), 1);
  - starts: n = 1 + max(ceil((P - roi) / interval), 0) windows at min(j interval, P - roi) per dim, the Cartesian
    product ordered first dim slowest, image-major over the batch; the predictor sees runs of sw_batch_size of them;
  - importance map: prod_d t_d(i_d), t = 1 ("constant") or exp(-(i - roi // 2)^2 / (2 (sigma roi)^2)) ("gaussian",
    the sampled Gaussian that MONAI 0.4.0's filtered delta amounts to), with underflowed taps raised to the dim's
    smallest positive tap (MONAI applies that floor to the whole map; the two differ only for sigma_scale below ~0.02);
  - output: sum_k w y_k / sum_k w over the windows covering each voxel, in fp64 (MONAI accumulates in fp32).
Parity with MONAI itself is unpinned (it is not installed here); tests/test_sliding_window.py pins this restatement
against a table of known geometries and against a brute-force count-map accumulation.
"""
import math

import numpy as np


def fall_back_roi(roi_size, size):
    return tuple(int(s) if r is None or r <= 0 else int(r) for r, s in zip(roi_size, size))


def scan_starts(size, roi, overlap):
    """(starts, lo) of one dim: window starts in padded coordinates and the padding before the image."""
    diff = max(roi - size, 0)
    padded = size + diff
    interval = roi if roi == padded else max(int(roi * (1 - overlap)), 1)
    n = 1 + max(math.ceil((padded - roi) / interval), 0)
    return [min(j * interval, padded - roi) for j in range(n)], diff // 2


def importance_taps(roi, mode, sigma):
    if mode == "constant":
        return np.ones(roi)
    i = np.arange(roi, dtype=np.float64)
    t = np.exp(-((i - roi // 2) ** 2) / (2.0 * (sigma * roi) ** 2))
    return np.where(t > 0, t, t[t > 0].min())


def geometry(size, roi_size, overlap):
    """Per dim: (roi, starts, lo)."""
    roi = fall_back_roi(roi_size, size)
    out = []
    for s, r in zip(size, roi):
        starts, lo = scan_starts(s, r, overlap)
        out.append((r, starts, lo))
    return out


def window_starts(geo):
    """Window starts (padded coordinates) of one image, in window order."""
    return [tuple(geo[d][1][j] for d, j in enumerate(idx)) for idx in np.ndindex(*[len(g[1]) for g in geo])]


def pad(x, geo, cval):
    """(B, C, *S) -> (B, C, *P) with ``cval`` around the image."""
    widths = [(0, 0), (0, 0)] + [(lo, r - s - lo) if r > s else (0, 0) for (r, _, lo), s in zip(geo, x.shape[2:])]
    return np.pad(x, widths, mode="constant", constant_values=cval)


def extract_windows(x, geo, first, count, cval):
    """Windows [first, first + count) of the global order, (count, C, *roi), in x's dtype (an exact copy)."""
    xp = pad(x, geo, cval)
    wins = window_starts(geo)
    out = []
    for k in range(first, first + count):
        b, w = divmod(k, len(wins))
        st = wins[w]
        out.append(xp[(b, slice(None)) + tuple(slice(s, s + g[0]) for s, g in zip(st, geo))])
    return np.stack(out)


def blend(preds, batch, geo, size, mode="constant", sigma_scale=0.125):
    """preds (batch * nwin, C, *roi) -> (batch, C, *S) fp64: the numerator summed window by window on the padded canvas,
    the denominator as the product of per-dim coverage sums."""
    nd = len(geo)
    sigmas = tuple(sigma_scale) if np.ndim(sigma_scale) else (sigma_scale,) * nd
    taps = [importance_taps(g[0], mode, s) for g, s in zip(geo, sigmas)]
    w = taps[0]
    for t in taps[1:]:
        w = np.multiply.outer(w, t)
    padded = [max(s, g[0]) for s, g in zip(size, geo)]
    wins = window_starts(geo)
    num = np.zeros((batch, preds.shape[1]) + tuple(padded))
    for k in range(batch * len(wins)):
        b, i = divmod(k, len(wins))
        st = wins[i]
        num[(b, slice(None)) + tuple(slice(s, s + g[0]) for s, g in zip(st, geo))] += w * preds[k].astype(np.float64)
    den = np.ones(())
    for (r, starts, _), p, t in zip(geo, padded, taps):
        dd = np.zeros(p)
        for s in starts:
            dd[s:s + r] += t
        den = np.multiply.outer(den, dd)
    crop = tuple(slice(lo, lo + s) for (_, _, lo), s in zip(geo, size))
    return (num / den)[(slice(None), slice(None)) + crop]


def sliding_window_inference(inputs, roi_size, sw_batch_size, predictor, overlap=0.25, mode="constant",
                             sigma_scale=0.125, cval=0.0):
    """inputs (B, C_in, *S) numpy; predictor: (n, C_in, *roi) float32 numpy -> (n, C_out, *roi) array.  fp64 result."""
    x = np.asarray(inputs)
    size = x.shape[2:]
    geo = geometry(size, roi_size, overlap)
    nwin = int(np.prod([len(g[1]) for g in geo]))
    total = x.shape[0] * nwin
    preds = []
    for first in range(0, total, sw_batch_size):
        n = min(sw_batch_size, total - first)
        preds.append(np.asarray(predictor(extract_windows(x, geo, first, n, cval)), dtype=np.float64))
    return blend(np.concatenate(preds), x.shape[0], geo, size, mode, sigma_scale)
