"""TEST INFRASTRUCTURE (oracle): numpy fp64 restatement of nearest-neighbour and cubic B-spline resampling between
physical grids.  Only tests/ and tools/ may import this module.

Follows ITK 5.1's ``ResampleImageFilter`` + ``IdentityTransform`` with a ``NearestNeighborInterpolateImageFunction``,
or with ``BSplineDecompositionImageFilter`` + ``BSplineInterpolateImageFunction`` of order 3, as recalled from ITK's
source.  ITK is not available here, so this restates the semantics pinned in include/mpgan.h; parity with ITK is not
claimed.  What is checked is agreement with scipy.ndimage (``map_coordinates(order=0)``; ``spline_filter`` and
``map_coordinates(order=3, mode="mirror")``).  The continuous index c and the inside test are oracle/resample.py's.
Every operation is a separate fp64 rounding (python floats and elementwise numpy ufuncs, no ``@``, ``einsum`` or
``dot``):

Nearest: per axis i_k = min(floor(c_k + 0.5), n_k - 1); the value is a copy of that input element, bits included.

Coefficients, per item, lines along x, then y, then z, each filtered in place (a line of N = 1 is left unchanged),
with z = sqrt(3) - 2, gain = (1 - z)(1 - 1/z), k = z / (z z - 1), z^j the repeated product (z^1 = z):
  c[n] = c[n] gain;
  N > 18: c[0] = ((c[0] + z c[1]) + z^2 c[2]) + ... + z^17 c[17]   (ITK's tolerance 1e-10: horizon 18)
  else:   s = c[0] + z^(N-1) c[N-1]; a = z; b = z^(N-1) (z^(N-1) (1/z));
          for n = 1 .. N-2: s = s + (a + b) c[n]; a = a z; b = b (1/z);   c[0] = s / (1 - a a)
  c[n] = c[n] + z c[n-1] for n = 1 .. N-1;   c[N-1] = k ((z c[N-2]) + c[N-1]);   c[n] = z (c[n+1] - c[n]) for n = N-2 .. 0.
Evaluation, per axis f = floor(c), w = c - f, w3 = ((1/6 w) w) w, w0 = (1/6 + (0.5 w)(w - 1)) - w3,
w2 = (w + w0) - 2 w3, w1 = ((1 - w0) - w2) - w3; taps f-1 .. f+2 mirrored with period 2n - 2; an axis of extent 1
contributes its single coefficient with weight 1.  Sums ((w0 a0 + w1 a1) + w2 a2) + w3 a3 along x, then y, then z;
one rounding to float32.  A NaN or inf input spreads along its lines through the recursions.
"""
import math

import numpy as np

from oracle import resample as ors

Z = math.sqrt(3.0) - 2.0
IZ = 1.0 / Z
GAIN = (1.0 - Z) * (1.0 - IZ)
K = Z / (Z * Z - 1.0)
HORIZON = 18
SIXTH = 1.0 / 6.0


def _size3(geometry):
    return tuple(geometry.size) + (1,) * (3 - geometry.rank)


def nearest_index(c, size):
    """(3, ...) int64 ITK-order indices of the nearest input voxel; meaningless where c is outside."""
    idx = []
    for k in range(3):
        ck = np.nan_to_num(c[k], nan=0.0)
        i = np.minimum(np.floor(ck + 0.5), size[k] - 1)
        idx.append(np.clip(i, 0, size[k] - 1).astype(np.int64))
    return idx


def resample_nearest(image, source, target, default_value=0):
    """image (*lead, *source.shape) of any dtype -> (*lead, *target.shape) of the same dtype, a bit copy."""
    image = np.asarray(image)
    lead = image.shape[:image.ndim - source.rank]
    size_in = _size3(source)
    x3 = image.reshape((-1,) + size_in[::-1])
    bits = x3.view(np.uint32) if x3.dtype.itemsize == 4 else x3.view(np.uint8)
    c = ors.continuous_index(source, target)
    ix, iy, iz = nearest_index(c, size_in)
    val = bits[:, iz, iy, ix]
    dflt = np.asarray(default_value, dtype=image.dtype).view(bits.dtype)
    out = np.where(ors.inside(c, size_in), val, dflt).astype(bits.dtype).view(image.dtype)
    return out.reshape(lead + tuple(target.shape))


def filter_lines(v):
    """In place: the cubic B-spline coefficients of every line v[:, ...] (the filtered axis first), fp64."""
    n = v.shape[0]
    if n == 1:
        return v
    v *= GAIN
    with np.errstate(invalid="ignore", over="ignore"):
        if n > HORIZON:
            s, zn = v[0].copy(), Z
            for j in range(1, HORIZON):
                s = s + zn * v[j]
                zn = zn * Z
        else:
            zl = Z
            for _ in range(2, n):
                zl = zl * Z
            s = v[0] + zl * v[n - 1]
            a, b = Z, zl * (zl * IZ)
            for j in range(1, n - 1):
                s = s + (a + b) * v[j]
                a, b = a * Z, b * IZ
            s = s / (1.0 - a * a)
        v[0] = s
        for j in range(1, n):
            v[j] = v[j] + Z * v[j - 1]
        v[n - 1] = K * (Z * v[n - 2] + v[n - 1])
        for j in range(n - 2, -1, -1):
            v[j] = Z * (v[j + 1] - v[j])
    return v


def bspline_coefficients(x3, rank=3):
    """x3 (items, nz, ny, nx) float32 -> fp64 coefficients of the same shape: lines along x, then y, then z."""
    coef = np.asarray(x3, dtype=np.float32).astype(np.float64)
    for axis in (3, 2, 1)[:rank]:
        filter_lines(np.moveaxis(coef, axis, 0))
    return coef


def _axis(c, n):
    """Taps (4, ...) int64 and weights (4, ...) fp64 of one axis at continuous indices c (inside)."""
    if n == 1:
        zero = np.zeros(c.shape, dtype=np.int64)
        return [zero] * 4, None
    with np.errstate(invalid="ignore"):
        f = np.floor(c)
        w = c - f
    w3 = ((SIXTH * w) * w) * w
    w0 = (SIXTH + (0.5 * w) * (w - 1.0)) - w3
    w2 = (w + w0) - 2.0 * w3
    w1 = ((1.0 - w0) - w2) - w3
    period = 2 * n - 2
    taps = []
    for t in range(4):
        j = np.abs(f.astype(np.int64) - 1 + t)
        j = np.where(j >= period, j - period, j)
        taps.append(np.where(j >= n, period - j, j))
    return taps, (w0, w1, w2, w3)


def _sum(a, w):
    if w is None:
        return a[0]
    return ((w[0] * a[0] + w[1] * a[1]) + w[2] * a[2]) + w[3] * a[3]


def interpolate_bspline(coef, c, size, chunk=1 << 21):
    """fp64 B-spline values of coef (items, nz, ny, nx) at continuous indices c (3, ...); c must be inside (clamped
    here so that outside positions give meaningless finite taps).  Returns (items, ...)."""
    shape = c.shape[1:]
    c = c.reshape(3, -1)
    out = np.empty((coef.shape[0], c.shape[1]), dtype=np.float64)
    for s in range(0, c.shape[1], chunk):
        cc = [np.clip(np.nan_to_num(c[k, s:s + chunk], nan=0.0), -0.5, size[k] - 0.5) for k in range(3)]
        (tx, wx), (ty, wy), (tz, wz) = (_axis(cc[k], size[k]) for k in range(3))
        with np.errstate(invalid="ignore", over="ignore"):
            az = []
            for kz in range(4 if wz is not None else 1):
                ay = [_sum([coef[:, tz[kz], ty[ky], tx[kx]] for kx in range(4)], wx) for ky in range(4)]
                az.append(_sum(ay, wy))
            out[:, s:s + chunk] = _sum(az, wz) if wz is not None else az[0]
    return out.reshape((coef.shape[0],) + shape)


def resample_bspline(image, source, target, default_value=0.0, coef=None):
    """image (*lead, *source.shape) float32 -> (*lead, *target.shape) float32.  ``coef``: precomputed
    ``bspline_coefficients`` of the image, (items, nz, ny, nx)."""
    image = np.asarray(image, dtype=np.float32)
    lead = image.shape[:image.ndim - source.rank]
    size_in = _size3(source)
    if coef is None:
        coef = bspline_coefficients(image.reshape((-1,) + size_in[::-1]), source.rank)
    c = ors.continuous_index(source, target)
    val = interpolate_bspline(coef, c, size_in)
    with np.errstate(invalid="ignore", over="ignore"):
        out = np.where(ors.inside(c, size_in), val, np.float64(np.float32(default_value))).astype(np.float32)
    return out.reshape(lead + tuple(target.shape))
