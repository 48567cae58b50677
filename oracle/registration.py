"""TEST INFRASTRUCTURE (oracle): numpy fp64 restatement of rigid registration by Mattes mutual information, of the
separable Gaussian filter its pyramid smooths with, and of resampling through the resulting transform.  Only tests/
and tools/ may import this module.

The definitions are the ones pinned in include/mpgan.h (section "rigid registration"); this module restates them with
elementwise numpy ufuncs (one IEEE fp64 rounding per operation, no ``@`` / ``einsum`` / ``dot``), so that where the
header promises bits the kernels and this module agree bit for bit:

- ``gaussian_filter``: scipy's taps (``mpgan.transforms.gaussian_taps``), reflect boundaries, fp64 sums over taps in
  order, x then y then z, one rounding to fp32 at the end.
- ``euler`` / ``compose``: ITK's Euler transform (rank 3: R = (Rz Rx) Ry; rank 2: the plane rotation), sin and cos
  from pinned polynomials (not libm, whose last bits differ between hosts and the device), composed with the fixed
  grid into the 24-word map of ``mpgan_resample_linear``.
- ``mattes``: the fixed-point joint histogram (bit-exact), -MI and its gradient.
- ``register``: the pyramid and the regular-step gradient descent.

No ITK parity is claimed: ITK is not available to the tests.
"""
import math

import numpy as np

from oracle import resample as ors

TWO32 = 2.0 ** 32
SIN_C = [((-1) ** k) / math.factorial(2 * k + 1) for k in range(14)]   # exactly rounded (int / int)
COS_C = [((-1) ** k) / math.factorial(2 * k) for k in range(15)]
TWO_PI_HI = float.fromhex("0x1.921fb54442d18p+2")
TWO_PI_LO = 2.4492935982947064e-16
INV_TWO_PI = float.fromhex("0x1.45f306dc9c883p-3")
TWO_THIRDS = 2.0 / 3.0

RUNNING, CONVERGED, ITERATIONS, OVERLAP, FLAT = -1, 0, 1, 2, 3


# ---- Gaussian filter -------------------------------------------------------------------------------------------------
def reflect(j, n):
    """scipy's "reflect" (d c b a | a b c d | d c b a) index into [0, n)."""
    j = np.mod(j, 2 * n)
    return np.where(j >= n, 2 * n - 1 - j, j)


def filter_axis(x, taps, axis):
    """fp64 correlation of x with ``taps`` (odd length) along ``axis``, reflect boundaries, taps summed in order."""
    n, r = x.shape[axis], len(taps) // 2
    idx = np.arange(n)
    acc = None
    for t, w in enumerate(taps):
        v = np.float64(w) * np.take(x, reflect(idx + t - r, n), axis=axis)
        acc = v if acc is None else acc + v
    return acc


def gaussian_filter(x, taps_xyz, rank):
    """x (..., [z,] y, x) float32 -> float32: the fp64 separable filter with taps per ITK axis (x, y, z)."""
    v = np.asarray(x, dtype=np.float32).astype(np.float64)
    for k in range(rank):
        v = filter_axis(v, taps_xyz[k], v.ndim - 1 - k)
    return v.astype(np.float32)


# ---- transform -------------------------------------------------------------------------------------------------------
def sincos(t):
    """Pinned sin and cos of fp64 arrays: reduction by 2 pi in two parts, then Horner polynomials in r^2."""
    t = np.asarray(t, dtype=np.float64)
    n = np.rint(t * INV_TWO_PI)
    r = (t - n * TWO_PI_HI) - n * TWO_PI_LO
    r2 = r * r
    s = np.float64(SIN_C[-1])
    for c in SIN_C[-2::-1]:
        s = c + r2 * s
    c_ = np.float64(COS_C[-1])
    for c in COS_C[-2::-1]:
        c_ = c + r2 * c_
    return r * s, c_


def matmul3(a, b):
    """3x3 nested lists of arrays: ((a_i0 b_0j + a_i1 b_1j) + a_i2 b_2j)."""
    return [[(a[i][0] * b[0][j] + a[i][1] * b[1][j]) + a[i][2] * b[2][j] for j in range(3)] for i in range(3)]


def euler(theta, rank):
    """(R, [dR/dtheta_j]) as 3x3 nested lists of fp64 arrays (rank 2 lifted with the identity's z)."""
    z = np.zeros_like(np.asarray(theta[0], dtype=np.float64))
    one = z + 1.0
    if rank == 2:
        s, c = sincos(theta[0])
        return [[c, -s, z], [s, c, z], [z, z, one]], [[[-s, -c, z], [c, -s, z], [z, z, z]]]
    (sx, cx), (sy, cy), (sz, cz) = (sincos(t) for t in theta)
    rx = [[one, z, z], [z, cx, -sx], [z, sx, cx]]
    ry = [[cy, z, sy], [z, one, z], [-sy, z, cy]]
    rz = [[cz, -sz, z], [sz, cz, z], [z, z, one]]
    drx = [[z, z, z], [z, -sx, -cx], [z, cx, -sx]]
    dry = [[-sy, z, cy], [z, z, z], [-cy, z, -sy]]
    drz = [[-sz, -cz, z], [cz, -sz, z], [z, z, z]]
    zx = matmul3(rz, rx)
    return matmul3(zx, ry), [matmul3(matmul3(rz, drx), ry), matmul3(zx, dry), matmul3(matmul3(drz, rx), ry)]


def n_params(rank):
    return 6 if rank == 3 else 3


def split(params, rank):
    """(rotation angles, translation t[3]) of a (..., P) parameter array."""
    p = np.asarray(params, dtype=np.float64)
    if rank == 2:
        return [p[..., 0]], [p[..., 1], p[..., 2], np.zeros_like(p[..., 0])]
    return [p[..., 0], p[..., 1], p[..., 2]], [p[..., 3], p[..., 4], p[..., 5]]


def _affine(rm, base, center, t):
    """(o'[3], M'[3][3]) of the map sending a fixed index through rm: M' = rm M_fixed, o' = (rm (o_fixed - c) + c) + t
    (t None: o' = rm (o_fixed - c), the derivative form)."""
    o, m = base[0:3], [base[3:6], base[6:9], base[9:12]]
    d = [o[k] - center[k] for k in range(3)]
    mm = matmul3(rm, [[np.float64(v) for v in row] for row in m])
    e = [(rm[k][0] * d[0] + rm[k][1] * d[1]) + rm[k][2] * d[2] for k in range(3)]
    oo = e if t is None else [(e[k] + center[k]) + t[k] for k in range(3)]
    return oo, mm


def compose(params, base, center, rank):
    """The 24-word map (o', M', o_moving, N_moving) of one parameter vector; ``base`` =
    ``mpgan.transforms.resample_map(moving, fixed)`` (o_fixed, M_fixed, o_moving, N_moving), ``center`` the fixed
    grid's centre.  Returns (map[24] as floats, rotation-derivative maps: list of (do[3], dM[3][3]))."""
    theta, t = split(params, rank)
    r, drs = euler(theta, rank)
    oo, mm = _affine(r, base, center, t)
    out = [float(v) for v in oo] + [float(mm[i][j]) for i in range(3) for j in range(3)] + [float(v) for v in base[12:]]
    ders = [_affine(dr, base, center, None) for dr in drs]
    return out, [([float(v) for v in do], [[float(v) for v in row] for row in dm]) for do, dm in ders]


def map_index(m, ix, iy, iz):
    """Continuous moving index (3, ...) of fixed indices under a 24-word map: the resample kernels' arithmetic."""
    oo, mm, oi, nn = m[0:3], m[3:12], m[12:15], m[15:24]
    p = [((oo[k] + mm[3 * k] * ix) + mm[3 * k + 1] * iy) + mm[3 * k + 2] * iz for k in range(3)]
    q = [p[k] - oi[k] for k in range(3)]
    return np.stack([((nn[3 * k] * q[0]) + nn[3 * k + 1] * q[1]) + nn[3 * k + 2] * q[2] for k in range(3)])


def grid_index(size):
    """(ix, iy, iz) fp64 arrays of shape (z, y, x) of a size[3] grid (ITK order)."""
    iz, iy, ix = np.meshgrid(*(np.arange(s, dtype=np.float64) for s in size[::-1]), indexing="ij")
    return ix, iy, iz


def resample_mapped(image, size_in, size_out, m, default_value=0.0, interpolation="linear"):
    """One item (source.shape) resampled onto size_out through a 24-word map, with the oracles of oracle/resample.py
    and oracle/resample_interpolation.py."""
    from oracle import resample_interpolation as ori
    c = map_index(m, *grid_index(size_out))
    image = np.asarray(image)
    x3 = image.reshape((1,) + tuple(size_in[::-1]))
    ok = ors.inside(c, size_in)
    if interpolation == "nearest":
        bits = x3.view(np.uint32) if x3.dtype.itemsize == 4 else x3.view(np.uint8)
        ix, iy, iz = ori.nearest_index(c, size_in)
        dflt = np.asarray(default_value, dtype=image.dtype).view(bits.dtype)
        return np.where(ok, bits[0, iz, iy, ix], dflt).astype(bits.dtype).view(image.dtype)
    if interpolation == "linear":
        val = ors.interpolate(x3.astype(np.float32), c, size_in)[0]
    else:
        coef = ori.bspline_coefficients(x3.astype(np.float32), 3 if size_in[2] > 1 else 2)
        val = ori.interpolate_bspline(coef, c, size_in)[0]
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(ok, val, np.float64(np.float32(default_value))).astype(np.float32)


# ---- Mattes mutual information -----------------------------------------------------------------------------------------
def bspline3(u):
    a = np.abs(u)
    a2 = a * a
    b = 2.0 - a
    return np.where(a < 1.0, (TWO_THIRDS - a2) + 0.5 * (a2 * a), np.where(a < 2.0, ((b * b) * b) / 6.0, 0.0))


def bspline3_deriv(u):
    a = np.abs(u)
    b = 2.0 - a
    return np.where(a < 1.0, u * (1.5 * a - 2.0), np.where(a < 2.0, np.copysign(0.5 * (b * b), -u), 0.0))


def index_gradient(m3):
    """(3, nz, ny, nx) float32: central differences of m3 (nz, ny, nx) along x, y, z; one-sided at the borders, 0
    along an extent of 1."""
    out = np.zeros((3,) + m3.shape, dtype=np.float32)
    for k in range(3):
        ax = 2 - k
        n = m3.shape[ax]
        if n == 1:
            continue
        v, g = np.moveaxis(m3, ax, 0), np.moveaxis(out[k], ax, 0)
        g[1:-1] = (v[2:] - v[:-2]) * np.float32(0.5)
        g[0] = v[1] - v[0]
        g[-1] = v[-1] - v[-2]
    return out


def sample_indices(fixed_size, shrink, mask=None):
    """(ix, iy, iz) int64 of the level's fixed samples in raster order; ``mask`` (z, y, x) restricts them."""
    ix, iy, iz = (a.astype(np.int64) for a in grid_index(fixed_size))
    keep = (ix % shrink == 0) & (iy % shrink == 0) & (iz % shrink == 0)
    if mask is not None:
        keep &= np.asarray(mask).reshape(keep.shape) != 0
    return ix[keep], iy[keep], iz[keep]


def ranges(f3, m3, samples):
    """(fixed min, fixed max, moving min, moving max, fixed samples) of one level: fp32 extremes as floats; NaN when an
    image holds NaN (np.min / np.max propagate it)."""
    ix, iy, iz = samples
    fv = f3[iz, iy, ix]
    if fv.size == 0:
        return math.nan, math.nan, float(np.min(m3)), float(np.max(m3)), 0
    return float(np.min(fv)), float(np.max(fv)), float(np.min(m3)), float(np.max(m3)), int(fv.size)


def rotation_scales(samples, fixed_size, fixed_matrix, rank, min_scale):
    """The optimiser's scale of each rotation angle for one level: the RMS distance of the samples from that rotation
    axis through the grid centre, at least ``min_scale``.  S = the exact int64 moments of (2 i - (n - 1)) over the
    samples, C = (M S) M^T in pinned fp64, v_k = C_kk / (4 n), scale_a = sqrt of the other two v (rank 2: v_x + v_y)."""
    ix, iy, iz = samples
    n = len(ix)
    a, b, c = (2 * ix - (fixed_size[0] - 1), 2 * iy - (fixed_size[1] - 1), 2 * iz - (fixed_size[2] - 1))
    mo = [int(np.sum(u * w)) for u, w in ((a, a), (b, b), (c, c), (a, b), (a, c), (b, c))]
    S = [[float(mo[0]), float(mo[3]), float(mo[4])], [float(mo[3]), float(mo[1]), float(mo[5])],
         [float(mo[4]), float(mo[5]), float(mo[2])]]
    m = [float(v) for v in fixed_matrix]
    v = []
    for k in range(3):
        t = [(m[3 * k] * S[0][j] + m[3 * k + 1] * S[1][j]) + m[3 * k + 2] * S[2][j] for j in range(3)]
        ck = (t[0] * m[3 * k] + t[1] * m[3 * k + 1]) + t[2] * m[3 * k + 2]
        v.append(ck / (4.0 * n) if n else 0.0)
    pairs = [(1, 2), (0, 2), (0, 1)] if rank == 3 else [(0, 1)]
    return [max(math.sqrt(v[p] + v[q]), min_scale) for p, q in pairs]


def level_flat(rng):
    fmin, fmax, mmin, mmax, _ = rng
    return not (fmax > fmin and mmax > mmin and all(math.isfinite(v) for v in rng[:4]))


def mattes(f3, m3, grad3, samples, rng, m, ders, moving_n, rank, bins, want_gradient=True):
    """One evaluation at the 24-word map ``m``: dict(hist int64 (B, B), inside, metric = -MI, gradient (P,) of -MI)."""
    ix, iy, iz = samples
    fmin, fmax, mmin, mmax, count = rng
    df = (fmax - fmin) / float(bins - 4)
    dm = (mmax - mmin) / float(bins - 4)
    c = map_index(m, ix.astype(np.float64), iy.astype(np.float64), iz.astype(np.float64))
    size_in = m3.shape[::-1]
    ok = ors.inside(c, size_in)
    c, ix, iy, iz = c[:, ok], ix[ok], iy[ok], iz[ok]
    f = f3[iz, iy, ix].astype(np.float64)
    v = ors.interpolate(m3[None], c, size_in)[0]
    xf = (f - fmin) / df + 2.0
    fb = np.clip(np.floor(xf), 2, bins - 3).astype(np.int64)
    xm = (v - mmin) / dm + 2.0
    mb = np.clip(np.floor(xm), 2, bins - 3).astype(np.int64)
    hist = np.zeros((bins, bins), dtype=np.int64)
    for j in range(4):
        k = mb - 1 + j
        q = np.rint(bspline3(k.astype(np.float64) - xm) * TWO32).astype(np.int64)
        np.add.at(hist, (fb, k), q)
    inside = int(ok.sum())
    res = {"hist": hist, "inside": inside, "metric": math.nan, "gradient": np.full(n_params(rank), math.nan)}
    if inside == 0 or 4 * inside < count:
        return res
    s = hist.sum()
    sd = float(s)
    hf, hm = hist.sum(axis=1), hist.sum(axis=0)
    p = hist / sd
    pf, pm = hf / sd, hm / sd
    nz = hist > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        term = np.where(nz, p * np.log(p / (pf[:, None] * pm[None, :])), 0.0)
        lt = np.where(nz, np.log(hist / hm[None, :].astype(np.float64)), 0.0)
    res["metric"] = -float(term.sum())
    if not want_gradient:
        return res
    a = np.zeros(inside)
    for j in range(4):
        k = mb - 1 + j
        a = a + bspline3_deriv(k.astype(np.float64) - xm) * lt[fb, k]
    gi = [ors.interpolate(grad3[kk][None], c, size_in)[0] for kk in range(3)]
    nn = moving_n
    gp = [(nn[0][k] * gi[0] + nn[1][k] * gi[1]) + nn[2][k] * gi[2] for k in range(3)]
    fx, fy, fz = ix.astype(np.float64), iy.astype(np.float64), iz.astype(np.float64)
    cols = []
    for do, dmx in ders:
        jac = [((do[k] + dmx[k][0] * fx) + dmx[k][1] * fy) + dmx[k][2] * fz for k in range(3)]
        cols.append((gp[0] * jac[0] + gp[1] * jac[1]) + gp[2] * jac[2])
    cols += gp[:rank]
    res["gradient"] = np.array([float(np.sum(a * col)) for col in cols]) * (TWO32 / (sd * dm))
    return res


# ---- registration ------------------------------------------------------------------------------------------------------
def register_one(fixed, moving, fixed_geometry, moving_geometry, fixed_mask=None, bins=50, shrink_factors=(4, 2, 1),
                 smoothing_sigmas=(2.0, 1.0, 0.0), iterations=100, initialize="geometry", initial_parameters=None,
                 trace=None):
    """One pair: dict(parameters, metric, status, map).  Mirrors mpgan.transforms.register_rigid, with its level
    constants from ``mpgan.transforms._registration_plan``."""
    from mpgan.transforms import _registration_plan, gaussian_taps
    plan = _registration_plan(fixed_geometry, moving_geometry, shrink_factors, smoothing_sigmas, initialize)
    rank = fixed_geometry.rank
    P = n_params(rank)
    fsize = tuple(fixed_geometry.size) + (1,) * (3 - rank)
    f3 = np.asarray(fixed, dtype=np.float32).reshape(fsize[::-1])
    m3raw = np.asarray(moving, dtype=np.float32).reshape(plan["moving_size"][::-1])
    mask = None if fixed_mask is None else np.asarray(fixed_mask).reshape(fsize[::-1])
    if initial_parameters is not None:
        mu = np.array(initial_parameters, dtype=np.float64)
    else:
        mu = np.zeros(P)
        mu[P - rank:] = plan["t0"][:rank]
    status, metric = RUNNING, math.nan
    nn = plan["base"][15:24]
    moving_n = [nn[0:3], nn[3:6], nn[6:9]]
    for lvl in plan["levels"]:
        fs = gaussian_filter(f3, [gaussian_taps(s) for s in lvl["fixed_sigmas"]], 3)
        ms = gaussian_filter(m3raw, [gaussian_taps(s) for s in lvl["moving_sigmas"]], 3)
        grad3 = index_gradient(ms)
        samples = sample_indices(fsize, lvl["shrink"], mask)
        rng = ranges(fs, ms, samples)
        if status in (OVERLAP, FLAT):
            break
        if level_flat(rng):
            status = FLAT if rng[4] > 0 else OVERLAP
            break
        status, step, gprev = RUNNING, lvl["step"], np.zeros(P)
        scales = np.array(rotation_scales(samples, fsize, plan["base"][3:12], rank, plan["min_scale"]) + [1.0] * rank)
        m, ders = compose(mu, plan["base"], plan["center"], rank)
        for it in range(iterations):
            r = mattes(fs, ms, grad3, samples, rng, m, ders, moving_n, rank, bins)
            if trace is not None:
                trace.append((lvl["shrink"], it, r["metric"], mu.copy()))
            if not math.isfinite(r["metric"]):
                status, metric = OVERLAP, math.nan
                break
            gu = r["gradient"] / scales
            dot = 0.0
            for j in range(P):
                dot = dot + gu[j] * gprev[j]
            if dot < 0.0:
                step = step * 0.5
            if step < plan["min_step"]:
                status = CONVERGED
                break
            nrm2 = 0.0
            for j in range(P):
                nrm2 = nrm2 + gu[j] * gu[j]
            nrm = math.sqrt(nrm2)
            if not nrm > 0.0:
                status = CONVERGED
                break
            mu = mu - ((step * gu) / nrm) / scales
            gprev = gu
            m, ders = compose(mu, plan["base"], plan["center"], rank)
            if it == iterations - 1:
                status = ITERATIONS
    if status in (CONVERGED, ITERATIONS):
        r = mattes(fs, ms, grad3, samples, rng, m, ders, moving_n, rank, bins, want_gradient=False)
        metric = r["metric"]
        if not math.isfinite(metric):
            status = OVERLAP
    m, _ = compose(mu, plan["base"], plan["center"], rank)
    return {"parameters": mu, "metric": metric, "status": status, "map": m}


def homogeneous(params, center, rank):
    """The (rank+1)^2 fp64 matrix of q = R (p - c) + c + t, from the pinned map arithmetic on an identity grid."""
    base = [0.0] * 3 + [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0] + [0.0] * 3 + [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0,
                                                                                      0.0, 1.0]
    m, _ = compose(params, base, center, rank)
    out = np.eye(rank + 1)
    for i in range(rank):
        out[i, :rank] = m[3 + 3 * i:3 + 3 * i + rank]
        out[i, rank] = m[i]
    return out


# ---- synthetic head phantom ----------------------------------------------------------------------------------------------
# Nested ellipsoids (centre mm, semi-axes mm, tissue) in the phantom's own frame, off-centre and tilted enough that
# no rotation or translation maps the head onto itself.  T1 and T2 intensities per tissue are ordered differently
# (T1: scalp > brain > csf > bone; T2: csf > brain > scalp > bone), so only a statistical metric can align them.
_ELLIPSOIDS = [((0.0, 0.0, 0.0), (70.0, 85.0, 60.0), "scalp"), ((0.0, 2.0, 1.0), (64.0, 79.0, 54.0), "bone"),
               ((0.0, 3.0, 2.0), (58.0, 72.0, 48.0), "brain"), ((-12.0, 10.0, 6.0), (9.0, 20.0, 10.0), "csf"),
               ((14.0, 6.0, 5.0), (7.0, 16.0, 9.0), "csf"), ((20.0, -35.0, -10.0), (12.0, 10.0, 12.0), "bone"),
               ((-25.0, -30.0, 15.0), (10.0, 14.0, 8.0), "csf")]
CONTRAST = {"t1": {"scalp": 0.9, "bone": 0.1, "brain": 0.6, "csf": 0.25},
            "t2": {"scalp": 0.35, "bone": 0.05, "brain": 0.55, "csf": 1.0}}


def phantom(geometry, contrast, params=None, center=None, edge_mm=2.0):
    """float32 image of the phantom on ``geometry`` (tensor layout), seen through the rigid transform ``params`` about
    ``center`` (fixed-space physical point p -> moving point q = R (p - c) + c + t): the image at q is the phantom at
    p = R^T (q - c - t) + c.  Tissue boundaries are smooth (logistic, ``edge_mm`` wide)."""
    rank = geometry.rank
    size = tuple(geometry.size) + (1,) * (3 - rank)
    ix, iy, iz = grid_index(size)
    from mpgan.transforms import _lift3
    m, o = _lift3(geometry.index_to_physical(), geometry.origin)
    q = [o[k] + m[k, 0] * ix + m[k, 1] * iy + m[k, 2] * iz for k in range(3)]
    if params is not None:
        theta, t = split(params, rank)
        r, _ = euler(theta, rank)
        d = [q[k] - center[k] - float(t[k]) for k in range(3)]
        q = [float(r[0][k]) * d[0] + float(r[1][k]) * d[1] + float(r[2][k]) * d[2] + center[k] for k in range(3)]
    img = np.zeros(q[0].shape)
    for ctr, axes, tissue in _ELLIPSOIDS:
        ax = axes if rank == 3 else axes[:2] + (1e9,)
        rr = np.sqrt(sum(((q[k] - ctr[k]) / ax[k]) ** 2 for k in range(3)))
        inside = 1.0 / (1.0 + np.exp(np.clip((rr - 1.0) * min(ax) / edge_mm * 4.0, -60, 60)))
        img = img * (1.0 - inside) + CONTRAST[contrast][tissue] * inside
    return img.astype(np.float32).reshape(geometry.shape)


def displacement(params_a, params_b, center, rank, points):
    """Mean |T_a(p) - T_b(p)| over physical points (3, N) of two parameter vectors about one centre."""
    out = []
    for prm in (params_a, params_b):
        theta, t = split(prm, rank)
        r, _ = euler(theta, rank)
        d = [points[k] - center[k] for k in range(3)]
        out.append(np.stack([(float(r[k][0]) * d[0] + float(r[k][1]) * d[1] + float(r[k][2]) * d[2]) + center[k]
                             + float(t[k]) for k in range(3)]))
    return float(np.mean(np.sqrt(((out[0] - out[1]) ** 2).sum(axis=0))))
