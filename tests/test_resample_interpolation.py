"""Nearest-neighbour and cubic B-spline resampling between physical grids (ITK's NearestNeighborInterpolateImageFunction
and, order 3, BSplineDecompositionImageFilter + BSplineInterpolateImageFunction inside ResampleImageFilter):
``mpgan.transforms.resample(..., interpolation="nearest" | "bspline")`` over the kernels in csrc/resample.cu.

ITK is not available here, so nothing is compared with ITK itself.  CPU tests pin the numpy fp64 restatement
(oracle/resample_interpolation.py) against scipy.ndimage (``map_coordinates(order=0)``, ``spline_filter`` and
``map_coordinates(order=3, mode="mirror")``) and against known answers (identity, axis permutations and flips, half
ties, the n - 0.5 clamp, extents 1 and 2, the edge voxel, NaN, every mask and label dtype), and check that argument
errors are raised before the device is touched and that the C ABI rejects bad input.  ``-m gpu`` tests compare the
kernels with the oracle bit for bit and run the native-grid scoring chain against the same chain built from oracles."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage
from scipy.spatial.transform import Rotation

from conftest import rel_l2
from oracle import resample as ors
from oracle import resample_interpolation as ori

gpu = pytest.mark.gpu
SENTINEL = 12345.0
MASK_DTYPES = {"float32": np.float32, "bool": np.bool_, "uint8": np.uint8, "int32": np.int32}


def _geometries():
    from mpgan.transforms import ImageGeometry, reference_grid
    return ImageGeometry, reference_grid


# geometry helpers: the pattern of tests/test_resample.py
def _rotation(seed, rank=3, max_angle=0.6):
    """A rotation about an oblique axis (rank 3) or in the plane (rank 2)."""
    rs = np.random.RandomState(seed)
    angle = rs.uniform(0.2, max_angle) * rs.choice([-1, 1])
    if rank == 2:
        return np.array([[math.cos(angle), -math.sin(angle)], [math.sin(angle), math.cos(angle)]])
    axis = rs.normal(size=3)
    return Rotation.from_rotvec(axis / np.linalg.norm(axis) * angle).as_matrix()


def _oblique(size, spacing, seed, centre=None):
    """A rotated grid whose centre lies at ``centre`` (default near the physical origin)."""
    ImageGeometry, _ = _geometries()
    rank = len(size)
    d = _rotation(seed, rank)
    rs = np.random.RandomState(seed + 100)
    centre = rs.uniform(-6, 6, rank) if centre is None else np.asarray(centre, dtype=np.float64)
    half = (np.asarray(size, dtype=np.float64) - 1) / 2 * np.asarray(spacing)
    origin = centre - d @ half
    return ImageGeometry(size, spacing, tuple(origin), d)


def _rand(shape, seed, lo=-1.0, hi=1.0):
    return np.random.RandomState(seed).uniform(lo, hi, shape).astype(np.float32)


def _values(shape, seed, dtype):
    """Random images of a mask or label dtype (float32: uniform in [-1, 1))."""
    rs = np.random.RandomState(seed)
    if dtype == np.float32:
        return _rand(shape, seed)
    if dtype == np.bool_:
        return rs.uniform(size=shape) < 0.5
    if dtype == np.uint8:
        return rs.randint(0, 256, shape).astype(np.uint8)
    return rs.randint(-2 ** 31, 2 ** 31 - 1, shape, dtype=np.int64).astype(np.int32)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype.itemsize == 4 else a.view(np.uint8)


def _same_bits(got, want):
    assert got.shape == want.shape and got.dtype == want.dtype
    assert np.array_equal(_bits(got), _bits(want))


def _within_ulps(got, want, ulps=1):
    assert got.shape == want.shape and got.dtype == np.float32
    assert np.all(np.abs(got.astype(np.float64) - want) <= ulps * np.spacing(np.abs(want).astype(np.float32)))


# ------------------------------------------------------------------------------------------ known answers (shared)
def _case_permutation(perm, flip, dtype):
    """Direction = an axis permutation with flips and anisotropic spacing: nearest resampling is a transpose / flip of
    the [z, y, x] array."""
    ImageGeometry, _ = _geometries()
    n_s, s_s, o_s = (7, 5, 4), (1.0, 2.0, 3.0), (10.0, -20.0, 30.0)
    src = ImageGeometry(n_s, s_s, o_s)
    d = np.zeros((3, 3))
    o_t = list(o_s)
    for j, k in enumerate(perm):
        d[k, j] = -1.0 if flip[j] else 1.0
        if flip[j]:
            o_t[k] = o_s[k] + (n_s[k] - 1) * s_s[k]
    tgt = ImageGeometry(tuple(n_s[k] for k in perm), tuple(s_s[k] for k in perm), tuple(o_t), d)
    x = _values((1,) + src.shape, 2, dtype)
    b = x[0].transpose(2, 1, 0).transpose(perm)
    b = np.flip(b, axis=tuple(j for j in range(3) if flip[j]))
    return x, src, tgt, 0, np.ascontiguousarray(b.transpose(2, 1, 0))[None]


def _case_identity(rank, dtype=np.float32):
    ImageGeometry, _ = _geometries()
    size, spacing, origin = ((13, 9, 6), (0.5, 1.0, 2.0), (-3.25, 7.0, 0.5))
    g = ImageGeometry(size[:rank], spacing[:rank], origin[:rank])   # powers of two: c = i exactly
    x = _values((2,) + g.shape, 1, dtype)
    return x, g, g, 0, x


def _case_half_ties():
    """Target centres exactly half-way between source voxels: round half up, c = -0.5 takes voxel 0, c = n - 0.5 is
    outside."""
    ImageGeometry, _ = _geometries()
    src = ImageGeometry((6, 5, 4), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    tgt = ImageGeometry((7, 5, 4), (1.0, 1.0, 1.0), (-0.5, 0.0, 0.0))   # c_x = -0.5, 0.5, ..., 5.5
    x = _values((1,) + src.shape, 5, np.float32)
    want = np.concatenate([x, np.full(x.shape[:-1] + (1,), -3.0, np.float32)], axis=-1)   # i -> voxel i; 5.5 outside
    return x, src, tgt, -3.0, want


def _case_nan():
    """NaN (with a payload) and inf inputs are copied exactly where their voxel is the nearest, and nowhere else."""
    ImageGeometry, _ = _geometries()
    src = ImageGeometry((6, 5, 4), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    tgt = ImageGeometry((12, 10, 8), (0.5, 0.5, 0.5), (-0.25, -0.25, -0.25))   # each source voxel -> a 2x2x2 block
    x = _values((1,) + src.shape, 6, np.float32)
    x[0, 1, 2, 3] = np.array(0x7FC01234, dtype=np.uint32).view(np.float32)
    x[0, 3, 4, 5] = -np.inf
    want = np.repeat(np.repeat(np.repeat(x, 2, axis=1), 2, axis=2), 2, axis=3)
    return x, src, tgt, 0, want


NEAREST_KNOWN = {"identity3": lambda: _case_identity(3), "identity2": lambda: _case_identity(2),
                 "identity3_bool": lambda: _case_identity(3, np.bool_),
                 "identity2_int32": lambda: _case_identity(2, np.int32),
                 "half_ties": _case_half_ties, "nan": _case_nan}
for _d in MASK_DTYPES:
    NEAREST_KNOWN[f"transpose_xz_{_d}"] = lambda d=_d: _case_permutation((2, 1, 0), (False,) * 3, MASK_DTYPES[d])
    NEAREST_KNOWN[f"cycle_flip_{_d}"] = lambda d=_d: _case_permutation((1, 2, 0), (True, False, True), MASK_DTYPES[d])
    NEAREST_KNOWN[f"swap_xy_flip_all_{_d}"] = lambda d=_d: _case_permutation((1, 0, 2), (True,) * 3, MASK_DTYPES[d])


def _case_clamp(n):
    """One target voxel at c_x one ulp below n - 0.5.  At n = 1, c + 0.5 rounds up to n (2^-54 below 1 is a tie
    that rounds to even), so the index must be clamped to n - 1; at larger n the sum is exact."""
    ImageGeometry, _ = _geometries()
    c = np.nextafter(n - 0.5, 0.0)
    src = ImageGeometry((n, 3), (1.0, 1.0), (0.0, 0.0))
    tgt = ImageGeometry((1, 3), (1.0, 1.0), (float(c), 0.0))
    x = _values((1,) + src.shape, 7, np.float32)
    return x, src, tgt, c


def _case_bspline_identity(rank):
    ImageGeometry, _ = _geometries()
    size, spacing, origin = ((13, 21, 6), (0.5, 1.0, 2.0), (-3.25, 7.0, 0.5))
    g = ImageGeometry(size[:rank], spacing[:rank], origin[:rank])
    x = _rand((2,) + g.shape, 8, 0.5, 2.0)
    return x, g, g


# ------------------------------------------------------------------------------------------------- oracle (CPU)
@pytest.mark.parametrize("name", sorted(NEAREST_KNOWN))
def test_oracle_nearest_known_answers(name):
    x, src, tgt, dflt, want = NEAREST_KNOWN[name]()
    _same_bits(ori.resample_nearest(x, src, tgt, dflt), want)


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("rank", [2, 3])
def test_oracle_nearest_matches_scipy(seed, rank):
    size_s = (13, 11, 9)[:rank]
    src = _oblique(size_s, (1.3, 0.9, 2.1)[:rank], seed)
    tgt = _oblique((17, 15, 12)[:rank], (1.1, 1.2, 1.6)[:rank], seed + 10)
    x = _rand((2,) + src.shape, seed)
    c = ors.continuous_index(src, tgt)
    ins = ors.inside(c, tuple(size_s) + (1,) * (3 - rank))
    assert 0.1 < ins.mean() < 0.9                                   # both sides of the boundary are exercised
    got = ori.resample_nearest(x, src, tgt, SENTINEL)
    coords = np.stack([c[k][ins] for k in reversed(range(rank))])    # array order (z, y, x)
    for i in range(2):
        ref = ndimage.map_coordinates(x[i], coords, order=0, mode="nearest")
        assert np.array_equal(got[i][ins.reshape(tgt.shape)], ref)
    assert (got[:, ~ins.reshape(tgt.shape)] == SENTINEL).all()


def test_oracle_nearest_rounds_half_up_like_scipy():
    """Including the fp64 rounding of c + 0.5: 2^-54 below 0.5 sums to 1 in both."""
    x = np.arange(6, dtype=np.float32)
    for c, want in ((0.5, 1), (2.5, 3), (-0.5, 0), (np.nextafter(0.5, 0), 1), (np.nextafter(1.5, 0), 1), (4.5, 5)):
        assert ndimage.map_coordinates(x, [[c]], order=0, mode="nearest")[0] == want
        assert ori.nearest_index(np.array([[c], [0.0], [0.0]]), (6, 1, 1))[0][0] == want


@pytest.mark.parametrize("n", [1, 2, 4, 1024])
def test_oracle_clamp_one_ulp_below_the_last_half(n):
    x, src, tgt, c = _case_clamp(n)
    assert np.floor(c + 0.5) == (n if n == 1 else n - 1)              # where the clamp is needed
    out = ori.resample_nearest(x, src, tgt, SENTINEL)
    assert np.array_equal(out[0, :, 0], x[0, :, n - 1])


@pytest.mark.parametrize("shape", [(7, 19, 30), (3, 1, 40), (5, 6, 18), (1, 2, 3), (2, 1, 1)])
def test_oracle_coefficients_match_spline_filter(shape):
    """The per-line bounds (1e-15 of the range for lines of <= 18, 1e-10 beyond), times 3 for every later filtered
    axis: the prefilter's gain is at most 3 (at Nyquist, 6 / (4 - 2)), so a difference left by one pass grows by at
    most that much in the next."""
    x = _rand((2,) + shape, 9, -3.0, 5.0)
    got = ori.bspline_coefficients(x, 3)
    short = max(shape) <= 18
    later = sum(n > 1 for n in shape) - 1
    for i in range(2):
        ref = ndimage.spline_filter(x[i].astype(np.float64), order=3, mode="mirror")
        err = np.abs(got[i] - ref).max() / float(x[i].max() - x[i].min())
        assert err <= (1e-15 if short else 1e-10) * 3 ** max(later, 0), err


def test_oracle_coefficient_lines_match_spline_filter1d():
    """Every line length from 1 to 70: exact mirror initialisation up to 18, ITK's truncated sum beyond."""
    rs = np.random.RandomState(10)
    for n in range(1, 71):
        x = rs.uniform(-1, 1, (3, n)).astype(np.float32)
        got = ori.bspline_coefficients(x[:, None, None, :], 1)[:, 0, 0]
        ref = ndimage.spline_filter1d(x.astype(np.float64), order=3, axis=1, mode="mirror")
        rng = float(x.max() - x.min())
        assert np.abs(got - ref).max() <= (1e-15 if n <= 18 else 1e-10) * rng, n


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("rank", [2, 3])
def test_oracle_bspline_matches_scipy(seed, rank):
    size_s = (13, 22, 9)[:rank]
    src = _oblique(size_s, (1.3, 0.9, 2.1)[:rank], seed)
    tgt = _oblique((17, 15, 12)[:rank], (1.1, 1.2, 1.6)[:rank], seed + 10)
    x = _rand((2,) + src.shape, seed, -2.0, 3.0)
    c = ors.continuous_index(src, tgt)
    size3 = tuple(size_s) + (1,) * (3 - rank)
    ins = ors.inside(c, size3)
    assert 0.1 < ins.mean() < 0.9
    coef = ori.bspline_coefficients(x.reshape((2,) + size3[::-1]), rank)
    got = ori.interpolate_bspline(coef, c, size3)[:, ins]
    coords = np.stack([c[k][ins] for k in reversed(range(rank))])
    for i in range(2):
        ref = ndimage.map_coordinates(x[i].astype(np.float64), coords, order=3, mode="mirror")
        assert np.abs(got[i] - ref).max() <= 1e-9 * float(x[i].max() - x[i].min())
    out = ori.resample_bspline(x, src, tgt, SENTINEL)
    assert (out[:, ~ins.reshape(tgt.shape)] == SENTINEL).all() and (out[:, ins.reshape(tgt.shape)] != SENTINEL).all()


@pytest.mark.parametrize("shape", [(1, 1, 5), (1, 2, 5), (2, 2, 2), (3, 1, 2)])
def test_oracle_bspline_small_extents_match_scipy(shape):
    """Extents 1 and 2: the period-(2n - 2) mirror and the single-coefficient axis."""
    x = _rand(shape, 11, -1.0, 2.0)
    rs = np.random.RandomState(12)
    c = np.stack([rs.uniform(-0.5, n - 0.5, 400) for n in shape[::-1]])      # ITK order
    coef = ori.bspline_coefficients(x[None], 3)
    got = ori.interpolate_bspline(coef, c, shape[::-1])[0]
    ref = ndimage.map_coordinates(x.astype(np.float64), c[::-1], order=3, mode="mirror")
    assert np.abs(got - ref).max() <= 1e-14


@pytest.mark.parametrize("rank", [2, 3])
def test_oracle_bspline_identity_and_constant(rank):
    x, g, _ = _case_bspline_identity(rank)
    _within_ulps(ori.resample_bspline(x, g, g), x)
    const = np.full((1,) + g.shape, 0.7, np.float32)
    centre = np.asarray(g.origin) + (np.asarray(g.size) - 1) / 2 * np.asarray(g.spacing)
    tgt = _oblique((9, 8, 7)[:rank], (1.1, 1.3, 0.9)[:rank], 13, centre=centre)
    out = ori.resample_bspline(const, g, tgt, SENTINEL)
    inside = out != SENTINEL
    assert inside.mean() > 0.3
    _within_ulps(out[inside], np.full(int(inside.sum()), 0.7, np.float32))


def test_oracle_bspline_nan_spreads_along_lines():
    x = _rand((1, 5, 6, 7), 14)
    x[0, 2, 3, 4] = np.nan
    coef = ori.bspline_coefficients(x, 3)
    assert np.isnan(coef).all()                                     # lines along x, then y, then z cover the volume
    x2 = _rand((1, 1, 6, 7), 14)
    x2[0, 0, 3, 4] = np.nan
    assert np.isnan(ori.bspline_coefficients(x2, 2)).all()


# ------------------------------------------------------------------------------------------- argument checks (CPU)
def test_resample_interpolation_arguments_are_validated_before_the_device():
    from mpgan.transforms import resample
    ImageGeometry, reference_grid = _geometries()
    src, tgt = ImageGeometry((6, 5, 4), (1, 1, 1), (0, 0, 0)), reference_grid(8)
    x = torch.zeros(2, 4, 5, 6)
    bad = [(x, dict(interpolation="cubic")), (x, dict(interpolation=None)), (x, dict(interpolation=3)),
           (x, dict(interpolation="Linear")), (x.double(), dict(interpolation="nearest")),
           (x.long(), dict(interpolation="nearest")), (x.short(), dict(interpolation="nearest")),
           (x.bool(), dict(interpolation="bspline")), (x.to(torch.uint8), dict(interpolation="bspline")),
           (x.double(), dict(interpolation="bspline")), (x.bool(), dict(interpolation="linear")),
           (x.bool(), dict(interpolation="nearest", default_value=2)),
           (x.bool(), dict(interpolation="nearest", default_value=0.5)),
           (x.to(torch.uint8), dict(interpolation="nearest", default_value=-1)),
           (x.to(torch.uint8), dict(interpolation="nearest", default_value=256)),
           (x.to(torch.uint8), dict(interpolation="nearest", default_value=math.nan)),
           (x.int(), dict(interpolation="nearest", default_value=2 ** 31)),
           (x.int(), dict(interpolation="nearest", default_value=-2 ** 31 - 1)),
           (x.int(), dict(interpolation="nearest", default_value=1.5)),
           (x.int(), dict(interpolation="nearest", default_value=math.inf)),
           (x, dict(interpolation="nearest", default_value="0")), (x, dict(interpolation="bspline", default_value=None)),
           (torch.zeros(2, 4, 6, 5), dict(interpolation="bspline"))]
    for img, kw in bad:
        with pytest.raises(ValueError):
            resample(img, src, tgt, **kw)
    ok = [(x, "nearest", -1.5), (x.bool(), "nearest", 1), (x.bool(), "nearest", False), (x.to(torch.uint8), "nearest", 255),
          (x.int(), "nearest", -2 ** 31), (x.int(), "nearest", 2 ** 31 - 1), (x, "bspline", -1.0), (x, "linear", 0)]
    for img, mode, dflt in ok:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            resample(img, src, tgt, default_value=dflt, interpolation=mode)


def test_c_abi_rejects_bad_input():
    import ctypes
    from mpgan import _lib
    from mpgan.transforms import resample_map
    lib = _lib.load()
    ImageGeometry, reference_grid = _geometries()
    p = 256   # device pointers are never dereferenced: the checks come first
    good3 = resample_map(_oblique((9, 8, 7), (1, 1, 1), 0), reference_grid(16))
    good2 = resample_map(ImageGeometry((9, 8), (1, 1), (0, 0), _rotation(1, 2)), reference_grid(16, rank=2))

    def grids(fn, m=good3, rank=3, ins=(9, 8, 7), outs=(16, 16, 16), items=1, x=p, y=p, sizes=True, mp=True, eb=4):
        i3 = (ctypes.c_int32 * 3)(*ins) if sizes else None
        o3 = (ctypes.c_int32 * 3)(*outs)
        mm = (ctypes.c_double * 24)(*m) if mp else None
        if fn == "nearest":
            return lib.mpgan_resample_nearest(x, eb, items, rank, i3, o3, mm, 0, y, None)
        return lib.mpgan_resample_bspline(x, items, rank, i3, o3, mm, 0.0, y, None)

    def edit(m, i, v):
        m = list(m)
        m[i] = v
        return m

    for fn in ("nearest", "bspline"):
        call = lambda **kw: grids(fn, **kw)   # noqa: E731
        for kw in (dict(x=None), dict(y=None), dict(sizes=False), dict(mp=False)):
            assert call(**kw) == -1 and "null" in _lib.last_error()
        assert call(items=0) == -1 and "items" in _lib.last_error()
        assert call(items=-3) == -1
        for r in (1, 4):
            assert call(rank=r) == -1 and "rank" in _lib.last_error()
        assert call(ins=(9, 0, 7)) == -1 and "extent" in _lib.last_error()
        assert call(outs=(16, 16, (1 << 22) + 1)) == -1 and "extent" in _lib.last_error()
        for i, v in ((0, math.nan), (7, math.inf), (20, -math.inf)):
            assert call(m=edit(good3, i, v)) == -1 and "not finite" in _lib.last_error()
        kw2 = dict(m=good2, rank=2, ins=(9, 8, 1), outs=(16, 16, 1))
        assert call(**dict(kw2, ins=(9, 8, 2))) == -1 and "z extents" in _lib.last_error()
        assert call(**dict(kw2, outs=(16, 16, 3))) == -1 and "z extents" in _lib.last_error()
        for i, v in ((3 + 2, 0.5), (3 + 7, 0.1), (3 + 8, 2.0), (15 + 6, 1.0), (15 + 5, -0.5)):
            assert call(**dict(kw2, m=edit(good2, i, v))) == -1 and "identity" in _lib.last_error()
        for i in (2, 14):
            assert call(**dict(kw2, m=edit(good2, i, 1.0))) == -1 and "z origins" in _lib.last_error()
        assert call(items=1 << 40) == -1 and "rows" in _lib.last_error()
    for eb in (0, 2, 3, 8, -1):
        assert grids("nearest", eb=eb) == -1 and "elem_bytes" in _lib.last_error()

    def coef(x=p, y=p, items=1, rank=3, size=(9, 8, 7), sizes=True):
        s3 = (ctypes.c_int32 * 3)(*size) if sizes else None
        return lib.mpgan_bspline_coefficients(x, items, rank, s3, y, None)

    for kw in (dict(x=None), dict(y=None), dict(sizes=False)):
        assert coef(**kw) == -1 and "null" in _lib.last_error()
    assert coef(items=0) == -1 and "items" in _lib.last_error()
    for r in (1, 4):
        assert coef(rank=r) == -1 and "rank" in _lib.last_error()
    assert coef(size=(9, 0, 7)) == -1 and "extent" in _lib.last_error()
    assert coef(size=((1 << 22) + 1, 1, 1)) == -1 and "extent" in _lib.last_error()
    assert coef(rank=2, size=(9, 8, 2)) == -1 and "z extents" in _lib.last_error()
    assert coef(items=1 << 40) == -1 and "rows" in _lib.last_error()
    assert coef(x=p, y=p) == -1 and "overlap" in _lib.last_error()


# ------------------------------------------------------------------------------------------------- CUDA kernels
def _dev(x, src, tgt, dflt=0, mode="nearest"):
    from mpgan.transforms import resample
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return resample(t, src, tgt, default_value=dflt, interpolation=mode).cpu().numpy()


def _dev_coef(x, rank):
    from mpgan import ops
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()
    coef = torch.empty(t.shape, dtype=torch.float64, device="cuda")
    size = tuple(t.shape[::-1][:rank]) + (1,) * (3 - rank)
    ops.bspline_coefficients(t, math.prod(t.shape[:t.dim() - rank]), rank, size, coef)
    return coef.cpu().numpy()


def _nearest_both_ways(x, native, model):
    fwd = _dev(x, native, model, 0)
    _same_bits(fwd, ori.resample_nearest(x, native, model, 0))
    back = _dev(fwd, model, native, 1)
    _same_bits(back, ori.resample_nearest(fwd, model, native, 1))


def _bspline_both_ways(x, native, model):
    rank = native.rank
    coef = _dev_coef(x, rank)
    want = ori.bspline_coefficients(x.reshape((-1,) + (native.size + (1,) * (3 - rank))[::-1]), rank)
    assert np.array_equal(coef.reshape(want.shape).view(np.uint64), want.view(np.uint64))
    fwd = _dev(x, native, model, SENTINEL, "bspline")
    _same_bits(fwd, ori.resample_bspline(x, native, model, SENTINEL, coef=want))
    inside = fwd != SENTINEL
    assert 0.01 < inside.mean() < 0.99
    back = _dev(fwd, model, native, SENTINEL, "bspline")
    _same_bits(back, ori.resample_bspline(fwd, model, native, SENTINEL))
    assert 0.01 < (back != SENTINEL).mean()


OBLIQUE = [((61, 67, 13), (1.7, 2.3, 4.1), 11), ((45, 70, 37), (3.1, 1.9, 2.6), 12), ((61, 67, 13), (4.3, 3.7, 9.5), 13)]


@gpu
@pytest.mark.parametrize("dtype", sorted(MASK_DTYPES))
@pytest.mark.parametrize("size,spacing,seed", OBLIQUE)
def test_nearest_oblique_round_trip_matches_oracle_bit_exact(size, spacing, seed, dtype):
    _, reference_grid = _geometries()
    native = _oblique(size, spacing, seed)
    _nearest_both_ways(_values((2,) + native.shape, seed, MASK_DTYPES[dtype]), native, reference_grid(128))


@gpu
@pytest.mark.parametrize("size,spacing,seed", OBLIQUE)
def test_bspline_oblique_round_trip_matches_oracle_bit_exact(size, spacing, seed):
    _, reference_grid = _geometries()
    native = _oblique(size, spacing, seed)
    _bspline_both_ways(_rand((2,) + native.shape, seed), native, reference_grid(128))


@gpu
def test_native_1mm_volume_matches_oracle_bit_exact():
    _, reference_grid = _geometries()
    native = _oblique((256, 256, 176), (1.0, 1.0, 1.0), 21)
    x = _rand(native.shape, 21, 0.0, 1000.0)
    _bspline_both_ways(x, native, reference_grid())
    for dtype in (np.uint8, np.int32):
        _nearest_both_ways(_values(native.shape, 21, dtype), native, reference_grid())


@gpu
def test_rank2_slices_match_oracle_bit_exact():
    _, reference_grid = _geometries()
    native = _oblique((512, 512), (0.5, 0.5), 22)
    model = reference_grid(256, 256.0, rank=2)
    _bspline_both_ways(_rand((3, 1) + native.shape, 22), native, model)
    for dtype in MASK_DTYPES.values():
        _nearest_both_ways(_values((3, 1) + native.shape, 22, dtype), native, model)


@gpu
@pytest.mark.parametrize("name", sorted(NEAREST_KNOWN))
def test_nearest_known_answers_on_device(name):
    x, src, tgt, dflt, want = NEAREST_KNOWN[name]()
    _same_bits(_dev(x, src, tgt, dflt), want)


@gpu
@pytest.mark.parametrize("n", [1, 2, 4, 1024])
def test_clamp_on_device(n):
    x, src, tgt, _ = _case_clamp(n)
    assert np.array_equal(_dev(x, src, tgt, SENTINEL)[0, :, 0], x[0, :, n - 1])
    _same_bits(_dev(x, src, tgt, SENTINEL, "bspline"), ori.resample_bspline(x, src, tgt, SENTINEL))


@gpu
@pytest.mark.parametrize("rank", [2, 3])
def test_bspline_known_answers_on_device(rank):
    x, g, _ = _case_bspline_identity(rank)
    _within_ulps(_dev(x, g, g, 0.0, "bspline"), x)
    const = np.full((1,) + g.shape, 0.7, np.float32)
    centre = np.asarray(g.origin) + (np.asarray(g.size) - 1) / 2 * np.asarray(g.spacing)
    tgt = _oblique((9, 8, 7)[:rank], (1.1, 1.3, 0.9)[:rank], 13, centre=centre)
    out = _dev(const, g, tgt, SENTINEL, "bspline")
    inside = out != SENTINEL
    assert inside.mean() > 0.3
    _within_ulps(out[inside], np.full(int(inside.sum()), 0.7, np.float32))


@gpu
@pytest.mark.parametrize("shape", [(1, 1, 5), (1, 2, 5), (2, 2, 2), (3, 1, 2), (40, 33, 1), (5, 70, 65)])
def test_bspline_small_and_chunk_edge_extents_on_device(shape):
    """Extents 1 and 2, and x extents around the x pass's 32-column chunks, against the oracle bit for bit."""
    ImageGeometry, _ = _geometries()
    x = _rand((2,) + shape, 23, -1.0, 2.0)
    src = ImageGeometry(shape[::-1], (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    coef = _dev_coef(x, 3)
    want = ori.bspline_coefficients(x, 3)
    assert np.array_equal(coef.view(np.uint64), want.view(np.uint64))
    tgt = _oblique(tuple(max(2 * n, 3) for n in shape[::-1]), (0.5, 0.5, 0.5), 24,
                   centre=(np.asarray(shape[::-1], dtype=np.float64) - 1) / 2)
    out = _dev(x, src, tgt, SENTINEL, "bspline")
    _same_bits(out, ori.resample_bspline(x, src, tgt, SENTINEL, coef=want))
    assert (out != SENTINEL).any()


@gpu
def test_nan_on_device():
    """Nearest copies a NaN payload only where its voxel is chosen; the spline spreads it where the oracle does."""
    x, src, tgt, dflt, want = _case_nan()
    _same_bits(_dev(x, src, tgt, dflt), want)
    x = _rand((1, 9, 10, 40), 25)
    x[0, 4, 5, 20] = np.nan
    ImageGeometry, _ = _geometries()
    src = ImageGeometry((40, 10, 9), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    tgt = _oblique((30, 12, 10), (1.2, 0.9, 1.0), 26, centre=(19.5, 4.5, 4.0))
    got, ref = _dev(x, src, tgt, SENTINEL, "bspline"), ori.resample_bspline(x, src, tgt, SENTINEL)
    assert np.array_equal(np.isnan(got), np.isnan(ref)) and np.isnan(got).any()
    assert np.array_equal(got[~np.isnan(got)], ref[~np.isnan(ref)])


@gpu
@pytest.mark.parametrize("mode,dtype", [("nearest", torch.uint8), ("nearest", torch.int32), ("bspline", torch.float32)])
def test_batched_call_equals_separate_calls(mode, dtype):
    from mpgan.transforms import resample
    _, reference_grid = _geometries()
    native = _oblique((45, 70, 37), (3.1, 1.9, 2.6), 31)
    x = torch.from_numpy(_rand((3,) + native.shape, 31, 0.0, 200.0)).cuda().to(dtype)
    tgt = reference_grid(64)
    both = resample(x, native, tgt, default_value=7, interpolation=mode)
    for i in range(3):
        assert torch.equal(both[i], resample(x[i], native, tgt, default_value=7, interpolation=mode))


@gpu
@pytest.mark.parametrize("mode", ["nearest", "bspline"])
def test_repetition_and_graph_replay_change_no_bit(mode):
    from mpgan.transforms import resample
    _, reference_grid = _geometries()
    native = _oblique((61, 67, 13), (1.7, 2.3, 4.1), 32)
    model = reference_grid(128)
    x = torch.from_numpy(_rand((2,) + native.shape, 32)).cuda()
    base = resample(x, native, model, default_value=SENTINEL, interpolation=mode)
    for _ in range(3):
        assert torch.equal(resample(x, native, model, default_value=SENTINEL, interpolation=mode), base)
    static = x.clone()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = resample(static, native, model, default_value=SENTINEL, interpolation=mode)
    for _ in range(2):
        out.fill_(0.0)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, base)
    static.copy_(torch.flip(x, [0]))
    g.replay()
    assert torch.equal(out, torch.flip(base, [0]))


@gpu
def test_native_grid_scoring_chain_end_to_end_against_oracle():
    """native T1 -> reference_grid(32) (linear) -> 32^3 generator -> back to native (bspline); the Otsu head mask of
    the model-grid truth, cleaned, moved to native (nearest); masked MAE on the native grid."""
    from mpgan import CasNetGenerator, inference
    from mpgan.transforms import ScaleIntensityRangePercentiles, foreground_mask, mean_absolute_error, resample
    from oracle import masked_metrics as omm
    from oracle import morphology as omo
    from oracle import transforms as otf
    from oracle.nets import CasNetGenerator as OGen
    _, reference_grid = _geometries()
    native = _oblique((45, 70, 37), (3.1, 4.4, 3.3), 41)
    model_grid = reference_grid(32)
    t1 = _rand(native.shape, 41, 0.0, 800.0)
    zz, yy, xx = np.meshgrid(*[np.linspace(-1, 1, n) for n in native.shape], indexing="ij")
    head = (zz ** 2 + yy ** 2 + xx ** 2) < 0.5
    t2 = np.where(head, _rand(native.shape, 42, 0.2, 1.0), _rand(native.shape, 43, -1.0, -0.9)).astype(np.float32)

    torch.manual_seed(0)
    ora = OGen((1, 32, 32, 32), 6, 3).eval()
    gen = CasNetGenerator((1, 32, 32, 32), precision="fp32")
    gen.load_state_dict(ora.state_dict())
    gen.cuda()

    x = ors.resample(t1, native, model_grid)
    x = otf.scale_intensity_range_percentiles(x, 1, 99, -1.0, 1.0, clip=True)
    with torch.no_grad():
        y = ora(torch.from_numpy(x)[None, None]).numpy()[0, 0]
    gen_ref = ori.resample_bspline(y, model_grid, native, -1.0)
    truth_model = ors.resample(t2, native, model_grid, -1.0)
    mask_model = omo.foreground_mask(truth_model, largest=True, fill=True)
    mask_ref = ori.resample_nearest(mask_model, model_grid, native, False)
    mae_ref = omm.mean_absolute_error(gen_ref, t2, mask_ref)

    def chain():
        v = resample(torch.from_numpy(t1).cuda(), native, model_grid)
        v = ScaleIntensityRangePercentiles(1, 99, -1.0, 1.0, clip=True)(v)
        out = inference.infer_volume(gen, v[None, None])
        g = resample(out[0, 0], model_grid, native, default_value=-1.0, interpolation="bspline")
        tm = resample(torch.from_numpy(t2).cuda(), native, model_grid, default_value=-1.0)
        m = foreground_mask(tm, largest_component=True, fill_holes=True)
        m = resample(m, model_grid, native, default_value=False, interpolation="nearest")
        return g, m, mean_absolute_error(g, torch.from_numpy(t2).cuda(), mask=m)

    g, m, mae = chain()
    assert g.shape == native.shape and m.dtype == torch.bool and rel_l2(g, torch.from_numpy(gen_ref)) <= 1e-4
    assert np.array_equal(m.cpu().numpy(), mask_ref) and 0.05 < mask_ref.mean() < 0.6
    assert abs(float(mae) - mae_ref) <= 1e-4 * abs(mae_ref)
    gen.set_precision("bf16")
    g, m, mae = chain()
    assert rel_l2(g, torch.from_numpy(gen_ref)) <= 1e-2 and abs(float(mae) - mae_ref) <= 1e-2 * abs(mae_ref)
