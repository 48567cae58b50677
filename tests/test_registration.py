"""Rigid registration by Mattes mutual information, the Gaussian filter of its pyramid, and resampling through the
registered transform: ``mpgan.transforms.register_rigid``, ``gaussian_filter`` and ``resample(..., transform=)`` over
csrc/registration.cu and the map-reading kernels of csrc/resample.cu.

CPU tests hold the numpy restatement (oracle/registration.py) to independent references: scipy's rotations and
Gaussian filter, finite differences of its own metric, known answers, and end-to-end recovery of known rigid offsets
on a phantom head whose T1 and T2 contrasts no monotonic map relates.  They also check that argument errors are raised
before the device is touched and that the C ABI rejects bad input.  ``-m gpu`` tests hold the kernels to the oracle
(bit for bit where include/mpgan.h promises bits) and run the recovery, batching, graph-capture and scoring chains."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy import ndimage
from scipy.spatial.transform import Rotation

from oracle import registration as orr

gpu = pytest.mark.gpu


def _tf():
    import mpgan.transforms as t
    return t


def _grid(size, spacing, origin=None, direction=None):
    t = _tf()
    rank = len(size)
    if origin is None:
        origin = tuple(-n * s / 2.0 for n, s in zip(size, (spacing,) * rank if np.isscalar(spacing) else spacing))
    return t.ImageGeometry(size, (spacing,) * rank if np.isscalar(spacing) else spacing, origin, direction)


def _oblique(rank, seed):
    rs = np.random.RandomState(seed)
    if rank == 2:
        a = rs.uniform(-0.4, 0.4)
        return [[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]]
    return Rotation.from_rotvec(rs.normal(size=3) * 0.3).as_matrix().tolist()


def _fixed_points(geometry, mask=None):
    """(3, N) physical points of the fixed voxels (in ``mask``)."""
    t = _tf()
    size = tuple(geometry.size) + (1,) * (3 - geometry.rank)
    ix, iy, iz = orr.sample_indices(size, 1, mask)
    m, o = t._lift3(geometry.index_to_physical(), geometry.origin)
    return np.stack([o[k] + m[k, 0] * ix + m[k, 1] * iy + m[k, 2] * iz for k in range(3)])


def _offsets(rank, seed, n):
    """n rigid offsets with angles up to 10 degrees and translations up to 10 mm."""
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        if rank == 3:
            ang = rs.normal(size=3)
            ang *= math.radians(rs.uniform(4, 10)) / np.linalg.norm(ang)
            tr = rs.normal(size=3)
            tr *= rs.uniform(4, 10) / np.linalg.norm(tr)
            out.append(np.concatenate([ang, tr]))
        else:
            tr = rs.normal(size=2)
            tr *= rs.uniform(4, 10) / np.linalg.norm(tr)
            out.append(np.array([rs.choice([-1, 1]) * math.radians(rs.uniform(4, 10)), *tr]))
    return out


def _level(f3, m3, moving_geometry, rank, shrink=1, mask=None):
    samples = orr.sample_indices(f3.shape[::-1], shrink, mask)
    rng = orr.ranges(f3, m3, samples)
    nn = _tf().resample_map(moving_geometry, moving_geometry)[15:24]
    return samples, rng, orr.index_gradient(m3), [nn[0:3], nn[3:6], nn[6:9]]


# ---- CPU: the oracle against independent references -------------------------------------------------------------------
def test_euler_matches_scipy_zxy():
    rs = np.random.RandomState(0)
    for _ in range(20):
        th = rs.uniform(-3.5, 3.5, 3)
        r, _ = orr.euler([np.float64(v) for v in th], 3)
        ref = Rotation.from_euler("ZXY", [th[2], th[0], th[1]]).as_matrix()
        assert np.abs(np.array(r, dtype=np.float64) - ref).max() < 1e-14
        r2, _ = orr.euler([np.float64(th[0])], 2)
        ref2 = Rotation.from_euler("z", th[0]).as_matrix()
        assert np.abs(np.array(r2, dtype=np.float64) - ref2).max() < 1e-14
    s, c = orr.sincos(np.linspace(-40, 40, 10001))
    assert np.abs(s - np.sin(np.linspace(-40, 40, 10001))).max() < 2e-15
    assert np.abs(c - np.cos(np.linspace(-40, 40, 10001))).max() < 2e-15


@pytest.mark.parametrize("rank", [2, 3])
def test_composed_map_sends_fixed_points_through_the_transform(rank):
    t = _tf()
    fg = _grid((7, 5, 4)[:rank], (1.5, 2.0, 2.5)[:rank], direction=_oblique(rank, 1))
    mg = _grid((6, 9, 5)[:rank], (1.0, 1.25, 3.0)[:rank], origin=(3.0, -4.0, 2.0)[:rank], direction=_oblique(rank, 2))
    c = t.grid_center(fg)
    prm = np.array([0.1, -0.2, 0.3, 4.0, -5.0, 6.0] if rank == 3 else [0.3, 4.0, -5.0])
    m, _ = orr.compose(prm, t.resample_map(mg, fg), c, rank)
    size = tuple(fg.size) + (1,) * (3 - rank)
    got = orr.map_index(m, *orr.grid_index(size))
    p = _fixed_points(fg)
    r = Rotation.from_euler("ZXY", [prm[2], prm[0], prm[1]]).as_matrix() if rank == 3 else \
        Rotation.from_euler("z", prm[0]).as_matrix()
    tt = list(prm[3:]) if rank == 3 else [prm[1], prm[2], 0.0]
    q = r @ (p - np.array(c)[:, None]) + np.array(c)[:, None] + np.array(tt)[:, None]
    mm, mo = t._lift3(mg.physical_to_index(), mg.origin)
    want = mm @ (q - np.array(mo)[:, None])
    assert np.abs(got.reshape(3, -1) - want).max() < 1e-9


def _smooth_pair(rank, n, seed, mask):
    fg = _grid((n,) * rank, 4.0)
    f = orr.phantom(fg, "t1", edge_mm=6.0)
    m = orr.phantom(fg, "t2", _offsets(rank, seed, 1)[0] * 0.5, _tf().grid_center(fg), edge_mm=6.0)
    taps = [_tf().gaussian_taps(2.0)] * rank + [[1.0]] * (3 - rank)
    f3 = orr.gaussian_filter(f.reshape((1,) * (3 - rank) + f.shape), taps, 3)
    m3 = orr.gaussian_filter(m.reshape(f3.shape), taps, 3)
    return fg, f3, m3, (f3 > 0.05) if mask else None


@pytest.mark.parametrize("rank,mask", [(2, False), (2, True), (3, False), (3, True)])
def test_oracle_gradient_matches_finite_differences(rank, mask):
    """The analytic gradient uses the central-difference image gradient, not the derivative of the linear interpolant
    the value uses; on these images, smoothed with sigma = 2 voxels, the two differ by 3-6 % of the gradient's norm
    (the largest component difference over the four cases), so the check is 10 % of the norm per component.  The step
    (1e-3 rad, 1e-2 mm) stays far inside a voxel and far above the 2^-32 quantisation of the histogram."""
    t = _tf()
    fg, f3, m3, mk = _smooth_pair(rank, 64 if rank == 2 else 32, 3, mask)
    samples, rng, g3, nn = _level(f3, m3, fg, rank, 1, mk)
    base, c = t.resample_map(fg, fg), t.grid_center(fg)
    rs = np.random.RandomState(rank)
    for _ in range(2):
        prm = np.concatenate([rs.uniform(-0.05, 0.05, 3 if rank == 3 else 1), rs.uniform(-3, 3, rank)])
        m, d = orr.compose(prm, base, c, rank)
        g = orr.mattes(f3, m3, g3, samples, rng, m, d, nn, rank, 50)["gradient"]
        fd = []
        for j in range(len(prm)):
            h = 1e-3 if j < len(prm) - rank else 1e-2
            v = []
            for sgn in (1, -1):
                q = prm.copy()
                q[j] += sgn * h
                mq, dq = orr.compose(q, base, c, rank)
                v.append(orr.mattes(f3, m3, g3, samples, rng, mq, dq, nn, rank, 50, want_gradient=False)["metric"])
            fd.append((v[0] - v[1]) / (2 * h))
        fd = np.array(fd)
        scale = np.array(orr.rotation_scales(samples, f3.shape[::-1], base[3:12], rank, 4.0) + [1.0] * rank)
        gu, fu = g / scale, fd / scale
        assert np.abs(gu - fu).max() <= 0.1 * np.linalg.norm(fu), (gu, fu)


@pytest.mark.parametrize("shape,sigma", [((17, 23), 1.3), ((5, 9, 12), (0.0, 2.0, 0.7)), ((2, 3, 40), 3.0)])
def test_oracle_gaussian_matches_scipy(shape, sigma):
    t = _tf()
    x = np.random.RandomState(0).normal(size=shape).astype(np.float32)
    per = list(sigma) if isinstance(sigma, tuple) else [sigma] * len(shape)
    taps = [t.gaussian_taps(s) for s in per[::-1]] + [[1.0]] * (3 - len(shape))
    got = orr.gaussian_filter(x.reshape((1,) * (3 - len(shape)) + shape), taps, 3).reshape(shape)
    ref = ndimage.gaussian_filter(x.astype(np.float64), per, mode="reflect", truncate=4.0)
    assert np.all(np.abs(got - ref) <= 2.0 ** -23 * np.abs(ref) + 1e-12)


def test_identical_images_at_identity_maximise_mi():
    t = _tf()
    fg = _grid((40, 40), 2.0)
    f = orr.phantom(fg, "t1", edge_mm=4.0)
    f3 = f.reshape((1,) + f.shape)
    samples, rng, g3, nn = _level(f3, f3, fg, 2)
    base, c = t.resample_map(fg, fg), t.grid_center(fg)
    at = lambda p: orr.mattes(f3, f3, g3, samples, rng, *orr.compose(np.array(p), base, c, 2), nn, 2, 50,
                              want_gradient=False)["metric"]
    m0 = at([0.0, 0.0, 0.0])
    for p in ([0.01, 0, 0], [-0.01, 0, 0], [0, 0.3, 0], [0, -0.3, 0], [0, 0, 0.3], [0, 0, -0.3], [0.005, 0.2, -0.2]):
        assert at(p) > m0


def test_flat_image_and_no_overlap_give_nan_and_status():
    fg = _grid((32, 32), 2.0)
    f = orr.phantom(fg, "t1")
    r = orr.register_one(f, np.full_like(f, 0.5), fg, fg, iterations=3)
    assert r["status"] == orr.FLAT and math.isnan(r["metric"])
    far = _grid((32, 32), 2.0, origin=(1000.0, 1000.0))
    r = orr.register_one(f, f, fg, far, initialize="identity", iterations=3)
    assert r["status"] == orr.OVERLAP and math.isnan(r["metric"])
    np.testing.assert_array_equal(r["parameters"], [0.0, 0.0, 0.0])


@pytest.mark.parametrize("rank,n,spacing,seed,count", [(2, 128, 2.0, 0, 3), (3, 48, 4.0, 1, 2)])
def test_oracle_recovers_known_offsets(rank, n, spacing, seed, count):
    """The algorithm and its defaults, before any GPU: mean displacement of the fixed head mask's voxels between the
    recovered and the true transform below a quarter of a fixed voxel."""
    t = _tf()
    fg = _grid((n,) * rank, spacing)
    c = t.grid_center(fg)
    fixed = orr.phantom(fg, "t1", edge_mm=1.5 * spacing)
    mask = fixed > 0.05
    pts = _fixed_points(fg, mask)
    for true in _offsets(rank, seed, count):
        moving = orr.phantom(fg, "t2", true, c, edge_mm=1.5 * spacing)
        r = orr.register_one(fixed, moving, fg, fg, fixed_mask=mask)
        assert r["status"] in (orr.CONVERGED, orr.ITERATIONS)
        assert orr.displacement(r["parameters"], true, c, rank, pts) < 0.25 * spacing, (true, r["parameters"])


# ---- CPU: validation and the C ABI ----------------------------------------------------------------------------------
def test_arguments_are_validated_before_the_device():
    t = _tf()
    fg = _grid((16, 16, 16), 2.0)
    f = torch.zeros(fg.shape)
    ok = dict(fixed_geometry=fg, moving_geometry=fg)
    bad = [dict(bins=7), dict(bins=129), dict(bins=50.0), dict(shrink_factors=(4, 2), smoothing_sigmas=(1.0,)),
           dict(shrink_factors=(0,), smoothing_sigmas=(0.0,)), dict(smoothing_sigmas=(2.0, -1.0, 0.0)),
           dict(smoothing_sigmas=(16.2, 1.0, 0.0)), dict(iterations=0), dict(initialize="moments"),
           dict(initial_parameters=torch.zeros(3, dtype=torch.float64)),
           dict(fixed_mask=torch.zeros(16, 16, dtype=torch.bool)), dict(fixed_mask=torch.zeros(fg.shape))]
    for kw in bad:
        with pytest.raises(ValueError):
            t.register_rigid(f, f, **ok, **kw)
    with pytest.raises(ValueError):
        t.register_rigid(f.double(), f, **ok)
    with pytest.raises(ValueError):
        t.register_rigid(f, torch.zeros(16, 16, 15), **ok)
    with pytest.raises(ValueError):
        t.register_rigid(f, f, fg, _grid((16, 16), 2.0))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        t.register_rigid(f, f, **ok)
    for sig in (-1.0, 16.2, float("nan"), (1.0, 1.0)):
        with pytest.raises(ValueError):
            t.gaussian_filter(f, sig)
    with pytest.raises(ValueError):
        t.gaussian_filter(f.double(), 1.0)
    tf3 = t.RigidTransform(torch.zeros(6, dtype=torch.float64), (0.0, 0.0, 0.0))
    tf2 = t.RigidTransform(torch.zeros(2, 3, dtype=torch.float64), (0.0, 0.0))
    with pytest.raises(ValueError):
        t.resample(f, fg, fg, transform=tf2)
    with pytest.raises(ValueError):
        t.resample(f, fg, fg, transform="identity")
    with pytest.raises(ValueError):
        t.resample(torch.zeros((2,) + fg.shape), fg, fg, transform=tf3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        t.resample(f, fg, fg, transform=tf3)
    with pytest.raises(ValueError):
        t.RigidTransform(torch.zeros(4, dtype=torch.float64), (0.0, 0.0))


def test_c_abi_rejects_bad_arguments():
    from mpgan import _lib
    lib = _lib.load()
    i3 = lambda *v: (ctypes.c_int32 * 3)(*v)
    d = lambda n, v=0.0: (ctypes.c_double * n)(*([v] * n))
    dummy = ctypes.c_void_p(4096)
    ws = lib.mpgan_mattes_workspace(1, i3(8, 8, 8), i3(8, 8, 8), 50)
    assert ws > 0
    E = -1
    cases = [
        lambda: lib.mpgan_mattes_prepare(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 8, 8), 1, 7, d(9, 1.0), 1.0, dummy, dummy,
                                         dummy, ws, None),                                          # bins
        lambda: lib.mpgan_mattes_prepare(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 8, 8), 0, 50, d(9, 1.0), 1.0, dummy, dummy,
                                         dummy, ws, None),                                          # shrink
        lambda: lib.mpgan_mattes_prepare(dummy, dummy, None, 1, 2, i3(8, 8, 2), i3(8, 8, 1), 1, 50, d(9, 1.0), 1.0, dummy, dummy,
                                         dummy, ws, None),                                          # rank-2 z
        lambda: lib.mpgan_mattes_prepare(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 8, 8), 1, 50, d(9, 1.0), 1.0, dummy, dummy,
                                         dummy, ws - 1, None),                                      # short workspace
        lambda: lib.mpgan_mattes_prepare(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 8, 8), 1, 50, d(9, 1.0), 0.0,
                                         dummy, dummy, dummy, ws, None),                            # min_scale
        lambda: lib.mpgan_mattes_evaluate(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 0, 8), 1, 50, 1, 1, dummy,
                                          dummy, dummy, dummy, dummy, ws, None),                    # extent
        lambda: lib.mpgan_mattes_evaluate(dummy, dummy, None, 1, 3, i3(8, 8, 8), i3(8, 8, 8), 1, 50, 1, 1, dummy,
                                          dummy, None, dummy, dummy, ws, None),                     # null hist
        lambda: lib.mpgan_gaussian_filter(dummy, 1, 3, i3(8, 8, 8), i3(1, 65, 1), d(200, 0.1), ctypes.c_void_p(8192),
                                          dummy, 1 << 20, None),                                    # radius
        lambda: lib.mpgan_gaussian_filter(dummy, 1, 3, i3(8, 8, 8), i3(0, 0, 0), d(3, 1.0), ctypes.c_void_p(8192),
                                          ctypes.c_void_p(1 << 20), 10, None),                      # workspace
        lambda: lib.mpgan_gaussian_filter(dummy, 1, 3, i3(8, 8, 8), i3(0, 0, 0), d(3, 1.0), ctypes.c_void_p(4096 + 64),
                                          ctypes.c_void_p(1 << 20), 1 << 20, None),                 # overlap
        lambda: lib.mpgan_gaussian_filter(dummy, 1, 3, i3(8, 8, 8), i3(0, 0, 0), d(3, float("nan")),
                                          ctypes.c_void_p(8192), ctypes.c_void_p(1 << 20), 1 << 20, None),  # taps
        lambda: lib.mpgan_rigid_step(dummy, dummy, 1, 3, d(24), d(3), 0.0, 0, None),               # min_step
        lambda: lib.mpgan_rigid_level(dummy, dummy, 1, 4, d(24), d(3), None, d(3), 1, 1.0, None),   # rank
        lambda: lib.mpgan_rigid_maps(dummy, 1, 3, d(24, float("inf")), d(3), dummy, None),          # base
        lambda: lib.mpgan_resample_linear_maps(dummy, 1, 2, i3(4, 4, 2), i3(4, 4, 1), dummy, 0.0, dummy, None),
        lambda: lib.mpgan_resample_nearest_maps(dummy, 2, 1, 3, i3(4, 4, 4), i3(4, 4, 4), dummy, 0, dummy, None),
        lambda: lib.mpgan_resample_bspline_maps(dummy, 1, 3, i3(4, 4, 4), i3(4, 4, 4), None, 0.0, dummy, None),
    ]
    for k, call in enumerate(cases):
        assert call() == E, (k, _lib.last_error())


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _cuda(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda() if dtype is None else \
        torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dtype)


METRIC_CASES = [  # rank, fixed size, moving size, oblique, mask, shrink, bins
    (2, (61, 47), (55, 70), False, False, 1, 50),
    (2, (61, 47), (55, 70), True, True, 2, 32),
    (3, (33, 29, 21), (30, 35, 27), True, True, 1, 50),
    (3, (33, 29, 21), (30, 35, 27), True, False, 2, 128),
    (3, (40, 37, 33), (36, 40, 31), False, True, 4, 8),
    (3, (40, 37, 33), (36, 40, 31), True, True, 3, 64),
]


@gpu
@pytest.mark.parametrize("case", METRIC_CASES)
def test_metric_kernels_match_oracle(case):
    from mpgan import ops
    t = _tf()
    rank, fs, ms, oblique, use_mask, shrink, bins = case
    fg = _grid(fs, 3.0, direction=_oblique(rank, 5) if oblique else None)
    mg = _grid(ms, (2.9, 3.1, 3.3)[:rank], origin=tuple(-n * 3.0 / 2 + 1.7 for n in ms),
               direction=_oblique(rank, 6) if oblique else None)
    c = t.grid_center(fg)
    fixed = orr.phantom(fg, "t1", edge_mm=5.0)
    prms = [np.array(p) * 0.4 for p in _offsets(rank, 7, 2)]
    moving = np.stack([orr.phantom(mg, "t2", p, c, edge_mm=5.0) for p in prms])
    fixed2 = np.stack([fixed, fixed[::-1].copy()])
    mask = (fixed2 > 0.05) if use_mask else None
    items = 2
    fsize, msize = tuple(fs) + (1,) * (3 - rank), tuple(ms) + (1,) * (3 - rank)
    plan = t._registration_plan(fg, mg, (shrink,), (0.0,), "identity")
    state = torch.empty(items, 96, dtype=torch.float64, device="cuda")
    status = torch.empty(items, dtype=torch.int32, device="cuda")
    hist = torch.empty(items, bins, bins, dtype=torch.int64, device="cuda")
    metric = torch.empty(items, dtype=torch.float64, device="cuda")
    ws = ops.mattes_workspace(items, fsize, msize, bins, "cuda")
    init = _cuda(np.stack(prms))
    fd, md = _cuda(fixed2), _cuda(moving)
    mk = None if mask is None else _cuda(mask).view(torch.uint8)
    ops.rigid_level(state, status, items, rank, plan["base"], plan["center"], init, [0.0] * 3, True, 1.0)
    ops.mattes_prepare(fd, md, mk, items, rank, fsize, msize, shrink, bins, plan["base"][3:12], 3.0, state, status,
                       ws)
    ops.mattes_evaluate(fd, md, mk, items, rank, fsize, msize, shrink, bins, True, True, state, status, hist, metric, ws)
    st, hs, mt = state.cpu().numpy(), hist.cpu().numpy(), metric.cpu().numpy()
    assert (status.cpu().numpy() == -1).all()
    nn = plan["base"][15:24]
    for i in range(items):
        m, d = orr.compose(prms[i], plan["base"], plan["center"], rank)
        np.testing.assert_array_equal(st[i, 6:30], np.array(m))
        f3 = fixed2[i].reshape(fsize[::-1])
        m3 = moving[i].reshape(msize[::-1])
        samples = orr.sample_indices(fsize, shrink, None if mask is None else mask[i])
        rng = orr.ranges(f3, m3, samples)
        ref = orr.mattes(f3, m3, orr.index_gradient(m3), samples, rng, m, d, [nn[0:3], nn[3:6], nn[6:9]], rank, bins)
        np.testing.assert_array_equal(hs[i], ref["hist"])
        nrot = 3 if rank == 3 else 1
        np.testing.assert_array_equal(st[i, 88:88 + nrot],
                                      orr.rotation_scales(samples, fsize, plan["base"][3:12], rank, 3.0))
        assert abs(mt[i] - ref["metric"]) <= 1e-12 * abs(ref["metric"])
        P = len(prms[i])
        assert np.abs(st[i, 66:66 + P] - ref["gradient"]).max() <= 1e-9 * np.linalg.norm(ref["gradient"])


@gpu
@pytest.mark.parametrize("shape,sigma,nd", [((3, 37, 129), 1.3, 2), ((2, 21, 34, 140), (0.0, 2.0, 0.7), 3),
                                            ((40, 41, 42), 3.0, 3), ((1, 9, 300), 15.0, 2)])
def test_gaussian_filter_matches_scipy_and_oracle(shape, sigma, nd):
    t = _tf()
    x = np.random.RandomState(1).normal(size=shape).astype(np.float32)
    got = t.gaussian_filter(_cuda(x), sigma, spatial_dims=nd).cpu().numpy()
    per = list(sigma) if isinstance(sigma, tuple) else [sigma] * nd
    taps = [t.gaussian_taps(s) for s in per[::-1]] + [[1.0]] * (3 - nd)
    lead = shape[:len(shape) - nd]
    x3 = x.reshape((-1,) + (1,) * (3 - nd) + shape[len(shape) - nd:])
    want = np.stack([orr.gaussian_filter(v, taps, 3) for v in x3]).reshape(shape)
    np.testing.assert_array_equal(got, want)
    ref = ndimage.gaussian_filter(x.astype(np.float64), [0.0] * len(lead) + per, mode="reflect", truncate=4.0)
    assert np.all(np.abs(got - ref) <= 2.0 ** -23 * np.abs(ref) + 1e-12)


@gpu
@pytest.mark.parametrize("rank", [2, 3])
def test_resample_through_transform_matches_oracle(rank):
    t = _tf()
    src = _grid((37, 29, 23)[:rank], (1.1, 1.3, 1.7)[:rank], direction=_oblique(rank, 8))
    dst = _grid((31, 33, 19)[:rank], (1.4, 1.2, 1.9)[:rank], origin=(-20.0, -19.0, -15.0)[:rank],
                direction=_oblique(rank, 9))
    prms = np.stack([np.array(p) * 0.5 for p in _offsets(rank, 11, 3)])
    tf = t.RigidTransform(_cuda(prms), t.grid_center(dst)[:rank])
    base = t.resample_map(src, dst)
    rs = np.random.RandomState(2)
    size_in, size_out = tuple(src.size) + (1,) * (3 - rank), tuple(dst.size) + (1,) * (3 - rank)
    imgs = {"float32": rs.normal(size=(3,) + src.shape).astype(np.float32),
            "bool": rs.uniform(size=(3,) + src.shape) > 0.5,
            "uint8": rs.randint(0, 255, size=(3,) + src.shape).astype(np.uint8),
            "int32": rs.randint(-9, 9, size=(3,) + src.shape).astype(np.int32)}
    maps = tf._maps(base).cpu().numpy()
    for i in range(3):
        np.testing.assert_array_equal(maps[i], orr.compose(prms[i], base, t.grid_center(dst), rank)[0])
    for mode, dtypes in (("linear", ["float32"]), ("bspline", ["float32"]), ("nearest", list(imgs))):
        for dt in dtypes:
            x = imgs[dt]
            dflt = 7 if dt != "bool" else 1
            got = t.resample(_cuda(x), src, dst, transform=tf, interpolation=mode, default_value=dflt).cpu().numpy()
            for i in range(3):
                want = orr.resample_mapped(x[i], size_in, size_out, list(maps[i]), dflt, mode).reshape(dst.shape)
                np.testing.assert_array_equal(got[i].view(np.uint8), want.view(np.uint8), err_msg=f"{mode} {dt}")
    ident = t.RigidTransform(torch.zeros(3, len(prms[0]), dtype=torch.float64, device="cuda"),
                             t.grid_center(dst)[:rank])
    x = _cuda(imgs["float32"])
    for mode in ("linear", "bspline", "nearest"):
        a = t.resample(x, src, dst, interpolation=mode)
        b = t.resample(x, src, dst, interpolation=mode, transform=ident)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def _phantom_batch(rank, n, spacing, seed, count):
    t = _tf()
    fg = _grid((n,) * rank, spacing)
    c = t.grid_center(fg)
    fixed = orr.phantom(fg, "t1", edge_mm=1.5 * spacing)
    trues = _offsets(rank, seed, count)
    moving = np.stack([orr.phantom(fg, "t2", p, c, edge_mm=1.5 * spacing) for p in trues])
    return fg, c, fixed, moving, trues


@gpu
def test_batched_recovery_at_128_cubed_and_determinism():
    t = _tf()
    fg, c, fixed, moving, trues = _phantom_batch(3, 128, 2.0, 21, 8)
    fx = _cuda(np.stack([fixed] * 8))
    mask = t.foreground_mask(fx, threshold=0.05)
    mv = _cuda(moving)
    tf = t.register_rigid(fx, mv, fg, fg, fixed_mask=mask)
    prm = tf.parameters.cpu().numpy()
    pts = _fixed_points(fg, fixed > 0.05)
    st = tf.status.cpu().numpy()
    assert set(st.tolist()) <= {0, 1}, st
    for i in range(8):
        assert orr.displacement(prm[i], trues[i], c, 3, pts) < 0.25 * 2.0, (i, trues[i], prm[i])
    again = t.register_rigid(fx, mv, fg, fg, fixed_mask=mask)
    assert torch.equal(again.parameters, tf.parameters) and torch.equal(again.metric, tf.metric)
    for i in (0, 5):
        one = t.register_rigid(fx[i:i + 1], mv[i:i + 1], fg, fg, fixed_mask=mask[i:i + 1])
        assert torch.equal(one.parameters[0], tf.parameters[i]) and torch.equal(one.metric[0], tf.metric[i])
        assert torch.equal(one.status[0], tf.status[i])


@gpu
def test_register_rigid_graph_replay_matches_eager():
    t = _tf()
    fg, c, fixed, moving, _ = _phantom_batch(2, 96, 2.0, 4, 2)
    fx, mv = _cuda(np.stack([fixed] * 2)), _cuda(moving)
    kw = dict(shrink_factors=(2, 1), smoothing_sigmas=(1.0, 0.0), iterations=30)
    eager = t.register_rigid(fx, mv, fg, fg, **kw)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        t.register_rigid(fx, mv, fg, fg, **kw)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = t.register_rigid(fx, mv, fg, fg, **kw)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(cap.parameters, eager.parameters) and torch.equal(cap.metric, eager.metric)
        assert torch.equal(cap.status, eager.status)


@gpu
def test_rank2_recovery_and_oracle_agreement():
    t = _tf()
    fg, c, fixed, moving, trues = _phantom_batch(2, 128, 2.0, 0, 3)
    fx = _cuda(np.stack([fixed] * 3))
    mask = fx > 0.05
    tf = t.register_rigid(fx, _cuda(moving), fg, fg, fixed_mask=mask)
    prm = tf.parameters.cpu().numpy()
    pts = _fixed_points(fg, fixed > 0.05)
    for i in range(3):
        assert orr.displacement(prm[i], trues[i], c, 2, pts) < 0.25 * 2.0
        ref = orr.register_one(fixed, moving[i], fg, fg, fixed_mask=fixed > 0.05)
        assert int(tf.status[i]) == ref["status"]
        assert orr.displacement(prm[i], ref["parameters"], c, 2, pts) < 0.05 * 2.0
    m = tf.matrix().cpu().numpy()
    for i in range(3):
        np.testing.assert_array_equal(m[i], orr.homogeneous(prm[i], tf.center + (0.0,), 2))


@gpu
def test_flat_and_no_overlap_statuses_on_device():
    t = _tf()
    fg = _grid((32, 32), 2.0)
    far = _grid((32, 32), 2.0, origin=(1000.0, 1000.0))
    f = orr.phantom(fg, "t1")
    fx = _cuda(np.stack([f, f]))
    mv = _cuda(np.stack([np.full_like(f, 0.5), f]))
    tf = t.register_rigid(fx, mv, fg, fg, iterations=3)
    assert int(tf.status[0]) == 3 and math.isnan(float(tf.metric[0])) and int(tf.status[1]) in (0, 1)
    tf = t.register_rigid(fx, _cuda(np.stack([f, f])), fg, far, initialize="identity", iterations=3)
    assert (tf.status.cpu() == 2).all() and torch.isnan(tf.metric).all()
    assert (tf.parameters == 0).all()


@gpu
def test_scoring_chain_registered_beats_unregistered():
    """T1 on the model grid, a misaligned true T2: register it onto the T1 (fixed mask = the T1's cleaned head mask),
    resample it through the transform, and score.  MAE against the T2 the generator should produce and the Dice of head
    masks both improve, and the chain equals the one built from oracles."""
    t = _tf()
    fg = _grid((96, 96, 96), 2.0)
    c = t.grid_center(fg)
    true = _offsets(3, 31, 1)[0]
    t1 = _cuda(orr.phantom(fg, "t1", edge_mm=3.0))
    t2_aligned = _cuda(orr.phantom(fg, "t2", edge_mm=3.0))
    t2 = _cuda(orr.phantom(fg, "t2", true, c, edge_mm=3.0))
    head = t.foreground_mask(t1, largest_component=True, fill_holes=True)
    tf = t.register_rigid(t1, t2, fg, fg, fixed_mask=head)
    reg = t.resample(t2, fg, fg, transform=tf)
    mae_before = t.mean_absolute_error(t2, t2_aligned, mask=head)
    mae_after = t.mean_absolute_error(reg, t2_aligned, mask=head)
    assert mae_after < 0.5 * mae_before
    truth = t.foreground_mask(t2_aligned, threshold=0.2)
    dice_before = float(t.mask_agreement(t.foreground_mask(t2, threshold=0.2), truth)["dice"])
    dice_after = float(t.mask_agreement(t.foreground_mask(reg, threshold=0.2), truth)["dice"])
    assert dice_after > dice_before
    m = orr.compose(tf.parameters.cpu().numpy(), t.resample_map(fg, fg), c, 3)[0]
    want = orr.resample_mapped(t2.cpu().numpy(), fg.size, fg.size, m).reshape(fg.shape)
    np.testing.assert_array_equal(reg.cpu().numpy(), want)
