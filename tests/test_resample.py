"""Linear resampling between physical grids (ITK 5.1 ResampleImageFilter + IdentityTransform +
LinearInterpolateImageFunction, the reference's ResampleT1T2d): ``mpgan.transforms.ImageGeometry`` / ``resample`` over
the kernel in csrc/resample.cu.

ITK is not available here, so nothing is compared with ITK itself.  CPU tests pin the numpy fp64 restatement
(oracle/resample.py) against scipy's ``map_coordinates`` and against known answers whose expected bytes follow from the
geometry alone (identity, axis permutations and flips, a 2x block mean, the half-open edges, a NaN that must not leak),
and check that every argument error is raised before the device is touched and that the C ABI rejects bad input.
``-m gpu`` tests compare the kernel with the oracle bit for bit, and run the native-grid chain (native T1 -> model grid
-> percentile scaling -> generator -> native grid) against the same chain built from the oracles."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage
from scipy.spatial.transform import Rotation

from conftest import rel_l2
from oracle import resample as ors

gpu = pytest.mark.gpu
SENTINEL = 12345.0


def _geometries():
    from mpgan.transforms import ImageGeometry, reference_grid
    return ImageGeometry, reference_grid


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


# ------------------------------------------------------------------------------------------ known answers (shared)
def _case_identity(rank):
    ImageGeometry, _ = _geometries()
    size, spacing, origin = ((13, 9, 6), (0.5, 1.0, 2.0), (-3.25, 7.0, 0.5))
    g = ImageGeometry(size[:rank], spacing[:rank], origin[:rank])   # powers of two: c = i exactly
    x = _rand((2,) + g.shape, 1)
    return x, g, g, 0.0, x, 0


def _case_permutation(perm, flip):
    """Direction = an axis permutation with flips and anisotropic spacing: the result is a transpose / flip of the
    [z, y, x] array.  Target axis j runs along source axis perm[j], reversed where flip[j]."""
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
    x = _rand((1,) + src.shape, 2)
    b = x[0].transpose(2, 1, 0).transpose(perm)                  # ITK order (x, y, z), permuted
    b = np.flip(b, axis=tuple(j for j in range(3) if flip[j]))
    return x, src, tgt, 0.0, np.ascontiguousarray(b.transpose(2, 1, 0))[None], 0


def _case_downsample():
    """2x down with the output origin half an input voxel in: every output voxel is the mean of a 2x2x2 block."""
    ImageGeometry, _ = _geometries()
    src = ImageGeometry((8, 6, 4), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    tgt = ImageGeometry((4, 3, 2), (2.0, 2.0, 2.0), (0.5, 0.5, 0.5))
    x = _rand((2,) + src.shape, 3, 0.5, 2.0)
    mean = x.astype(np.float64).reshape(2, 2, 2, 3, 2, 4, 2).mean(axis=(2, 4, 6))
    return x, src, tgt, 0.0, mean.astype(np.float32), 1


def _case_edges():
    """Output centres exactly on c = -0.5 (takes voxel 0) and c = n - 0.5 (outside: default_value)."""
    ImageGeometry, _ = _geometries()
    src = ImageGeometry((5, 4, 3), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0))
    tgt = ImageGeometry((2, 4, 3), (5.0, 1.0, 1.0), (-0.5, 0.0, 0.0))
    x = _rand((1,) + src.shape, 4)
    want = np.stack([x[..., 0], np.full_like(x[..., 0], -7.0)], axis=-1)
    return x, src, tgt, -7.0, want, 0


def _case_nan():
    """A NaN (and an inf) input voxel appears only at its own position under the identity geometry."""
    x, g, _, _, _, _ = _case_identity(3)
    x = x.copy()
    x[1, 3, 4, 5] = np.nan
    x[0, 2, 0, 12] = np.inf
    return x, g, g, 0.0, x, 0


KNOWN = {"identity3": lambda: _case_identity(3), "identity2": lambda: _case_identity(2),
         "transpose_xz": lambda: _case_permutation((2, 1, 0), (False, False, False)),
         "cycle_flip": lambda: _case_permutation((1, 2, 0), (True, False, True)),
         "flip_y": lambda: _case_permutation((0, 1, 2), (False, True, False)),
         "swap_xy_flip_all": lambda: _case_permutation((1, 0, 2), (True, True, True)),
         "downsample2x": _case_downsample, "edges": _case_edges, "nan": _case_nan}


def _check_known(got, want, ulps):
    assert got.shape == want.shape and got.dtype == np.float32
    if ulps == 0:
        assert np.array_equal(got, want, equal_nan=True)
        assert np.array_equal(np.isnan(got), np.isnan(want))
    else:
        assert (got > 0).all() and (want > 0).all()
        assert np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32)).max() <= ulps


# ------------------------------------------------------------------------------------------------- oracle (CPU)
@pytest.mark.parametrize("name", sorted(KNOWN))
def test_oracle_known_answers(name):
    x, src, tgt, dflt, want, ulps = KNOWN[name]()
    _check_known(ors.resample(x, src, tgt, dflt), want, ulps)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
@pytest.mark.parametrize("rank", [2, 3])
def test_oracle_matches_scipy_map_coordinates(seed, rank):
    size_s = (13, 11, 9)[:rank]
    src = _oblique(size_s, (1.3, 0.9, 2.1)[:rank], seed)
    tgt = _oblique((17, 15, 12)[:rank], (1.1, 1.2, 1.6)[:rank], seed + 10)
    x = _rand((2,) + src.shape, seed)
    c = ors.continuous_index(src, tgt)
    size3 = tuple(size_s) + (1,) * (3 - rank)
    ins = ors.inside(c, size3)
    assert 0.1 < ins.mean() < 0.9                                  # both sides of the boundary are exercised
    got = ors.interpolate(x.reshape((2,) + size3[::-1]), c, size3)[:, ins]
    coords = np.stack([c[k][ins] for k in reversed(range(rank))])   # array order (z, y, x)
    for i in range(2):
        ref = ndimage.map_coordinates(x[i].astype(np.float64), coords, order=1, mode="nearest")
        np.testing.assert_allclose(got[i], ref, rtol=1e-12, atol=1e-12)
    out, mask = ors.resample(x, src, tgt, SENTINEL), ins.reshape(tgt.shape)
    assert (out[:, ~mask] == SENTINEL).all() and (out[:, mask] != SENTINEL).all()


def test_oracle_inside_is_half_open():
    n = 5
    vals = np.array([-0.5, np.nextafter(-0.5, -1), n - 0.5, np.nextafter(n - 0.5, 0), 0.0, np.nan, 2.3])
    c = np.stack([vals, np.zeros_like(vals), np.zeros_like(vals)])
    assert ors.inside(c, (n, 1, 1)).tolist() == [True, False, False, True, True, False, True]


def test_reference_grid():
    _, reference_grid = _geometries()
    g = reference_grid()
    assert g.size == (128,) * 3 and g.spacing == (2.0,) * 3 and g.origin == (-128.0,) * 3 and g.shape == (128,) * 3
    assert np.array_equal(g.direction, np.eye(3)) and np.array_equal(g.physical_to_index(), np.eye(3) / 2)
    g32 = reference_grid(32)
    assert g32.spacing == (8.0,) * 3 and g32.origin == (-128.0,) * 3
    g2 = reference_grid(256, 256.0, rank=2)
    assert g2.size == (256, 256) and g2.spacing == (1.0, 1.0) and g2.origin == (-128.0, -128.0)


def test_image_geometry():
    ImageGeometry, _ = _geometries()
    g = ImageGeometry((4, 5, 6), (1.0, 2.0, 3.0), (0.0, 1.0, 2.0), np.eye(3)[[1, 0, 2]])
    assert g.rank == 3 and g.shape == (6, 5, 4)
    assert np.array_equal(g.index_to_physical(), [[0, 2, 0], [1, 0, 0], [0, 0, 3]])
    assert np.allclose(g.physical_to_index() @ g.index_to_physical(), np.eye(3), atol=1e-15)
    o = _oblique((9, 8, 7), (1.3, 0.7, 2.2), 5)
    assert np.allclose(o.physical_to_index() @ o.index_to_physical(), np.eye(3), atol=1e-14)
    bad = [dict(size=(4,)), dict(size=(4, 4, 4, 4), spacing=(1,) * 4, origin=(0,) * 4), dict(size=(4, 0, 4)),
           dict(size=(4, 2.5, 4)), dict(size=(4, True, 4)), dict(spacing=(1.0, 1.0)), dict(origin=(0.0,) * 4),
           dict(spacing=(1.0, 0.0, 1.0)), dict(spacing=(1.0, -2.0, 1.0)), dict(spacing=(1.0, math.inf, 1.0)),
           dict(origin=(0.0, math.nan, 0.0)), dict(direction=np.eye(2)), dict(direction=[[1, 0, 0], [0, 1, 0]]),
           dict(direction=[[1, 0, 0], [0, 1, 0], [1, 1, 0]]), dict(direction=[[1, 0, 0], [0, math.nan, 0], [0, 0, 1]]),
           dict(direction=np.zeros((3, 3)))]
    for kw in bad:
        args = dict(size=(4, 5, 6), spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0))
        args.update(kw)
        with pytest.raises(ValueError):
            ImageGeometry(**args)


# ------------------------------------------------------------------------------------------- argument checks (CPU)
def test_resample_arguments_are_validated_before_the_device():
    from mpgan.transforms import resample
    ImageGeometry, reference_grid = _geometries()
    src, tgt = ImageGeometry((6, 5, 4), (1, 1, 1), (0, 0, 0)), reference_grid(8)
    x = torch.zeros(2, 4, 5, 6)
    bad = [(x, "src", tgt, {}), (x, src, reference_grid(8, rank=2), {}), (x.numpy(), src, tgt, {}),
           (x.double(), src, tgt, {}), (torch.zeros(2, 4, 6, 5), src, tgt, {}), (torch.zeros(5, 6), src, tgt, {}),
           (x, src, tgt, dict(default_value="0")), (x, src, tgt, dict(default_value=None)),
           (x, src, ImageGeometry(((1 << 22) + 1, 1, 1), (1, 1, 1), (0, 0, 0)), {})]
    for img, s, t, kw in bad:
        with pytest.raises(ValueError):
            resample(img, s, t, **kw)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        resample(x, src, tgt, default_value=-1)


def test_c_abi_rejects_bad_input():
    import ctypes
    from mpgan import _lib
    from mpgan.transforms import resample_map
    lib = _lib.load()
    ImageGeometry, reference_grid = _geometries()
    p = 256   # device pointers are never dereferenced: the checks come first
    good3 = resample_map(_oblique((9, 8, 7), (1, 1, 1), 0), reference_grid(16))
    good2 = resample_map(ImageGeometry((9, 8), (1, 1), (0, 0), _rotation(1, 2)), reference_grid(16, rank=2))

    def call(m=good3, rank=3, ins=(9, 8, 7), outs=(16, 16, 16), items=1, x=p, y=p, sizes=True, mp=True):
        i3 = (ctypes.c_int32 * 3)(*ins) if sizes else None
        o3 = (ctypes.c_int32 * 3)(*outs)
        mm = (ctypes.c_double * 24)(*m) if mp else None
        return lib.mpgan_resample_linear(x, items, rank, i3, o3, mm, 0.0, y, None)

    def edit(m, i, v):
        m = list(m)
        m[i] = v
        return m

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
    for i, v in ((3 + 2, 0.5), (3 + 7, 0.1), (3 + 8, 2.0), (15 + 6, 1.0), (15 + 5, -0.5)):   # M_out / N_in z row, column
        assert call(**dict(kw2, m=edit(good2, i, v))) == -1 and "identity" in _lib.last_error()
    for i in (2, 14):
        assert call(**dict(kw2, m=edit(good2, i, 1.0))) == -1 and "z origins" in _lib.last_error()
    assert call(items=1 << 40) == -1 and "rows" in _lib.last_error()


# ------------------------------------------------------------------------------------------------- CUDA kernel
def _dev(x, src, tgt, dflt=0.0):
    from mpgan.transforms import resample
    return resample(torch.from_numpy(np.ascontiguousarray(x)).cuda(), src, tgt, default_value=dflt).cpu().numpy()


def _both_ways_bit_exact(x, native, model):
    fwd = _dev(x, native, model, SENTINEL)
    assert np.array_equal(fwd, ors.resample(x, native, model, SENTINEL))
    inside = fwd != SENTINEL
    assert 0.01 < inside.mean() < 0.99                             # the inside masks agree on both sides
    back = _dev(fwd, model, native, SENTINEL)
    assert np.array_equal(back, ors.resample(fwd, model, native, SENTINEL))
    assert 0.01 < (back != SENTINEL).mean()
    return fwd, back


@gpu
@pytest.mark.parametrize("size,spacing,seed", [((61, 67, 13), (1.7, 2.3, 4.1), 11), ((45, 70, 37), (3.1, 1.9, 2.6), 12),
                                               ((61, 67, 13), (4.3, 3.7, 9.5), 13)])
def test_oblique_round_trip_matches_oracle_bit_exact(size, spacing, seed):
    _, reference_grid = _geometries()
    native = _oblique(size, spacing, seed)
    x = _rand((2,) + native.shape, seed)
    _both_ways_bit_exact(x, native, reference_grid(128))


@gpu
def test_native_1mm_volume_round_trip_matches_oracle_bit_exact():
    _, reference_grid = _geometries()
    native = _oblique((256, 256, 176), (1.0, 1.0, 1.0), 21)
    x = _rand(native.shape, 21, 0.0, 1000.0)
    _both_ways_bit_exact(x, native, reference_grid())


@gpu
def test_rank2_slices_match_oracle_bit_exact():
    _, reference_grid = _geometries()
    native = _oblique((512, 512), (0.5, 0.5), 22)
    x = _rand((3, 1) + native.shape, 22)
    fwd, back = _both_ways_bit_exact(x, native, reference_grid(256, 256.0, rank=2))
    assert fwd.shape == (3, 1, 256, 256) and back.shape == (3, 1, 512, 512)


@gpu
@pytest.mark.parametrize("name", sorted(KNOWN))
def test_known_answers_on_device(name):
    x, src, tgt, dflt, want, ulps = KNOWN[name]()
    _check_known(_dev(x, src, tgt, dflt), want, ulps)


@gpu
def test_batched_call_equals_separate_calls():
    from mpgan.transforms import resample
    _, reference_grid = _geometries()
    native = _oblique((45, 70, 37), (3.1, 1.9, 2.6), 31)
    x = torch.from_numpy(_rand((3,) + native.shape, 31)).cuda()
    tgt = reference_grid(64)
    both = resample(x, native, tgt, default_value=-1.0)
    for i in range(3):
        assert torch.equal(both[i], resample(x[i], native, tgt, default_value=-1.0))


@gpu
def test_repetition_and_graph_replay_change_no_bit():
    from mpgan.transforms import resample
    _, reference_grid = _geometries()
    native = _oblique((61, 67, 13), (1.7, 2.3, 4.1), 32)
    model = reference_grid(128)
    x = torch.from_numpy(_rand((2,) + native.shape, 32)).cuda()
    base = resample(x, native, model, default_value=SENTINEL)
    for _ in range(3):
        assert torch.equal(resample(x, native, model, default_value=SENTINEL), base)
    static = x.clone()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = resample(static, native, model, default_value=SENTINEL)
    for _ in range(2):
        out.fill_(0.0)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, base)
    static.copy_(torch.flip(x, [0]))
    g.replay()
    assert torch.equal(out, torch.flip(base, [0]))


@gpu
def test_native_grid_chain_end_to_end_against_oracle():
    """native T1 -> reference_grid(32) -> percentiles 1/99 to [-1, 1] -> 32^3 generator -> back to the native grid."""
    from mpgan import CasNetGenerator, inference
    from mpgan.transforms import ScaleIntensityRangePercentiles, resample
    from oracle import transforms as otf
    from oracle.nets import CasNetGenerator as OGen
    _, reference_grid = _geometries()
    native = _oblique((45, 70, 37), (3.1, 4.4, 3.3), 41)   # 308 mm along y: sticks out of the model grid
    model_grid = reference_grid(32)
    t1 = _rand(native.shape, 41, 0.0, 800.0)

    torch.manual_seed(0)
    ora = OGen((1, 32, 32, 32), 6, 3).eval()
    gen = CasNetGenerator((1, 32, 32, 32), precision="fp32")
    gen.load_state_dict(ora.state_dict())
    gen.cuda()

    x = ors.resample(t1, native, model_grid)
    x = otf.scale_intensity_range_percentiles(x, 1, 99, -1.0, 1.0, clip=True)
    with torch.no_grad():
        y = ora(torch.from_numpy(x)[None, None]).numpy()[0, 0]
    ref = torch.from_numpy(ors.resample(y, model_grid, native, -1.0))

    def chain():
        v = resample(torch.from_numpy(t1).cuda(), native, model_grid)
        v = ScaleIntensityRangePercentiles(1, 99, -1.0, 1.0, clip=True)(v)
        out = inference.infer_volume(gen, v[None, None])
        return resample(out[0, 0], model_grid, native, default_value=-1.0)

    got = chain()
    assert got.shape == native.shape and rel_l2(got, ref) <= 1e-4
    assert (got == -1.0).any() and (got != -1.0).float().mean() > 0.5
    gen.set_precision("bf16")
    assert rel_l2(chain(), ref) <= 1e-2
