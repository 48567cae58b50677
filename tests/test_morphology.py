"""Connected-component labelling, largest component, hole filling and binary erosion / dilation of masks.

CPU tests pin the oracle (oracle/morphology.py, a thin layer over scipy.ndimage) with known answers: raster-order
numbering, the tie rule of the largest component, hole filling as "background components touching no face", depth-1
images at rank 3, empty and full images.  They also check the argument errors and the C ABI's error returns.  ``-m gpu``
tests compare the kernels with scipy.ndimage bit for bit, for every connectivity at ranks 2 and 3."""
import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import masked_metrics as omm
from oracle import morphology as omo

gpu = pytest.mark.gpu
RANK_CONN = [(2, 1), (2, 2), (3, 1), (3, 2), (3, 3)]


def _random(shape, p, seed):
    return np.random.RandomState(seed).rand(*shape) < p


def _head(shape, seed):
    """The bright noisy ellipsoid in a dark noisy field of tests/test_masked_metrics.py, with two darker spheres inside
    (sinus-like holes for Otsu)."""
    rng = np.random.RandomState(seed)
    grids = np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij")
    inside = sum((g / 0.7) ** 2 for g in grids) < 1
    v = np.where(inside, rng.gamma(4.0, 100.0, size=shape), rng.gamma(1.0, 10.0, size=shape))
    for c in (0.25, -0.3):
        v[sum((g - c) ** 2 for g in grids) < 0.15 ** 2] = rng.gamma(1.0, 10.0)
    return v.astype(np.float32)


def _serpentine(d, h, w):
    """One path through the whole volume: each slice a serpentine of rows, slices joined at alternating corners, so the
    component's smallest index is far (along the path) from most of its voxels."""
    m = np.zeros((d, h, w), bool)
    for z in range(d):
        m[z, ::2, :] = True
        for y in range(1, h - 1, 2):
            m[z, y, (w - 1) if (y // 2) % 2 == 0 else 0] = True
    for z in range(0, d - 1):                       # a path in z between a corner voxel of slice z and z + 1
        m[z, -1 if z % 2 == 0 else 0, -1] = True
    m[1::2] = m[1::2, ::-1]                          # every other slice runs the other way
    return m


def _shells(n, radii=(4, 8, 12, 16)):
    g = np.meshgrid(*[np.arange(n) - n / 2 + 0.5] * 3, indexing="ij")
    r = np.sqrt(sum(a * a for a in g))
    return np.logical_or.reduce([np.abs(r - q) < 0.9 for q in radii])


def _checkerboard(shape):
    return np.indices(shape).sum(axis=0) % 2 == 0


# ------------------------------------------------------------------------------------------------- oracle (CPU)
def test_label_numbers_in_raster_order_of_first_voxel():
    m = np.array([[0, 0, 1, 1], [1, 0, 0, 1], [1, 0, 1, 0], [0, 0, 1, 1]], bool)
    lab, k = omo.label(m)
    assert k == 3 and lab.tolist() == [[0, 0, 1, 1], [2, 0, 0, 1], [2, 0, 3, 0], [0, 0, 3, 3]]
    lab8, k8 = omo.label(m, connectivity=2)
    assert k8 == 2 and lab8[2, 2] == 1
    for nd, conn in RANK_CONN:
        shape = (30, 31) if nd == 2 else (12, 13, 14)
        lab, k = omo.label(_random(shape, 0.2, nd + conn), conn)
        firsts = [np.flatnonzero(lab.ravel() == j)[0] for j in range(1, k + 1)]
        assert k > 1 and firsts == sorted(firsts)


def test_largest_component_ties_go_to_the_lowest_label():
    m = np.zeros((3, 9, 9), bool)
    m[0, 5:7, 1:3] = True            # 4 voxels, label 2
    m[0, 1:3, 5:7] = True            # 4 voxels, label 1: wins the tie
    m[1, 0, 0] = True                # image 1: one voxel
    big = omo.largest_component(m, spatial_dims=2)
    assert big[0].sum() == 4 and big[0, 1:3, 5:7].all() and big[1, 0, 0] and big[1].sum() == 1 and not big[2].any()
    m[0, 7, 1] = True                # now the lower component is larger
    assert omo.largest_component(m, spatial_dims=2)[0, 5:8, 1:3].sum() == 5


def test_fill_holes_is_background_components_touching_no_face():
    for nd, conn in RANK_CONN:
        shape = (40, 41) if nd == 2 else (15, 16, 17)
        for p in (0.3, 0.5, 0.7):
            m = _random(shape, p, int(p * 10) + conn)
            assert np.array_equal(omo.fill_holes(m, conn), omo.fill_holes_by_components(m, conn)), (nd, conn, p)
    shells = _shells(32)
    assert np.array_equal(omo.fill_holes(shells), omo.fill_holes_by_components(shells))
    assert omo.fill_holes(shells).sum() > 1.5 * shells.sum()


def test_depth_one_images_at_rank_3_fill_nothing():
    ring = np.zeros((1, 9, 9), bool)
    ring[0, 2:7, 2:7] = True
    ring[0, 3:6, 3:6] = False
    assert np.array_equal(omo.fill_holes(ring), ring)
    assert omo.fill_holes(ring, spatial_dims=2)[0, 3:6, 3:6].all()
    assert not omo.binary_erosion(ring).any()            # the structure reaches outside in z: border_value 0
    assert omo.binary_erosion(ring, spatial_dims=2).sum() == 0 and omo.binary_erosion(ring[0] | True).sum() == 49


def test_empty_and_full_images():
    for shape in ((6, 7), (4, 6, 7)):
        empty, full = np.zeros(shape, bool), np.ones(shape, bool)
        assert omo.label(empty)[1] == 0 and not omo.largest_component(empty).any() and not omo.fill_holes(empty).any()
        lab, k = omo.label(full)
        assert k == 1 and (lab == 1).all() and omo.largest_component(full).all() and omo.fill_holes(full).all()
        inner = omo.binary_erosion(full)
        assert inner.sum() == np.prod([s - 2 for s in shape]) and omo.binary_dilation(empty, 3).sum() == 0


def test_iterated_morphology_is_repeated_single_steps():
    for nd, conn in RANK_CONN:
        m = _random((20, 21) if nd == 2 else (10, 11, 12), 0.6, conn)
        for op in (omo.binary_erosion, omo.binary_dilation):
            step = m
            for it in (1, 2, 3):
                step = op(step, 1, conn)
                assert np.array_equal(op(m, it, conn), step), (op, nd, conn, it)


def test_arguments_are_validated_before_the_device():
    from mpgan import transforms as T
    m = torch.ones(2, 8, 9, 10, dtype=torch.bool)
    fns = [T.label, T.largest_component, T.fill_holes, T.binary_erosion, T.binary_dilation]
    for fn in fns:
        for bad in (m.float(), m.to(torch.int32), m.numpy(), torch.zeros(3, 0, 4, dtype=torch.bool), m[0, 0, 0]):
            with pytest.raises(ValueError):
                fn(bad)
        for kw in (dict(connectivity=0), dict(connectivity=4), dict(connectivity=True), dict(connectivity=1.0),
                   dict(spatial_dims=1), dict(spatial_dims=4), dict(spatial_dims=True),
                   dict(spatial_dims=2, connectivity=3)):
            with pytest.raises(ValueError):
                fn(m, **kw)
        for ok in (m, m.to(torch.uint8)):
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                fn(ok, connectivity=3)
    for fn in (T.binary_erosion, T.binary_dilation):
        for it in (0, -1, 1.0, True, None):
            with pytest.raises(ValueError):
                fn(m, iterations=it)
    x = torch.zeros(2, 16, 16, 16)
    for kw in (dict(largest_component=1), dict(fill_holes="yes"), dict(connectivity=0), dict(connectivity=4)):
        with pytest.raises(ValueError):
            T.foreground_mask(x, **kw)
    with pytest.raises(ValueError):
        T.foreground_mask(torch.zeros(16, 16), fill_holes=True, connectivity=3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.foreground_mask(x, largest_component=True, fill_holes=True, connectivity=3)


def test_c_abi_rejects_bad_arguments():
    from mpgan import _lib
    lib = _lib.load()
    need = lib.mpgan_morphology_workspace(2, 4, 5, 6)
    assert need >= 8 * 2 * 120 and lib.mpgan_morphology_workspace(0, 4, 5, 6) == 0
    assert lib.mpgan_morphology_workspace(1, 2 ** 11, 2 ** 10, 2 ** 10) == 0
    m, o, c, ws = 1 << 20, 1 << 30, 1 << 31, 1 << 32      # never dereferenced: the checks come first

    def label(mask=m, rank=3, items=2, d=4, h=5, w=6, conn=1, out=o, count=c, wsp=ws, nbytes=need):
        return lib.mpgan_label(mask, rank, items, d, h, w, conn, out, count, wsp, nbytes, None)

    def other(name, mask=m, rank=3, items=2, d=4, h=5, w=6, conn=1, out=o, wsp=ws, nbytes=need, extra=()):
        return getattr(lib, name)(mask, rank, items, d, h, w, conn, *extra, out, wsp, nbytes, None)

    for kw in (dict(mask=None), dict(out=None), dict(count=None), dict(wsp=None)):
        assert label(**kw) == -1 and "null" in _lib.last_error()
    names = [("mpgan_largest_component", ()), ("mpgan_fill_holes", ()), ("mpgan_binary_morphology", (0, 2))]
    cases = [(dict(rank=1), "rank"), (dict(rank=4), "rank"), (dict(conn=0), "connectivity"),
             (dict(conn=4), "connectivity"), (dict(rank=2, conn=3, d=1), "connectivity"), (dict(rank=2), "d 4"),
             (dict(items=0), "size"), (dict(w=0), "size"), (dict(d=2 ** 11, h=2 ** 10, w=2 ** 10), "voxels"),
             (dict(nbytes=need - 1), "workspace"), (dict(out=m + 100), "overlap"), (dict(wsp=o - 8), "overlap")]
    for kw, text in cases:
        assert label(**kw) == -1 and text in _lib.last_error(), (kw, _lib.last_error())
        for name, extra in names:
            assert other(name, extra=extra, **kw) == -1 and text in _lib.last_error(), (name, kw, _lib.last_error())
    assert label(count=o + 4) == -1 and "count" in _lib.last_error()
    for extra, text in (((2, 1), "op"), ((-1, 1), "op"), ((0, 0), "iterations"), ((1, -3), "iterations")):
        assert other("mpgan_binary_morphology", extra=extra) == -1 and text in _lib.last_error()


# ------------------------------------------------------------------------------------------------- CUDA kernels
def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _diff(got, ref):
    got = got.cpu().numpy()
    return f"{int((got != ref).sum())} of {ref.size} voxels differ"


def _check(mask, conn, spatial_dims=None, iterations=(1,)):
    """Every kernel against scipy.ndimage for one mask: labels and counts, largest component, filled holes, erosion and
    dilation."""
    from mpgan import transforms as T
    (tm,) = _cuda(mask)
    lab, cnt = T.label(tm, connectivity=conn, spatial_dims=spatial_dims)
    rl, rc = omo.label(mask, conn, spatial_dims)
    assert lab.dtype == torch.int32 and cnt.dtype == torch.int32 and tuple(cnt.shape) == rc.shape
    assert np.array_equal(cnt.cpu().numpy(), rc), (cnt, rc)
    assert np.array_equal(lab.cpu().numpy(), rl), _diff(lab, rl)
    for fn, ref in ((T.largest_component, omo.largest_component), (T.fill_holes, omo.fill_holes)):
        got = fn(tm, connectivity=conn, spatial_dims=spatial_dims)
        r = ref(mask, conn, spatial_dims)
        assert got.dtype == torch.bool and np.array_equal(got.cpu().numpy(), r), (fn.__name__, _diff(got, r))
    for it in iterations:
        for fn, ref in ((T.binary_erosion, omo.binary_erosion), (T.binary_dilation, omo.binary_dilation)):
            got = fn(tm, iterations=it, connectivity=conn, spatial_dims=spatial_dims)
            r = ref(mask, it, conn, spatial_dims)
            assert got.dtype == torch.bool and np.array_equal(got.cpu().numpy(), r), (fn.__name__, it, _diff(got, r))
    return rc


@gpu
@pytest.mark.parametrize("rank,conn", RANK_CONN)
def test_kernels_match_scipy(rank, conn):
    sd = rank
    # odd extents (no tile multiple; the scalar stencil path) and a 16-multiple width (16-byte stencil rows)
    for shape in ((37, 41, 43), (6, 40, 48, 64)):
        for p in (0.2, 0.5, 0.8):
            _check(_random(shape, p, int(10 * p) + conn), conn, sd, iterations=(1, 2, 3))
    for shape in ((1, 1, 1000), (1000, 1, 1), (1, 1, 1), (3, 1, 2049)):   # lines, a single voxel, a chunk boundary
        _check(_random(shape, 0.7, 1), conn, sd)
    _check(_checkerboard((33, 34, 35)), conn, sd, iterations=(1, 2))
    if rank == 2:
        for p in (0.5927, 0.407):                                          # site / 8-neighbour percolation thresholds
            _check(_random((3, 700, 900), p, 2), conn, 2)
        k = _check(_serpentine(1, 301, 257)[0], conn, 2)
        assert k == 1
    else:
        for p in (0.3116, 0.2, 0.1):                                       # near 6-, 18-, 26-neighbour thresholds
            _check(_random((96, 128, 160), p, 3), conn, 3)
        k = _check(_serpentine(40, 61, 67), conn, 3)
        assert k == 1
        _check(_shells(48), conn, 3, iterations=(1, 3))
    batch = _random((5, 24, 25, 26) if rank == 3 else (5, 40, 41), 0.4, 4)
    batch[2] = False                                                       # an empty image between non-empty ones
    batch[4] = True                                                        # and a full one
    counts = _check(batch, conn, sd, iterations=(1, 2))
    assert counts[2] == 0 and counts[4] == 1


@gpu
@pytest.mark.parametrize("conn", [1, 2, 3])
def test_otsu_head_mask_128(conn):
    from mpgan import transforms as T
    x = _head((128, 128, 128), 5)
    m = omm.foreground_mask(x)
    assert 0.05 < m.mean() < 0.5
    _check(m, conn, iterations=(1, 2))
    (tx,) = _cuda(x)
    for largest, fill in ((False, False), (True, False), (False, True), (True, True)):
        got = T.foreground_mask(tx, largest_component=largest, fill_holes=fill, connectivity=conn)
        ref = omo.foreground_mask(x, largest, fill, conn)
        assert got.dtype == torch.bool and np.array_equal(got.cpu().numpy(), ref), (largest, fill, _diff(got, ref))
    clean = omo.foreground_mask(x, True, True, conn)
    assert ndimage.label(clean, omo.structure(3, conn))[1] == 1 and clean.sum() > m.sum()


@gpu
def test_slice_stack_and_batched_foreground_masks():
    from mpgan import transforms as T
    x = _head((9, 1, 97, 101), 6)
    m = omm.foreground_mask(x[:, 0], spatial_dims=2)[:, None]
    for conn in (1, 2):
        _check(m, conn, spatial_dims=2, iterations=(1, 2))
    (tm,) = _cuda(m)
    assert not T.fill_holes(tm).cpu().numpy()[m == 0].any()              # rank 3 with depth 1: all face
    xs = np.stack([_head((40, 41, 43), s) for s in range(3)])
    xs[1] = 0.0                                                            # a constant image: an empty mask
    (tx,) = _cuda(xs)
    got = T.foreground_mask(tx, largest_component=True, fill_holes=True).cpu().numpy()
    for i in range(3):
        assert np.array_equal(got[i], omo.foreground_mask(xs[i], True, True)), i
    assert not got[1].any()


@gpu
def test_large_volumes_and_determinism():
    from mpgan import transforms as T
    x = _head((256, 512, 512), 7)
    m = omm.foreground_mask(x)
    _check(m, 1)
    (tx,) = _cuda(x)
    got = T.foreground_mask(tx, largest_component=True, fill_holes=True)
    assert np.array_equal(got.cpu().numpy(), omo.foreground_mask(x, True, True))
    del tx, got
    r = _random((256, 512, 512), 0.3116, 8)
    (tr,) = _cuda(r)
    lab, cnt = T.label(tr)
    ref, k = ndimage.label(r)
    assert int(cnt) == k and k > 3_000_000 and np.array_equal(lab.cpu().numpy(), ref)
    lab2, cnt2 = T.label(tr)
    assert torch.equal(lab, lab2) and torch.equal(cnt, cnt2)
    big = T.largest_component(tr).cpu().numpy()
    assert np.array_equal(big, omo._largest(ref))


@gpu
def test_graph_capture_and_replay_on_a_new_input():
    from mpgan import transforms as T
    x = _head((2, 64, 72, 80), 9)
    (tx,) = _cuda(x)
    static = tx.clone()

    def pipeline(v):
        m = T.foreground_mask(v, largest_component=True, fill_holes=True, connectivity=2)
        return m, T.label(m)[0], T.binary_dilation(T.binary_erosion(m, iterations=2), iterations=2)

    base = pipeline(tx)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = pipeline(static)
    for o in outs:
        o.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(outs, base))
    y = _head((2, 64, 72, 80), 10)
    static.copy_(torch.from_numpy(y).cuda())
    g.replay()
    torch.cuda.synchronize()
    m = omo.foreground_mask(y, True, True, 2)
    assert np.array_equal(outs[0].cpu().numpy(), m)
    assert np.array_equal(outs[1].cpu().numpy(), omo.label(m, 1)[0])
    opened = omo.binary_dilation(omo.binary_erosion(m, 2), 2)
    assert np.array_equal(outs[2].cpu().numpy(), opened)
