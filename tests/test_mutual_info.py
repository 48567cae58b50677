"""Mutual information of generated-vs-true volumes (the third score the reference reports, code/eval/*.xml), defined as
the numpy/scipy computation behind scikit-image's ``normalized_mutual_information(x, y, bins)``.

CPU tests pin the oracle (oracle/mutual_info.py): its fp32 edge restatement against ``np.histogramdd``'s edges, and the
entropies against known answers; they also check that every argument error is raised before the device is touched and
that the C ABI rejects bad sizes.  ``-m gpu`` tests compare ``mpgan_mutual_info`` with the oracle: counts and edges bit
for bit, entropies to 1e-12."""
import numpy as np
import pytest
import torch

from oracle import mutual_info as om
from oracle import transforms as ot

gpu = pytest.mark.gpu


def _volume(shape, seed, background=0.4):
    """Synthetic MRI-like volume: positive intensities with a large exactly-zero background."""
    rng = np.random.RandomState(seed)
    v = rng.gamma(2.0, 150.0, size=shape).astype(np.float32)
    v[rng.rand(*shape) < background] = 0.0
    return v


def _display_pair(shape, seed):
    """(generated, truth) on the display range 0..255 (integers): a noisy copy of the truth, and the truth."""
    v = _volume(shape, seed)
    noise = np.random.RandomState(seed + 100).normal(1.0, 0.2, size=shape).astype(np.float32)
    return ot.to_display_range(v * noise), ot.to_display_range(v)


def _unit_pair(shape, seed):
    """(generated, truth) in [-1, 1], the generator's output range."""
    rng = np.random.RandomState(seed)
    truth = (rng.rand(*shape) * 2 - 1).astype(np.float32)
    return np.clip(truth + rng.normal(0, 0.3, shape), -1, 1).astype(np.float32), truth


# ------------------------------------------------------------------------------------------------- oracle (CPU)
def _edges_agree(x, bins):
    lo, hi = om.outer_range(x)
    e = om.histogram_edges(lo, hi, bins)
    ref = np.histogramdd([x.ravel(), x.ravel()], bins=bins)[1][0]
    assert ref.dtype == np.float32 and np.array_equal(e.view(np.uint32), ref.view(np.uint32)), (lo, hi, bins)
    # the kernel walks the table as a sorted one; it is non-decreasing unless the step is subnormal (a whole image
    # range below ~1e-36), where numpy's own searchsorted bins then depend on the order of the values
    if np.float32(np.float32(hi - lo) / np.float32(bins)) >= np.finfo(np.float32).tiny:
        assert np.all(np.diff(e) >= 0), (lo, hi, bins)


def test_oracle_edges_match_numpy():
    rng = np.random.RandomState(0)
    for t in range(3000):
        bins = 2 + t % 127
        scale = 10.0 ** rng.uniform(-3, 3)
        x = (rng.randn(6) * scale + rng.randn() * scale * rng.choice([0, 1, 100])).astype(np.float32)
        _edges_agree(x, bins)
    for bins in range(2, 129):
        for c in (0.0, -0.0, 1.0, -3.7, 255.0, 2.0 ** 23 + 1, 2.0 ** 25, 1e30):          # constant images
            _edges_agree(np.full(5, c, np.float32), bins)
        for scale in (1e-44, 1e-40, 1e-38, 1e6, 1e7):                                    # subnormal and 1e6 scale
            x = (rng.randn(6) * scale).astype(np.float32)
            _edges_agree(x, bins)
            _edges_agree((x + np.float32(3e6)).astype(np.float32), bins)


def test_oracle_known_answers():
    x = _display_pair((12, 13, 14), 0)[0]
    h1, h2, h12, mi, nmi = om.entropies(om.joint_histogram(x, x.copy(), 100)[0])
    assert nmi == pytest.approx(2.0, rel=1e-14) and mi == pytest.approx(h1, rel=1e-14) and h1 == h2
    rng = np.random.RandomState(1)
    y = rng.rand(20, 30).astype(np.float32)
    for c in (0.0, 7.5):
        _, h2, h12, mi, _ = om.entropies(om.joint_histogram(np.full_like(y, c), y, 64)[0])
        assert abs(mi) <= 1e-14 and h12 == pytest.approx(h2, rel=1e-14)
    assert np.isnan(om.normalized_mutual_information(np.full((4, 5), 2.0), np.full((4, 5), -1.0)))
    # one value per bin (the bin centres), against a copy whose values are a permutation of those bin values
    bins = 50
    centres = (np.arange(bins, dtype=np.float32) + np.float32(0.5)) * np.float32(2.0)
    a = centres[rng.randint(0, bins, 5000)]
    a[:bins] = centres
    perm = rng.permutation(bins)
    b = centres[perm[np.searchsorted(centres, a)]]
    counts = om.joint_histogram(a, b, bins)[0]
    assert np.count_nonzero(counts) == bins and np.all(np.count_nonzero(counts, axis=0) == 1)
    assert om.normalized_mutual_information(a, b, bins) == pytest.approx(2.0, rel=1e-14)
    # independent uniform noise: MI is the plug-in estimator's bias (B - 1)^2 / 2N within a few of its standard
    # deviations sqrt(2 (B - 1)^2) / 2N (2N MI is chi-square with (B - 1)^2 degrees of freedom)
    n, bins = 1 << 20, 16
    mi = om.mutual_information(rng.rand(n).astype(np.float32), rng.rand(n).astype(np.float32), bins)
    dof = (bins - 1) ** 2
    assert abs(mi - dof / (2 * n)) <= 6 * np.sqrt(2 * dof) / (2 * n)


def test_arguments_are_validated_before_the_device():
    from mpgan import inference
    from mpgan import transforms as T
    x, y = torch.zeros(4, 20, 20, 20), torch.zeros(4, 20, 20, 20)
    fns = (T.joint_histogram, T.mutual_information, T.normalized_mutual_information)
    bad = [dict(bins=1), dict(bins=129), dict(bins=0), dict(bins=-5), dict(bins=100.0), dict(bins=True),
           dict(bins="100"), dict(bins=None), dict(spatial_dims=1), dict(spatial_dims=4), dict(spatial_dims=2.5),
           dict(spatial_dims=True)]
    for fn in fns:
        for kw in bad:
            with pytest.raises(ValueError):
                fn(x, y, **kw)
        with pytest.raises(ValueError):                    # shape mismatch
            fn(x, y[:, :, :, :19])
        with pytest.raises(ValueError):                    # not float32
            fn(x.double(), y.double())
        with pytest.raises(ValueError):
            fn(x, y.half())
        with pytest.raises(ValueError):
            fn(x.numpy(), y)
        with pytest.raises(ValueError):                    # rank below spatial_dims
            fn(torch.zeros(20, 20), torch.zeros(20, 20), spatial_dims=3)
        with pytest.raises(ValueError):                    # empty image
            fn(torch.zeros(3, 0, 20), torch.zeros(3, 0, 20))
    for bins in (1, 129, 2.5, True):
        with pytest.raises(ValueError):
            inference.evaluate(x, y, mi_bins=bins)
    # valid arguments on CPU tensors: the library's no-fallback error
    for fn in fns:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(x, y, bins=128)


def test_c_abi_rejects_bad_sizes():
    from mpgan import _lib
    lib = _lib.load()
    p = 256   # never dereferenced: the checks come first
    need = lib.mpgan_mutual_info_workspace(3)
    assert need >= 3 * 16 and lib.mpgan_mutual_info_workspace(0) == 0

    def call(items=3, n=1000, bins=100, ws=need, a=p, counts=p, out5=p, workspace=p):
        return lib.mpgan_mutual_info(a, p, items, n, bins, counts, None, out5, workspace, ws, None)

    assert call(bins=1) == -1 and "bins" in _lib.last_error()
    assert call(bins=129) == -1 and "bins" in _lib.last_error()
    assert call(items=0) == -1 and "items" in _lib.last_error()
    assert call(items=-2) == -1
    assert call(n=0) == -1 and "voxels" in _lib.last_error()
    assert call(n=2 ** 31) == -1 and "voxels" in _lib.last_error()
    assert call(ws=need - 1) == -1 and "workspace" in _lib.last_error()
    for kw in (dict(a=None), dict(counts=None), dict(out5=None), dict(workspace=None)):
        assert call(**kw) == -1 and "null" in _lib.last_error()


# ------------------------------------------------------------------------------------------------- CUDA kernel
def _assert_entropies(got, ref):
    """H1, H2, H12 and NMI to 1e-12 relative; MI = H1 + H2 - H12 is a difference, so its error is relative to them."""
    got = [float(v) for v in got]
    for k in (0, 1, 2, 4):
        if np.isnan(ref[k]):
            assert np.isnan(got[k])
        else:
            assert abs(got[k] - ref[k]) <= 1e-12 * abs(ref[k]), (k, got[k], ref[k])
    assert abs(got[3] - ref[3]) <= 1e-12 * max(abs(ref[3]), ref[0] + ref[1]), (got[3], ref[3])


def _out5(ta, tb, bins, nd):
    """(items, 5) [H1, H2, H12, MI, NMI] from the ops-level call (the public functions return MI and NMI only)."""
    from mpgan import ops
    lead = tuple(ta.shape[:ta.dim() - nd])
    items, n = int(np.prod(lead)), int(np.prod(ta.shape[ta.dim() - nd:]))
    counts = torch.empty(items, bins, bins, dtype=torch.int64, device="cuda")
    out5 = torch.empty(items, 5, dtype=torch.float64, device="cuda")
    ops.mutual_info(ta.contiguous(), tb.contiguous(), items, n, bins, counts, None, out5)
    return out5


def _same(x, y):
    """Bit-identical tensors (NaN where NaN)."""
    x, y = x.detach().cpu().numpy().reshape(-1), y.detach().cpu().numpy().reshape(-1)
    return x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _check(a, b, bins, spatial_dims=None, ta=None, tb=None):
    """Device joint histogram, edges and entropies of every leading item against the oracle: counts and edges bit for
    bit, entropies by ``_assert_entropies``.  Returns the device results."""
    from mpgan import transforms as T
    ta = torch.from_numpy(a).cuda() if ta is None else ta
    tb = torch.from_numpy(b).cuda() if tb is None else tb
    counts, e1, e2 = T.joint_histogram(ta, tb, bins=bins, spatial_dims=spatial_dims)
    mi = T.mutual_information(ta, tb, bins=bins, spatial_dims=spatial_dims)
    nmi = T.normalized_mutual_information(ta, tb, bins=bins, spatial_dims=spatial_dims)
    nd = spatial_dims or min(a.ndim, 3)
    lead = a.shape[:a.ndim - nd]
    assert counts.dtype == torch.int64 and tuple(counts.shape) == lead + (bins, bins)
    assert e1.dtype == torch.float32 and tuple(e1.shape) == tuple(e2.shape) == lead + (bins + 1,)
    assert mi.dtype == nmi.dtype == torch.float64 and mi.is_cuda and tuple(mi.shape) == tuple(nmi.shape) == lead
    h = _out5(ta, tb, bins, nd)
    assert _same(mi.reshape(-1), h[:, 3]) and _same(nmi.reshape(-1), h[:, 4])
    c = counts.cpu().numpy().reshape(-1, bins, bins)
    g1, g2 = e1.cpu().numpy().reshape(-1, bins + 1), e2.cpu().numpy().reshape(-1, bins + 1)
    h = h.cpu().numpy()
    ia = a.reshape((-1,) + a.shape[a.ndim - nd:])
    ib = b.reshape((-1,) + b.shape[b.ndim - nd:])
    for i in range(ia.shape[0]):
        rc, r1, r2 = om.joint_histogram(ia[i], ib[i], bins)
        assert np.array_equal(c[i], rc), i
        for g, r, x in ((g1[i], r1, ia[i]), (g2[i], r2, ib[i])):
            assert np.array_equal(g.view(np.uint32), r.view(np.uint32)), i
            assert np.array_equal(g.view(np.uint32), om.histogram_edges(*om.outer_range(x), bins).view(np.uint32))
        _assert_entropies(h[i], om.entropies(rc))
    return counts, e1, e2, mi, nmi


@gpu
@pytest.mark.parametrize("bins", [100, 128, 2, 37])
def test_128_cube_display_range_pair(bins):
    gen, truth = _display_pair((128, 128, 128), 1)
    _check(gen, truth, bins)


@gpu
def test_unit_range_pair_and_ragged_volume():
    _check(*_unit_pair((64, 96, 80), 2), 100)
    _check(*_display_pair((61, 67, 13), 3), 100)        # 53131 voxels: a ragged float4 body and tail
    _check(*_unit_pair((61, 67, 13), 4), 64)


@gpu
def test_per_slice_2d_batch_and_batching_is_invisible():
    """A (S, 1, H, W) stack scored per slice, items starting at every alignment (H W odd), and a copy of the first image
    shifted by one float so that the two images are aligned differently (the all-scalar path)."""
    from mpgan import transforms as T
    gen, truth = _unit_pair((7, 1, 97, 101), 5)
    counts, e1, e2, mi, nmi = _check(gen, truth, 100, spatial_dims=2)
    assert tuple(counts.shape) == (7, 1, 100, 100)
    ta, tb = torch.from_numpy(gen).cuda(), torch.from_numpy(truth).cuda()
    flat = torch.empty(gen.size + 1, device="cuda")
    flat[1:] = ta.reshape(-1)
    shifted = flat[1:].view(ta.shape)
    for x in (ta, shifted):
        for i in range(7):
            one = T.joint_histogram(x[i, 0], tb[i, 0], bins=100)
            assert torch.equal(one[0], counts[i, 0]) and torch.equal(one[1], e1[i, 0]) and torch.equal(one[2], e2[i, 0])
            assert _same(T.mutual_information(x[i, 0], tb[i, 0]), mi[i, 0])
            assert _same(T.normalized_mutual_information(x[i, 0], tb[i, 0]), nmi[i, 0])
    both = _out5(shifted, tb, 100, 2)
    assert _same(both, _out5(ta, tb, 100, 2))


@gpu
def test_3d_batch_is_invisible():
    from mpgan import transforms as T
    pairs = [_display_pair((24, 40, 50), s) for s in (6, 7, 8)]
    gen = torch.from_numpy(np.stack([p[0] for p in pairs])).cuda()
    truth = torch.from_numpy(np.stack([p[1] for p in pairs])).cuda()
    counts, e1, e2 = T.joint_histogram(gen, truth)
    mi = T.mutual_information(gen, truth)
    for i in range(3):
        one = T.joint_histogram(gen[i], truth[i])
        assert torch.equal(one[0], counts[i]) and torch.equal(one[1], e1[i]) and torch.equal(one[2], e2[i])
        assert _same(T.mutual_information(gen[i], truth[i]), mi[i])


@gpu
def test_volume_larger_than_l2():
    """BASELINE config 5's 256 x 512 x 512 volume: 536 MB of inputs, more than the B200's L2.  The oracle histograms it in
    slabs with the whole volume's edges (np.histogramdd with explicit edges bins the same way) and sums the counts."""
    from mpgan import transforms as T
    gen, truth = _display_pair((256, 512, 512), 11)
    counts, e1, e2 = T.joint_histogram(torch.from_numpy(gen).cuda(), torch.from_numpy(truth).cuda())
    h = _out5(torch.from_numpy(gen).cuda(), torch.from_numpy(truth).cuda(), 100, 3)[0].cpu().numpy()
    r1, r2 = (om.histogram_edges(*om.outer_range(v), 100) for v in (gen, truth))
    assert np.array_equal(e1.cpu().numpy().view(np.uint32), r1.view(np.uint32))
    assert np.array_equal(e2.cpu().numpy().view(np.uint32), r2.view(np.uint32))
    ref = np.zeros((100, 100), np.int64)
    for z in range(0, 256, 32):
        ref += np.histogramdd([gen[z:z + 32].ravel(), truth[z:z + 32].ravel()], bins=[r1, r2])[0].astype(np.int64)
    assert np.array_equal(counts.cpu().numpy(), ref)
    _assert_entropies(h, om.entropies(ref))


@gpu
def test_values_on_interior_and_last_edges():
    """Every edge value, the float just below and just above each, lo and hi themselves: the bins must be
    searchsorted's, including values exactly on an interior edge and on the last edge."""
    rng = np.random.RandomState(12)
    for lo, hi, bins in ((-1.0, 1.0, 100), (0.0, 255.0, 100), (0.1, 0.7, 128), (-3.3e-3, 7.9e4, 37), (1e6, 1e6 + 40, 97),
                         (2.0, 2.0 + 2 ** -20, 64)):
        lo, hi = np.float32(lo), np.float32(hi)
        e = om.histogram_edges(lo, hi, bins)
        vals = np.concatenate([e, np.nextafter(e, np.float32(-np.inf)), np.nextafter(e, np.float32(np.inf))])
        vals = vals[(vals >= lo) & (vals <= hi)].astype(np.float32)
        x = np.concatenate([vals, rng.choice(vals, 4099)]).astype(np.float32)
        y = rng.permutation(x)
        assert om.outer_range(x) == (lo, hi)
        _check(x.reshape(1, -1), y.reshape(1, -1), bins, spatial_dims=2)
        _check(np.stack([x, y])[:, None], np.stack([y, x])[:, None], bins, spatial_dims=2)


@gpu
def test_constant_items():
    rng = np.random.RandomState(13)
    y = (rng.rand(3, 17, 19) * 10).astype(np.float32)
    for c in (0.0, 255.0, -1.0, 2.0 ** 25):          # 2^25: lo - 0.5 == lo, every edge equal
        x = np.full_like(y, c)
        _check(x, y, 100, spatial_dims=2)
        _check(y, x, 50, spatial_dims=2)
        _, _, _, mi, nmi = _check(x, np.full_like(y, -7.0), 100, spatial_dims=2)
        assert torch.all(mi == 0) and torch.all(torch.isnan(nmi))


@gpu
def test_non_finite_items_are_nan_and_leave_neighbours_alone():
    from mpgan import transforms as T
    gen, truth = _unit_pair((4, 33, 35), 14)
    bad = gen.copy(), truth.copy()
    bad[0][1, 5, 7] = np.nan
    bad[1][2, 0, 0] = np.inf
    bad[0][3, 9, 9] = -np.inf
    ta, tb = torch.from_numpy(bad[0]).cuda(), torch.from_numpy(bad[1]).cuda()
    counts, e1, e2 = T.joint_histogram(ta, tb, spatial_dims=2)
    mi, nmi = T.mutual_information(ta, tb, spatial_dims=2), T.normalized_mutual_information(ta, tb, spatial_dims=2)
    h = _out5(ta, tb, 100, 2)
    for i in (1, 2, 3):
        assert torch.all(counts[i] == 0) and torch.all(torch.isnan(e1[i])) and torch.all(torch.isnan(e2[i]))
        assert torch.all(torch.isnan(h[i])) and torch.isnan(mi[i]) and torch.isnan(nmi[i])
        with pytest.raises(ValueError):
            om.joint_histogram(bad[0][i], bad[1][i], 100)
    clean = T.joint_histogram(ta[0], tb[0])
    assert torch.equal(clean[0], counts[0]) and torch.equal(clean[1], e1[0]) and torch.equal(clean[2], e2[0])
    assert _same(h[0], _out5(ta[0], tb[0], 100, 2)[0])
    _check(gen[:1], truth[:1], 100, spatial_dims=2)


@gpu
def test_repetition_and_graph_replay_change_no_bit():
    from mpgan import transforms as T
    gen, truth = _display_pair((4, 40, 41, 43), 15)
    ta, tb = torch.from_numpy(gen).cuda(), torch.from_numpy(truth).cuda()
    base = T.joint_histogram(ta, tb, bins=100)
    base_mi = T.mutual_information(ta, tb)
    for _ in range(3):
        again = T.joint_histogram(ta, tb, bins=100)
        assert all(torch.equal(u, v) for u, v in zip(again, base))
        assert _same(T.mutual_information(ta, tb), base_mi)
    sa, sb = ta.clone(), tb.clone()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = T.joint_histogram(sa, sb, bins=100)
        out_mi = T.mutual_information(sa, sb)
    for _ in range(2):
        for t in out:
            t.fill_(7)
        out_mi.fill_(-1.0)
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(u, v) for u, v in zip(out, base)) and _same(out_mi, base_mi)
    sa.copy_(torch.flip(ta, [0]))
    sb.copy_(torch.flip(tb, [0]))
    g.replay()
    assert all(torch.equal(u, torch.flip(v, [0])) for u, v in zip(out, base))
    assert _same(out_mi, torch.flip(base_mi, [0]))


@gpu
def test_evaluate_mutual_information_of_a_generator_output():
    import mpgan
    from mpgan import inference
    from mpgan import transforms as T
    torch.manual_seed(0)
    model = mpgan.GAN(1, 64, 64, precision="fp32").cuda().freeze()
    t1 = torch.from_numpy(_unit_pair((12, 1, 64, 64), 16)[1]).cuda()
    gen = inference.to_display_range(inference.infer_volume(model, t1))
    truth = inference.to_display_range(torch.from_numpy(_display_pair((12, 1, 64, 64), 17)[1]).cuda())
    plain = inference.evaluate(gen, truth)
    s = T.error_sums(gen, truth).tolist()
    assert plain == {"mae": s[0] / gen.numel(), "mse": s[1] / gen.numel()}
    assert inference.evaluate(gen, truth, data_range=255).keys() == {"mae", "mse", "psnr", "ssim"}
    m = inference.evaluate(gen, truth, mi_bins=100)
    assert m.keys() == {"mae", "mse", "mi", "nmi"} and m["mae"] == plain["mae"] and m["mse"] == plain["mse"]
    g, t = gen.cpu().numpy()[:, 0], truth.cpu().numpy()[:, 0]                 # the stack is one volume
    ref = om.entropies(om.joint_histogram(g, t, 100)[0])
    assert abs(m["mi"] - ref[3]) <= 1e-12 * (ref[0] + ref[1]) and abs(m["nmi"] - ref[4]) <= 1e-12 * ref[4]
    both = inference.evaluate(gen, truth, data_range=255, mi_bins=100)
    assert both.keys() == {"mae", "mse", "psnr", "ssim", "mi", "nmi"} and both["mi"] == m["mi"]
    vols = [_display_pair((16, 24, 28), s) for s in (18, 19)]             # (S, 1, D, H, W): mean over the volumes
    g5 = torch.from_numpy(np.stack([v[0] for v in vols])).cuda().unsqueeze(1)
    t5 = torch.from_numpy(np.stack([v[1] for v in vols])).cuda().unsqueeze(1)
    m5 = inference.evaluate(g5, t5, mi_bins=64)
    refs = [om.entropies(om.joint_histogram(v[0], v[1], 64)[0]) for v in vols]
    assert abs(m5["mi"] - np.mean([r[3] for r in refs])) <= 1e-12 * np.mean([r[0] + r[1] for r in refs])
    assert abs(m5["nmi"] - np.mean([r[4] for r in refs])) <= 1e-12
