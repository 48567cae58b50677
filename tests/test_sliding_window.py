"""Sliding-window inference (MONAI 0.4.0 ``sliding_window_inference``, the call minipig_inference.py:110-114 leaves
commented out): ``mpgan.inference.sliding_window_inference`` / ``infer_volume_sliding`` over the window gather and blend
kernels (csrc/window.cu).

CPU tests pin the numpy fp64 oracle (oracle/sliding_window.py) against known geometries and a brute-force MONAI-style
count-map accumulation, and check that every argument error is raised before the device is touched and that the C ABI
rejects bad geometry tables.  ``-m gpu`` tests compare the kernels with the oracle (gather bit-exact, blend to 1e-6), run
the generator end to end against the oracle generator, and check that chunking, graph replay and repetition change no
bit."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from oracle import sliding_window as osw

gpu = pytest.mark.gpu

# (S, roi, overlap) -> (starts, lo)
GEOMETRIES = [((200, 128, 0.25), ([0, 72], 0)), ((128, 128, 0.25), ([0], 0)), ((100, 128, 0.25), ([0], 14)),
              ((256, 128, 0.5), ([0, 64, 128], 0)), ((256, 128, 0.0), ([0, 128], 0)),
              ((257, 128, 0.0), ([0, 128, 129], 0)), ((512, 256, 0.25), ([0, 192, 256], 0)),
              ((70, 32, 0.25), ([0, 24, 38], 0))]
MODES = ["constant", "gaussian"]


def _table(size, roi_size, overlap, mode="constant", sigma=0.125, device="cuda"):
    from mpgan import ops
    geo = osw.geometry(size, roi_size, overlap)
    taps = [osw.importance_taps(r, mode, sigma) for r, _, _ in geo]
    return geo, ops.WindowTable(size, [g[0] for g in geo], [g[1] for g in geo], taps, device)


# ------------------------------------------------------------------------------------------------- oracle (CPU)
@pytest.mark.parametrize("case,expected", GEOMETRIES)
def test_oracle_geometry_table(case, expected):
    s, roi, overlap = case
    assert osw.scan_starts(s, roi, overlap) == expected
    from mpgan import inference
    assert inference._window_starts(s, roi, overlap) == expected[0]


def test_roi_fall_back():
    assert osw.fall_back_roi((None, 0, -1, 32), (5, 6, 7, 8)) == (5, 6, 7, 32)
    from mpgan import inference
    assert inference._roi_of((None, 0, -1, 32), (5, 6, 7, 8)) == (5, 6, 7, 32)


def _brute_force(preds, batch, size, roi_size, overlap, mode, sigma):
    """MONAI's loop: output += w * y and count += w on the padded canvas, then crop."""
    geo = osw.geometry(size, roi_size, overlap)
    w = np.ones(())
    for r, _, _ in geo:
        w = np.multiply.outer(w, osw.importance_taps(r, mode, sigma))
    padded = tuple(max(s, g[0]) for s, g in zip(size, geo))
    out = np.zeros((batch, preds.shape[1]) + padded)
    count = np.zeros(padded)
    k = 0
    for b in range(batch):
        for st in osw.window_starts(geo):
            sl = tuple(slice(s, s + g[0]) for s, g in zip(st, geo))
            out[(b, slice(None)) + sl] += w * preds[k]
            count[sl] += w if b == 0 else 0.0
            k += 1
    crop = tuple(slice(g[2], g[2] + s) for s, g in zip(size, geo))
    return (out / count)[(slice(None), slice(None)) + crop]


@pytest.mark.parametrize("size,roi,overlap", [((40, 33), (16, 16), 0.25), ((9, 21), (16, 8), 0.5),
                                              ((13, 7, 20), (8, 8, 8), 0.25), ((5, 11, 6), (8, 4, 8), 0.6)])
@pytest.mark.parametrize("mode", MODES)
def test_oracle_blend_matches_count_map_accumulation(size, roi, overlap, mode):
    geo = osw.geometry(size, roi, overlap)
    nwin = len(osw.window_starts(geo))
    preds = np.random.RandomState(0).uniform(-1, 1, (2 * nwin, 3) + roi)
    got = osw.blend(preds, 2, geo, size, mode, 0.125)
    ref = _brute_force(preds, 2, size, roi, overlap, mode, 0.125)
    assert got.shape == (2, 3) + size
    assert np.abs(got - ref).max() <= 1e-12


def test_oracle_identity_and_padding():
    x = np.random.RandomState(1).uniform(-1, 1, (2, 1, 20, 9)).astype(np.float32)
    assert np.array_equal(osw.sliding_window_inference(x, (8, 16), 3, lambda w: w), x)
    win = osw.extract_windows(x, osw.geometry((20, 9), (8, 16), 0.25), 0, 1, -1.0)
    assert win.shape == (1, 1, 8, 16) and (win[..., :3] == -1).all() and (win[..., 12:] == -1).all()
    assert np.array_equal(win[0, 0, :, 3:12], x[0, 0, :8])


# ------------------------------------------------------------------------------------------- argument checks (CPU)
def test_arguments_are_validated_before_the_device():
    from mpgan import inference
    x = torch.zeros(2, 1, 40, 30)
    ident = lambda t: t  # noqa: E731
    bad = [dict(roi_size=(16,)), dict(roi_size=(16, 16, 16)), dict(roi_size=(16.0, 16)), dict(roi_size=16),
           dict(sw_batch_size=0), dict(sw_batch_size=1.5), dict(overlap=1.0), dict(overlap=-0.1),
           dict(overlap=float("nan")), dict(mode="bilinear"), dict(padding_mode="reflect"), dict(sigma_scale=0.0),
           dict(sigma_scale=(0.1,)), dict(sigma_scale=(0.1, -1.0)), dict(sigma_scale=float("inf")),
           dict(cval=float("nan")), dict(predictor=None)]
    for kw in bad:
        args = dict(inputs=x, roi_size=(16, 16), sw_batch_size=2, predictor=ident)
        args.update(kw)
        with pytest.raises(ValueError):
            inference.sliding_window_inference(**args)
    for inp in (torch.zeros(40, 30), torch.zeros(1, 1, 1, 4, 4, 4), torch.zeros(2, 1, 40, 30, dtype=torch.float64)):
        with pytest.raises(ValueError):
            inference.sliding_window_inference(inp, (16, 16), 2, ident)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        inference.sliding_window_inference(x, (16, None), 2, ident, mode="gaussian", sigma_scale=(0.1, 0.2))


def test_generator_roi_must_divide_by_the_stride_product():
    from mpgan import CasNetGenerator, inference
    final = CasNetGenerator((1, 64, 64), n_unet_blocks=1, precision="fp32")
    perceptual = CasNetGenerator((1, 64, 64), n_unet_blocks=1, channels=(32, 64, 128, 256), strides=(2, 2, 2, 2),
                                 precision="fp32")
    x = torch.zeros(1, 1, 100, 90)
    with pytest.raises(ValueError, match="divisible by 8"):
        inference.infer_volume_sliding(final, x, (60, 64))
    with pytest.raises(ValueError, match="divisible by 8"):
        inference.infer_volume_sliding(final, x, (None, 64))      # falls back to 100
    with pytest.raises(ValueError, match="divisible by 16"):
        inference.infer_volume_sliding(perceptual, x, (72, 64))
    with pytest.raises(ValueError):
        inference.infer_volume_sliding(final, torch.zeros(1, 2, 64, 64), (64, 64))     # one input channel
    with pytest.raises(ValueError):
        inference.infer_volume_sliding(final, torch.zeros(1, 1, 64, 64, 64), (64, 64, 64))   # rank of the generator
    final.train()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        inference.infer_volume_sliding(final, x, (64, 64))
    assert final.training                                           # the training flag is restored


def test_c_abi_rejects_bad_geometry():
    from mpgan import _lib
    lib = _lib.load()
    _, tab = _table((45, 70, 37), (32, 32, 32), 0.25, "gaussian", device="cpu")
    good = tab.host
    p = 256   # device pointers are never dereferenced: the checks come first

    def gather(t, first=0, count=1, x=p, words=None):
        words = t.numel() if words is None else words
        return lib.mpgan_window_gather(x, 1, 1, t.data_ptr(), p, words, first, count, 0.0, p, None)

    def blend(t, words=None):
        return lib.mpgan_window_blend(p, 1, 1, t.data_ptr(), p, t.numel() if words is None else words, p, None)

    def edit(i, v, dtype=torch.int32):
        t = good.clone()
        if dtype == torch.int32:
            t[i] = v
        else:
            t.view(torch.float64)[i] = v
        return t

    nwin = 2 * 3 * 2
    assert gather(good, x=None) == -1 and "null" in _lib.last_error()
    assert lib.mpgan_window_blend(p, 1, 1, None, p, good.numel(), p, None) == -1
    assert lib.mpgan_window_blend(p, 1, 1, good.data_ptr(), None, good.numel(), p, None) == -1
    for f in (gather, blend):
        assert f(edit(0, 4)) == -1 and "rank" in _lib.last_error()
        assert f(edit(2, 0)) == -1 and "positive" in _lib.last_error()
        assert f(edit(5, -3)) == -1
        assert f(edit(8, 1)) == -1 and "lo" in _lib.last_error()        # lo of dim 1 must be 0 for S 70 >= roi 32
        assert f(good, words=good.numel() - 2) == -1 and "words" in _lib.last_error()
        assert f(edit(16 + 1, 14)) == -1 and "past padded extent" in _lib.last_error()   # 14 + 32 > 45
        assert f(edit(16 + 2 + 1, 0)) == -1 and "increasing" in _lib.last_error()
        assert f(edit(16 + 7 + 2 * 40, 0)) == -1 and "coverage" in _lib.last_error()     # dim 0, p = 40: windows [1, 1]
        taps_at = good.numel() - 2 * (32 * 3)
        assert f(edit(taps_at // 2 + 5, 0.0, torch.float64)) == -1 and "tap" in _lib.last_error()
    assert gather(good, first=nwin - 1, count=2) == -1 and "outside" in _lib.last_error()
    assert gather(good, first=-1) == -1 and gather(good, count=0) == -1
    _, tab2 = _table((40, 30), (16, 16), 0.25, device="cpu")
    t = tab2.host.clone()
    t[1] = 2                                                        # rank 2 with a non-trivial leading dim
    assert gather(t) == -1 and "rank 2" in _lib.last_error()


# ------------------------------------------------------------------------------------------------- CUDA kernels
def _rand(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g) * 2 - 1


@gpu
@pytest.mark.parametrize("size,roi,overlap", [((70, 45), (32, 64), 0.25), ((20, 37, 45), (16, 48, 32), 0.25),
                                              ((33, 128), (32, 64), 0.5)])
def test_gather_matches_oracle_bit_exact(size, roi, overlap):
    from mpgan import ops
    x = _rand((3, 2) + size, 1)
    xd = x.cuda()
    geo, tab = _table(size, roi, overlap)
    nwin = tab.nwin
    total = 3 * nwin
    for first, count in [(0, total), (nwin - 1, 3), (2 * nwin - 2, 2), (total - 1, 1)]:   # chunks straddle images
        out = torch.full((count, 2) + roi, 7.0, device="cuda")
        ops.window_gather(xd, tab, first, count, -0.5, out)
        ref = osw.extract_windows(x.numpy(), geo, first, count, -0.5)
        assert np.array_equal(out.cpu().numpy(), ref), (first, count)
    view = xd[1:]                                                   # an input at a storage offset
    out = torch.empty((nwin, 2) + roi, device="cuda")
    ops.window_gather(view, tab, 0, nwin, 0.0, out)
    assert np.array_equal(out.cpu().numpy(), osw.extract_windows(x[1:].numpy(), geo, 0, nwin, 0.0))


@gpu
@pytest.mark.parametrize("size,roi,overlap", [((70, 45), (32, 64), 0.25), ((20, 37, 45), (16, 48, 32), 0.25),
                                              ((17, 9, 40), (8, 8, 16), 0.6)])
@pytest.mark.parametrize("mode", MODES)
def test_blend_matches_oracle(size, roi, overlap, mode):
    from mpgan import ops
    geo, tab = _table(size, roi, overlap, mode, 0.125)
    preds = _rand((2 * tab.nwin, 3) + roi, 2)
    out = ops.window_blend(preds.cuda(), 2, tab, torch.empty((2, 3) + size, device="cuda"))
    ref = osw.blend(preds.numpy(), 2, geo, size, mode, 0.125)
    assert np.abs(out.cpu().numpy() - ref).max() <= 1e-6


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_end_to_end_with_channel_changing_predictor(mode):
    """C_in = 2 -> C_out = 3 through a nonlinear predictor; sigma per dim; chunks of 5 windows spanning images."""
    from mpgan import inference
    x = _rand((2, 2, 30, 41, 19), 3)

    def pred_t(w):
        return torch.cat([torch.sin(3 * w[:, :1]), w[:, 1:] * w[:, :1], torch.tanh(w.sum(1, keepdim=True))], 1)

    got = inference.sliding_window_inference(x.cuda(), (16, 24, 32), 5, pred_t, overlap=0.4, mode=mode,
                                             sigma_scale=(0.1, 0.2, 0.15), cval=0.25)
    ref = osw.sliding_window_inference(x.numpy(), (16, 24, 32), 5, lambda w: pred_t(torch.from_numpy(w)).numpy(),
                                       overlap=0.4, mode=mode, sigma_scale=(0.1, 0.2, 0.15), cval=0.25)
    assert got.shape == (2, 3, 30, 41, 19) and got.dtype == torch.float32
    assert np.abs(got.cpu().numpy() - ref).max() <= 1e-6


@gpu
@pytest.mark.parametrize("size,roi", [((2, 3, 200, 173), (128, 128)), ((1, 2, 45, 70, 37), (32, 32, 32)),
                                      ((2, 1, 100, 300), (128, 64))])
def test_identity_predictor_returns_the_input(size, roi):
    from mpgan import inference
    x = _rand(size, 4).cuda()
    same = inference.sliding_window_inference(x, roi, 4, lambda w: w, mode="constant")
    assert torch.equal(same, x)
    g = inference.sliding_window_inference(x, roi, 4, lambda w: w, mode="gaussian")
    assert (g.view(torch.int32) - x.view(torch.int32)).abs().max() <= 1          # <= 1 fp32 ulp


@gpu
def test_predictor_results_are_checked():
    from mpgan import inference
    x = torch.zeros(1, 1, 40, 40, device="cuda")
    for f in (lambda w: w[:, :, :8], lambda w: w.double(), lambda w: w.cpu(), lambda w: w[0], lambda w: None):
        with pytest.raises(ValueError):
            inference.sliding_window_inference(x, (16, 16), 2, f)
    calls = []

    def varying(w):                                                # C_out changes between chunks
        calls.append(1)
        return w if len(calls) == 1 else torch.cat([w, w], 1)
    with pytest.raises(ValueError):
        inference.sliding_window_inference(x, (16, 16), 2, varying)


def _models_2d(size):
    import mpgan
    from oracle.gan import GANOracle
    torch.manual_seed(0)
    ora = GANOracle("final", dims=2, spatial=size).eval()
    model = mpgan.GAN(1, size, size, precision="fp32")
    model.load_state_dict(ora.state_dict())
    model.cuda().freeze()
    return ora, model


def _oracle_predictor(gen):
    def f(w):
        with torch.no_grad():
            return gen(torch.from_numpy(w)).numpy()
    return f


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_roi_equal_to_the_image_is_infer_volume(mode):
    from mpgan import inference
    _, model = _models_2d(64)
    t1 = _rand((5, 1, 64, 64), 5).cuda()
    ref = inference.infer_volume(model, t1, batch=2)
    got = inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=2, mode=mode)
    assert torch.equal(got, ref)


@gpu
def test_generator_2d_end_to_end_against_oracle():
    from mpgan import inference
    ora, model = _models_2d(128)
    cases = [((3, 1, 200, 173), 6, dict(mode="gaussian")), ((2, 1, 100, 300), 4, dict(mode="constant", cval=-1.0))]
    for shape, seed, kw in cases:
        t1 = _rand(shape, seed)
        ref = osw.sliding_window_inference(t1.numpy(), (128, 128), 4, _oracle_predictor(ora.generator), overlap=0.25,
                                           **kw)
        model.generator.set_precision("fp32")
        got = inference.infer_volume_sliding(model, t1.cuda(), (128, 128), sw_batch_size=4, overlap=0.25, **kw)
        assert got.shape == shape
        assert rel_l2(got, torch.from_numpy(ref)) <= 1e-4, shape
        model.generator.set_precision("bf16")
        got16 = inference.infer_volume_sliding(model, t1.cuda(), (128, 128), sw_batch_size=4, overlap=0.25, **kw)
        assert rel_l2(got16, torch.from_numpy(ref)) <= 1e-2, shape


@gpu
def test_generator_3d_end_to_end_against_oracle():
    from mpgan import CasNetGenerator, inference
    from oracle.nets import CasNetGenerator as OGen
    torch.manual_seed(0)
    ora = OGen((1, 32, 32, 32), 6, 3).eval()
    gen = CasNetGenerator((1, 32, 32, 32), precision="fp32")
    gen.load_state_dict(ora.state_dict())
    gen.cuda()
    t1 = _rand((1, 1, 45, 70, 37), 7)
    got = inference.infer_volume_sliding(gen, t1.cuda(), (32, 32, 32), sw_batch_size=4, mode="gaussian")
    ref = osw.sliding_window_inference(t1.numpy(), (32, 32, 32), 4, _oracle_predictor(ora), mode="gaussian")
    assert got.shape == t1.shape and rel_l2(got, torch.from_numpy(ref)) <= 1e-4


@gpu
def test_chunking_graph_replay_and_repetition_change_no_bit():
    from mpgan import inference
    _, model = _models_2d(64)
    t1 = _rand((2, 1, 100, 90), 8).cuda()                           # 4 windows per image, 8 in all
    base = inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=1, mode="gaussian")
    for sw in (3, 8):
        assert torch.equal(inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=sw, mode="gaussian"), base)
    gg = inference.GraphedGenerator(model, (3, 1, 64, 64), torch.device("cuda"))
    graphed = inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=3, mode="gaussian", graphed=gg)
    assert torch.equal(graphed, base)                               # 3 + 3 replayed, the last 2 eager
    again = inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=3, mode="gaussian", graphed=gg)
    assert torch.equal(again, base)
    with pytest.raises(ValueError):
        inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=4, graphed=gg)
    model.generator.train()
    inference.infer_volume_sliding(model, t1, (64, 64), sw_batch_size=8)
    assert model.generator.training
