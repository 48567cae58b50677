"""Generator-only inference over a volume and the post-processing the reference applies to it (SURVEY.md 8f, N1).

Mirrors /root/reference/code/GAN/inferrence.py:147-204 (and minipig_inference.py:101-128): ``model.eval()``,
``model.freeze()``, ``model.generator.forward(t1)`` under ``torch.no_grad()``, then
``ScaleIntensityRangePercentilesd(lower=0, upper=100, b_min=0, b_max=255, clip=True)`` + ``np.round`` on the generated
and ground-truth volumes and ``MeanAbsoluteError`` between them.  The reference feeds one volume per call; here the
slices (2-D) or sub-volumes (3-D) are batched, the rescale / round / metric kernels run on the device and nothing is
copied to the host except the two percentile scalars.
"""
import math
import numbers

import torch

from . import ops
from .nets import UNet
from .transforms import (ScaleIntensityRangePercentiles, _check_bins, _check_data_range, _masked_mean,
                         _mutual_info, _psnr, error_sums, structural_similarity)


class GraphedGenerator:
    """Eval-mode generator forward for a fixed batch shape, captured once into a CUDA graph (the forward is ~180 kernel
    launches; replaying the graph removes the host from the loop).  ``g(x)`` copies ``x`` into the static input, replays
    and returns a copy of the static output."""

    def __init__(self, model, shape, device):
        self.gen = getattr(model, "generator", model)
        self.gen.eval()
        self.x = torch.zeros(shape, dtype=torch.float32, device=device)
        with torch.no_grad():
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self.gen.run_forward(self.x, save=False, need_wgrad=False)      # warm-up outside the capture
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.y, _ = self.gen.run_forward(self.x, save=False, need_wgrad=False)

    def __call__(self, x):
        self.x.copy_(x)
        self.graph.replay()
        return self.y.clone()


@torch.no_grad()
def infer_volume(model, t1, batch=64, graphed=None):
    """``t1``: (S, 1, H, W) slices or (S, 1, D, H, W) sub-volumes, CUDA fp32 in [-1, 1].  Returns the generated T2
    tensor of the same shape.  ``model`` is a ``GAN`` or a ``CasNetGenerator``; BatchNorm uses running statistics.
    ``graphed``: an optional ``GraphedGenerator`` for the full-batch shape."""
    gen = getattr(model, "generator", model)
    if not t1.is_cuda:
        raise RuntimeError("mpgan inference needs CUDA tensors on a B200: there is no CPU fallback")
    was_training = gen.training
    gen.eval()
    try:
        outs = []
        for s in range(0, t1.shape[0], batch):
            x = t1[s:s + batch].contiguous()
            if graphed is not None and tuple(x.shape) == tuple(graphed.x.shape):
                outs.append(graphed(x))        # full batches replay the captured graph; a ragged tail runs eagerly
                continue
            y, _ = gen.run_forward(x, save=False, need_wgrad=False)
            outs.append(y)
        return torch.cat(outs, dim=0) if len(outs) != 1 else outs[0]
    finally:
        gen.train(was_training)


def _roi_of(roi_size, size):
    """MONAI's ``fall_back_tuple``: an entry that is None or <= 0 takes the image extent."""
    if isinstance(roi_size, (str, bytes)) or not hasattr(roi_size, "__len__") or len(roi_size) != len(size):
        raise ValueError(f"roi_size {roi_size!r} needs one entry per spatial dim of {tuple(size)}")
    roi = []
    for r, s in zip(roi_size, size):
        if r is not None and (isinstance(r, bool) or not isinstance(r, numbers.Integral)):
            raise ValueError(f"roi_size {roi_size!r}: entries are integers or None")
        roi.append(int(s) if r is None or r <= 0 else int(r))
    return tuple(roi)


def _window_starts(size, roi, overlap):
    """MONAI 0.4.0 ``_get_scan_interval`` / ``dense_patch_slices`` along one dim, in padded coordinates."""
    padded = max(size, roi)
    iv = roi if roi == padded else max(int(roi * (1 - overlap)), 1)
    n = 1 + max(-(-(padded - roi) // iv), 0)
    return [min(j * iv, padded - roi) for j in range(n)]


def _importance_taps(roi, mode, sigma):
    """One dim of the separable importance map: all ones, or the sampled Gaussian exp(-(i - roi//2)^2 / (2 (sigma
    roi)^2)) in fp64 with underflowed taps raised to the dim's smallest positive tap."""
    if mode == "constant":
        return [1.0] * roi
    sd = sigma * roi
    t = [math.exp(-((i - roi // 2) ** 2) / (2.0 * sd * sd)) for i in range(roi)]
    floor = min(v for v in t if v > 0.0)
    return [v if v > 0.0 else floor for v in t]


def _real(v):
    return isinstance(v, numbers.Real) and not isinstance(v, bool) and math.isfinite(v)


@torch.no_grad()
def sliding_window_inference(inputs, roi_size, sw_batch_size, predictor, overlap=0.25, mode="constant",
                             sigma_scale=0.125, padding_mode="constant", cval=0.0):
    """MONAI 0.4.0 ``sliding_window_inference`` on the device: run ``predictor`` over overlapping ``roi_size`` windows
    of ``inputs`` and blend its predictions into one output of the input's spatial size.

    ``inputs``: (B, C_in, *S) CUDA fp32, 2 or 3 spatial dims.  ``roi_size``: one entry per spatial dim; None or <= 0
    takes the image extent.  A dim shorter than its roi is padded with ``cval`` (split as MONAI does: the smaller half
    before); padding is virtual, read by the gather kernel.  Windows step by ``max(int(roi (1 - overlap)), 1)`` and the
    last one is aligned to the padded end; they are ordered image-major, first spatial dim slowest, and ``predictor``
    sees them in consecutive runs of at most ``sw_batch_size`` ((n, C_in, *roi) -> (n, C_out, *roi), CUDA fp32; a run
    may span two images).  ``mode``: "constant" (plain mean of the covering windows) or "gaussian" (importance map
    prod_d exp(-(i_d - roi_d // 2)^2 / (2 (sigma_d roi_d)^2)), ``sigma_scale`` a scalar or one per dim: the sampled
    Gaussian, which is what MONAI 0.4.0's filtered delta amounts to; later MONAI releases build it differently).
    Returns (B, C_out, *S) fp32.  The weighted sums are fp64 with one rounding to fp32 (MONAI accumulates in fp32, a
    difference of ~1e-7 relative), and the result is bit-identical run to run.

    Memory: the predictions of every window are kept until the blend, B * nwin * C_out * prod(roi) * 4 bytes
    (nwin = windows per image), plus one chunk of sw_batch_size input windows.  Only ``padding_mode="constant"``."""
    if not torch.is_tensor(inputs) or inputs.dim() not in (4, 5):
        raise ValueError("sliding_window_inference takes (B, C, *S) inputs with 2 or 3 spatial dims")
    if inputs.dtype != torch.float32:
        raise ValueError(f"sliding_window_inference takes fp32 inputs, got {inputs.dtype}")
    size = tuple(inputs.shape[2:])
    if min(inputs.shape) < 1:
        raise ValueError(f"empty inputs {tuple(inputs.shape)}")
    roi = _roi_of(roi_size, size)
    if isinstance(sw_batch_size, bool) or not isinstance(sw_batch_size, numbers.Integral) or sw_batch_size < 1:
        raise ValueError(f"sw_batch_size must be a positive integer, got {sw_batch_size!r}")
    if not _real(overlap) or not 0 <= overlap < 1:
        raise ValueError(f"overlap must be in [0, 1), got {overlap!r}")
    if mode not in ("constant", "gaussian"):
        raise ValueError(f"mode must be 'constant' or 'gaussian', got {mode!r}")
    if padding_mode != "constant":
        raise ValueError(f"only padding_mode='constant' is supported, got {padding_mode!r}")
    sigmas = tuple(sigma_scale) if hasattr(sigma_scale, "__len__") else (sigma_scale,) * len(size)
    if len(sigmas) != len(size) or not all(_real(v) and v > 0 for v in sigmas):
        raise ValueError(f"sigma_scale must be > 0, a scalar or one per spatial dim, got {sigma_scale!r}")
    if not _real(cval):
        raise ValueError(f"cval must be a finite number, got {cval!r}")
    if not callable(predictor):
        raise ValueError("predictor must be callable")
    if not inputs.is_cuda:
        raise RuntimeError("mpgan inference needs CUDA tensors on a B200: there is no CPU fallback")

    starts = [_window_starts(s, r, overlap) for s, r in zip(size, roi)]
    taps = [_importance_taps(r, mode, float(sg)) for r, sg in zip(roi, sigmas)]
    table = ops.WindowTable(size, roi, starts, taps, inputs.device)
    x = inputs.contiguous()
    batch = x.shape[0]
    total = batch * table.nwin
    chunk = torch.empty((min(sw_batch_size, total), x.shape[1]) + roi, dtype=torch.float32, device=x.device)
    preds = None
    for first in range(0, total, sw_batch_size):
        n = min(sw_batch_size, total - first)
        y = predictor(ops.window_gather(x, table, first, n, float(cval), chunk[:n]))
        c_out = y.shape[1] if torch.is_tensor(y) and y.dim() == 2 + len(roi) else -1
        if (not torch.is_tensor(y) or not y.is_cuda or y.device != x.device or y.dtype != torch.float32
                or tuple(y.shape) != (n, c_out) + roi or (preds is not None and c_out != preds.shape[1])):
            got = (tuple(y.shape), y.dtype, str(y.device)) if torch.is_tensor(y) else type(y)
            raise ValueError(f"predictor must return ({n}, C_out, *{roi}) fp32 on {x.device} with the same C_out for "
                             f"every chunk, got {got}")
        if preds is None:
            preds = torch.empty((total, c_out) + roi, dtype=torch.float32, device=x.device)
        preds[first:first + n].copy_(y)
    out = torch.empty((batch, preds.shape[1]) + size, dtype=torch.float32, device=x.device)
    return ops.window_blend(preds, batch, table, out)


def infer_volume_sliding(model, t1, roi_size, sw_batch_size=4, overlap=0.25, mode="constant", sigma_scale=0.125,
                         cval=0.0, graphed=None):
    """``infer_volume`` for volumes of any size: ``sliding_window_inference`` with the generator as the predictor.

    ``t1``: (B, 1, *S) CUDA fp32, 2 or 3 spatial dims matching the generator; ``model``: a ``GAN`` or a
    ``CasNetGenerator``, run in eval mode (the training flag is restored afterwards).  Every roi extent must be divisible
    by the product of the generator's UNet strides (8 for GAN_final.py's (2, 2, 2), 16 for the perceptual variant's
    (2, 2, 2, 2)); the generator is trained on one size, so ``roi_size`` is normally that size.  Each chunk of windows
    runs as ``infer_volume(model, chunk, batch=sw_batch_size, graphed=graphed)``: with ``graphed``, a
    ``GraphedGenerator`` of shape (sw_batch_size, 1, *roi), full chunks replay the graph and a ragged last chunk runs
    eagerly.  ``cval`` fills the padding of dims shorter than the roi: -1 is the background of [-1, 1]-scaled volumes.
    Returns the generated T2 volume, (B, 1, *S) fp32."""
    gen = getattr(model, "generator", model)
    unet = next(m for m in gen.model if isinstance(m, UNet))
    factor = math.prod(unet.strides)
    if not torch.is_tensor(t1) or t1.dim() != 2 + gen.dims or t1.shape[1] != 1:
        raise ValueError(f"infer_volume_sliding takes (B, 1, *S) with {gen.dims} spatial dims for this generator, got "
                         f"{tuple(t1.shape) if torch.is_tensor(t1) else type(t1)}")
    roi = _roi_of(roi_size, tuple(t1.shape[2:]))
    if any(r % factor for r in roi):
        raise ValueError(f"roi {roi}: every extent must be divisible by {factor}, the product of the generator's UNet "
                         f"strides {tuple(unet.strides)}")
    if graphed is not None and tuple(graphed.x.shape) != (sw_batch_size, 1) + roi:
        raise ValueError(f"graphed generator of shape {tuple(graphed.x.shape)}, need {(sw_batch_size, 1) + roi}")
    was_training = gen.training
    gen.eval()
    try:
        return sliding_window_inference(t1, roi, sw_batch_size,
                                        lambda x: infer_volume(model, x, batch=sw_batch_size, graphed=graphed),
                                        overlap=overlap, mode=mode, sigma_scale=sigma_scale, cval=cval)
    finally:
        gen.train(was_training)


def to_display_range(vol, out_dtype=torch.float32):
    """inferrence.py:152-161 / 190-199: 0/100-percentile rescale to [0, 255], clip, round half to even."""
    return ScaleIntensityRangePercentiles(0, 100, 0, 255, clip=True)(vol, round_half_even=True, out_dtype=out_dtype)


def evaluate(generated, truth, data_range=None, mi_bins=None, mask=None):
    """{"mae", "mse"} between two volumes (torchmetrics MeanAbsoluteError / MeanSquaredError, one pass).

    With ``data_range`` (255 for display-range volumes) also "psnr" and "ssim", scikit-image's defaults as
    psnr_ssim_metric.py:88-95 scores whole volumes: a slice stack (S, 1, H, W) is the one volume (S, H, W), and
    (S, 1, D, H, W) gives the mean of the S volume SSIMs.  With ``mi_bins`` (100 is scikit-image's default) also "mi"
    and "nmi", the mutual information and scikit-image's normalized mutual information of the same volumes in nats
    (``transforms.mutual_information``), a batch again giving the mean over its volumes.

    With ``mask`` (bool or uint8, the shape of ``generated``; e.g. ``transforms.foreground_mask(truth)``) every score is
    taken inside it, with the same keys: MAE / MSE / PSNR over the voxels in the mask, SSIM over the voxels whose centre
    is in it, MI / NMI from the histogram of those voxels.  The mask is squeezed as the images are.  A volume with an
    empty mask scores NaN."""
    if data_range is not None:
        _check_data_range(data_range)
    if mi_bins is not None:
        _check_bins(mi_bins)
    if mask is None:
        s = error_sums(generated, truth).tolist()
        n = max(generated.numel(), 1)
        res = {"mae": s[0] / n, "mse": s[1] / n}
    else:
        s = error_sums(generated, truth, mask).tolist()
        res = {"mae": _masked_mean(s, 0), "mse": _masked_mean(s, 1)}
    if data_range is None and mi_bins is None:
        return res
    g, t, m = generated, truth, mask
    if g.dim() in (4, 5):
        if g.shape[1] != 1:
            raise ValueError(f"evaluate scores one-channel stacks (S, 1, ...), got {tuple(g.shape)}")
        g, t = g.squeeze(1), t.squeeze(1)
        m = None if m is None else m.squeeze(1)
    if data_range is not None:
        res["psnr"] = _psnr(res["mse"], data_range)
        res["ssim"] = float(structural_similarity(g, t, data_range=data_range, mask=m).mean())
    if mi_bins is not None:
        h = _mutual_info(g.float(), t.float(), mi_bins, None, False, m)[2].reshape(-1, 5).mean(dim=0).tolist()
        res["mi"], res["nmi"] = h[3], h[4]
    return res
