"""Generator-only inference over a volume and the post-processing the reference applies to it (SURVEY.md 8f, N1).

Mirrors /root/reference/code/GAN/inferrence.py:147-204 (and minipig_inference.py:101-128): ``model.eval()``,
``model.freeze()``, ``model.generator.forward(t1)`` under ``torch.no_grad()``, then
``ScaleIntensityRangePercentilesd(lower=0, upper=100, b_min=0, b_max=255, clip=True)`` + ``np.round`` on the generated
and ground-truth volumes and ``MeanAbsoluteError`` between them.  The reference feeds one volume per call; here the
slices (2-D) or sub-volumes (3-D) are batched, the rescale / round / metric kernels run on the device and nothing is
copied to the host except the two percentile scalars.
"""
import torch

from .transforms import ScaleIntensityRangePercentiles, _check_data_range, _psnr, error_sums, structural_similarity


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


def to_display_range(vol, out_dtype=torch.float32):
    """inferrence.py:152-161 / 190-199: 0/100-percentile rescale to [0, 255], clip, round half to even."""
    return ScaleIntensityRangePercentiles(0, 100, 0, 255, clip=True)(vol, round_half_even=True, out_dtype=out_dtype)


def evaluate(generated, truth, data_range=None):
    """{"mae", "mse"} between two volumes (torchmetrics MeanAbsoluteError / MeanSquaredError, one pass).

    With ``data_range`` (255 for display-range volumes) also "psnr" and "ssim", scikit-image's defaults as
    psnr_ssim_metric.py:88-95 scores whole volumes: a slice stack (S, 1, H, W) is the one volume (S, H, W), and
    (S, 1, D, H, W) gives the mean of the S volume SSIMs."""
    if data_range is not None:
        _check_data_range(data_range)
    s = error_sums(generated, truth).tolist()
    n = max(generated.numel(), 1)
    res = {"mae": s[0] / n, "mse": s[1] / n}
    if data_range is None:
        return res
    g, t = generated, truth
    if g.dim() in (4, 5):
        if g.shape[1] != 1:
            raise ValueError(f"evaluate scores one-channel stacks (S, 1, ...), got {tuple(g.shape)}")
        g, t = g.squeeze(1), t.squeeze(1)
    res["psnr"] = _psnr(res["mse"], data_range)
    res["ssim"] = float(structural_similarity(g, t, data_range=data_range).mean())
    return res
