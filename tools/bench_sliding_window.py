"""Sliding-window inference on the device (mpgan.inference.infer_volume_sliding): CUDA-event times after warm-up, one
JSON line.  Cases: the reference-literal 3-D generator (GAN_final.py: 6 UNets, channels 16..128, trained at 128^3) over a
256^3 volume with roi 128^3, overlap 0.25 and 0.5, Gaussian blend; the 2-D generator trained at 256^2 over 256 slices of
512^2 with roi 256^2, next to whole-slice infer_volume at 512^2.  For each case: the call's device time, the time of
the same number of bare GraphedGenerator replays, and the gather and blend kernels on their own with achieved GB/s
against the bytes they must move (computed below from shapes).  The predictions buffer (226 MB and 604 MB) is larger than
the B200's 126 MB L2, so the blend streams it from HBM; the 3-D gather reads a 67 MB input that fits in L2.
usage: python tools/bench_sliding_window.py [reps]"""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
import mpgan  # noqa: E402
from mpgan import inference, ops  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_GBS = 7700.0   # data sheet, HGX B200 per GPU


def timed(fn, n):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def inside(starts, roi, lo, size):
    """Voxels of each window inside the image, summed over the windows of one image (per dim, then multiplied)."""
    tot = 1
    for st, r, l, s in zip(starts, roi, lo, size):
        tot *= sum(max(0, min(a + r, l + s) - max(a, l)) for a in st)
    return tot


def case(model, x, roi, sw, overlap, mode="gaussian"):
    size, batch = tuple(x.shape[2:]), x.shape[0]
    gg = inference.GraphedGenerator(model, (sw, 1) + roi, dev)
    run = lambda: inference.infer_volume_sliding(model, x, roi, sw_batch_size=sw, overlap=overlap, mode=mode,  # noqa: E731
                                                 graphed=gg)
    ms_call, _ = timed(run, reps)
    starts = [inference._window_starts(s, r, overlap) for s, r in zip(size, roi)]
    taps = [inference._importance_taps(r, mode, 0.125) for r in roi]
    table = ops.WindowTable(size, roi, starts, taps, dev)
    total = batch * table.nwin
    chunks = math.ceil(total / sw)
    win = torch.randn((sw, 1) + roi, device=dev)
    ms_gen, _ = timed(lambda: [gg(win) for _ in range(chunks)], reps)
    xc = x.contiguous()

    def gather_all():
        for first in range(0, total, sw):
            ops.window_gather(xc, table, first, min(sw, total - first), -1.0, win[:min(sw, total - first)])
    ms_gather, _ = timed(gather_all, reps)
    preds = torch.rand((total, 1) + roi, device=dev) * 2 - 1
    out = torch.empty_like(x)
    ms_blend, _ = timed(lambda: ops.window_blend(preds, batch, table, out), reps)
    vox = math.prod(roi)
    lo = [max(r - s, 0) // 2 for s, r in zip(size, roi)]
    in_img = batch * inside(starts, roi, lo, size)
    gather_bytes = 4 * (total * vox + in_img)              # every window element written, the in-image ones read
    blend_bytes = 4 * (in_img + x.numel())                 # in-image predictions read once, the output written once
    return {"windows": total, "sw_batch_size": sw, "chunks": chunks, "call_ms": ms_call,
            "bare_graph_replays_ms": ms_gen, "gather_ms": ms_gather, "blend_ms": ms_blend,
            "gather_plus_blend_share_of_call": (ms_gather + ms_blend) / ms_call,
            "gather_gbs": gather_bytes / (ms_gather * 1e-3) / 1e9, "blend_gbs": blend_bytes / (ms_blend * 1e-3) / 1e9,
            "blend_frac_hbm_datasheet": blend_bytes / (ms_blend * 1e-3) / 1e9 / HBM_GBS,
            "predictions_mb": total * vox * 4 / 1e6}


g = torch.Generator().manual_seed(0)
torch.manual_seed(0)
res = {}
m3 = mpgan.GAN(1, 128, 128, 128).cuda().freeze()
vol = (torch.rand((1, 1, 256, 256, 256), generator=g) * 2 - 1).to(dev)
for ov in (0.25, 0.5):
    res[f"3d_256cube_roi128_overlap{ov}"] = case(m3, vol, (128, 128, 128), 3, ov)
del m3
torch.cuda.empty_cache()
m2 = mpgan.GAN(1, 256, 256).cuda().freeze()
slices = (torch.rand((256, 1, 512, 512), generator=g) * 2 - 1).to(dev)
res["2d_256x512x512_roi256_overlap0.25"] = r2 = case(m2, slices, (256, 256), 64, 0.25)
g512 = inference.GraphedGenerator(m2, (64, 1, 512, 512), dev)
r2["whole_slice_infer_volume_512_ms"], _ = timed(lambda: inference.infer_volume(m2, slices, batch=64, graphed=g512), reps)
print(json.dumps({
    "metric": "sliding_window_3d_256cube_roi128_ms", "value": res["3d_256cube_roi128_overlap0.25"]["call_ms"],
    "unit": "ms", "card": card, "hbm_peak_gbs": HBM_GBS, "hbm_peak_source": "data sheet (HGX B200, per GPU)",
    "precision": mpgan.DEFAULT_PRECISION, "reps": reps, "cases": res}))
