"""Foreground-masked metrics against their unmasked forms on the device: CUDA-event time per call, written as one JSON
line to the given path (default profiles/bench_masked_metrics.json) and printed.

Cases (those of tools/bench_mutual_info.py and tools/bench_metrics.py):
  1. one display-range 128^3 generated/true pair (0..255 integers, 40 % background);
  2. a batch of 32 such pairs in one call;
  3. a 256x512x512 pair: 537 MB of inputs, so every call reads HBM, not the 126 MB L2.
The mask is ``foreground_mask(truth)`` (Otsu).  For each case and metric (error sums for MAE / MSE / PSNR, SSIM with
the default 7^3 uniform window, MI with bins 100) the unmasked and the masked call are timed in the same run,
alternating, ``rounds`` windows of about ``seconds`` each; the median of each is reported with their ratio.  Otsu's
threshold and the mask it gives (``foreground_mask``) are timed alone.  The mask adds 1 B per voxel to the 8 B (error
sums, SSIM) or 16 B (MI: two passes) per voxel the unmasked calls read.  The card's name and power limit are read in
the same run.
usage: python tools/bench_masked_metrics.py [out.json] [seconds per window] [rounds]"""
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from mpgan import transforms as T  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_masked_metrics.json")
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 0.2
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
if not torch.cuda.is_available():
    raise SystemExit("bench_masked_metrics needs a B200")
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
BINS = 100


def calls_for(fn):
    """Warm up, and the number of calls that fill about ``seconds``."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return max(10, math.ceil(seconds * 1e3 / (e0.elapsed_time(e1) / 5)))


def window(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def compare(plain, masked):
    """Median ms per call of each over ``rounds`` alternating windows, and masked / unmasked."""
    n_p, n_m = calls_for(plain), calls_for(masked)
    tp, tm = [], []
    for _ in range(rounds):
        tp.append(window(plain, n_p))
        tm.append(window(masked, n_m))
    p, m = statistics.median(tp), statistics.median(tm)
    return {"unmasked_ms": p, "masked_ms": m, "ratio": m / p, "unmasked_spread_ms": [min(tp), max(tp)],
            "masked_spread_ms": [min(tm), max(tm)], "calls_per_window": [n_p, n_m]}


def display_pair(shape, g):
    """A display-range pair, moved to the device: gamma-like intensities, 40 % zero background, and a noisy copy, both
    rounded to 0..255 (the post-processing of inference.to_display_range)."""
    v = torch.distributions.Gamma(2.0, 1 / 150.0).sample(shape).to(dev)
    v[torch.rand(shape, generator=g).to(dev) < 0.4] = 0.0
    noisy = v * (1.0 + 0.2 * torch.randn(shape, generator=g).to(dev))
    return tuple(torch.round(255 * (x - x.min()) / (x.max() - x.min())).contiguous() for x in (noisy, v))


def case(a, b):
    m = T.foreground_mask(b)
    res = {"voxels": a.numel(), "mask_fraction": float(m.float().mean())}
    res["error_sums"] = compare(lambda: T.error_sums(a, b), lambda: T.error_sums(a, b, mask=m))
    res["ssim"] = compare(lambda: T.structural_similarity(a, b, data_range=255, spatial_dims=3),
                          lambda: T.structural_similarity(a, b, data_range=255, spatial_dims=3, mask=m))
    res["mutual_information"] = compare(lambda: T.mutual_information(a, b, bins=BINS, spatial_dims=3),
                                        lambda: T.mutual_information(a, b, bins=BINS, spatial_dims=3, mask=m))
    n = calls_for(lambda: T.foreground_mask(b))
    res["otsu_threshold_ms"] = statistics.median(window(lambda: T.otsu_threshold(b), n) for _ in range(rounds))
    res["foreground_mask_ms"] = statistics.median(window(lambda: T.foreground_mask(b), n) for _ in range(rounds))
    return res


g = torch.Generator().manual_seed(0)
torch.manual_seed(0)
res = {}
a, b = display_pair((128, 128, 128), g)
res["display_128cube_pair"] = case(a, b)
a32, b32 = display_pair((32, 128, 128, 128), g)
res["display_128cube_batch32"] = case(a32, b32)
del a32, b32
torch.cuda.empty_cache()
a, b = display_pair((256, 512, 512), g)
res["display_256x512x512_pair"] = case(a, b)
line = json.dumps({
    "metric": "masked_over_unmasked_mutual_information_128cube_batch32",
    "value": res["display_128cube_batch32"]["mutual_information"]["ratio"], "unit": "ratio", "bins": BINS,
    "card": card, "seconds_per_window": seconds, "rounds": rounds, "cases": res})
print(line)
with open(out_path, "w") as f:
    f.write(line + "\n")
