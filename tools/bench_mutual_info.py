"""Mutual information on the device (mpgan.transforms.mutual_information, bins 100): CUDA-event time per call after
warm-up, written as one JSON line to the given path (default profiles/bench_mutual_info.json) and printed.

Cases:
  1. one display-range 128^3 generated/true pair (0..255 integers, 40 % background);
  2. a batch of 32 such pairs in one call, the shape of the reference's 438-volume evaluation (code/eval/*.xml);
  3. a 256x512x512 pair (BASELINE config 5's volume): 537 MB of inputs, so every call reads HBM, not the 126 MB L2;
  4. an all-background 128^3 pair (every voxel in one joint bin): the worst case for histogram contention.
A call is three kernels (min/max pass, histogram pass, entropies), so each input byte is read twice.  For each case:
the time per call over about ``seconds`` of calls, bytes moved = 2 passes x 2 images x 4 B per voxel, the rate they
imply and its share of the data sheet's 7.7 TB/s, and whether the inputs fit the L2 (repeated calls then read them
from there).  The card's name and power limit are read in the same run.
usage: python tools/bench_mutual_info.py [out.json] [seconds per case]"""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from mpgan import transforms as T  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_mutual_info.json")
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 0.5
if not torch.cuda.is_available():
    raise SystemExit("bench_mutual_info needs a B200")
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_GBS = 7700.0            # data sheet, HGX B200 per GPU
L2_MB = 126.0
BINS = 100


def timed(fn):
    """ms per call: warm up, size the window to about ``seconds``, time it with CUDA events."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(10, math.ceil(seconds * 1e3 / (e0.elapsed_time(e1) / 5)))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def display_pair(shape, g):
    """A display-range pair, moved to the device: gamma-like intensities, 40 % zero background, and a noisy copy, both
    rounded to 0..255 (the post-processing of inference.to_display_range)."""
    v = torch.distributions.Gamma(2.0, 1 / 150.0).sample(shape).to(dev)
    v[torch.rand(shape, generator=g).to(dev) < 0.4] = 0.0
    noisy = v * (1.0 + 0.2 * torch.randn(shape, generator=g).to(dev))
    return tuple(torch.round(255 * (x - x.min()) / (x.max() - x.min())).contiguous() for x in (noisy, v))


def case(a, b):
    ms, calls = timed(lambda: T.mutual_information(a, b, bins=BINS, spatial_dims=3))
    nbytes = 2 * 2 * 4 * a.numel()
    return {"ms": ms, "calls": calls, "voxels": a.numel(), "input_mb": 2 * 4 * a.numel() / 1e6,
            "input_l2_resident": 2 * 4 * a.numel() / 1e6 < L2_MB, "bytes_moved": nbytes,
            "algorithmic_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_hbm_datasheet": nbytes / (ms * 1e-3) / 1e9 / HBM_GBS}


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
del a, b
torch.cuda.empty_cache()
z = torch.zeros((128, 128, 128), device=dev)
res["all_background_128cube_pair"] = case(z, z.clone())
line = json.dumps({
    "metric": "mutual_information_display_128cube_batch32_ms", "value": res["display_128cube_batch32"]["ms"],
    "unit": "ms", "bins": BINS, "card": card, "hbm_peak_gbs": HBM_GBS, "peak_source": "data sheet (HGX B200, per GPU)",
    "cases": res})
print(line)
with open(out_path, "w") as f:
    f.write(line + "\n")
