"""Connected components and binary morphology of masks on the device: CUDA-event time per call, written as one JSON
line to the given path (default profiles/bench_morphology.json) and printed.

Cases:
  1. the Otsu mask of one 128^3 head-like volume (a bright noisy ellipsoid in a dark noisy field);
  2. 32 such masks in one call;
  3. the Otsu mask of one 256x512x512 head-like volume (67 M voxels: the label pipeline's arrays exceed the 126 MB L2);
  4. a 256x512x512 random mask at p = 0.3116, the 6-neighbour site-percolation threshold: millions of components,
     the adversarial case for union-find.
Operations (connectivity 1): ``label``, ``largest_component``, ``fill_holes``, one ``binary_erosion``, and
``foreground_mask`` of the volume without and with the clean-up (largest component, then fill holes).  Each is timed
over ``rounds`` windows of about ``seconds``; the median is reported.

Floor: every operation here is bound by memory traffic (no arithmetic to speak of), so its floor is the bytes per voxel
its passes must stream over 7.7 TB/s, the B200's HBM3e bandwidth from the data sheet (at a 1000 W power limit), not a
measured rate.  Bytes per voxel, from the passes of csrc/morphology.cu:
  label              21: mask 1 + parent 4 (tile pass), parent 4 (flatten), parent 4 (root flags), parent 4 + labels 4
                     (propagation)
  largest_component  18: mask 1 + parent 4, parent 4 (flatten + sizes), parent 4 (best root), parent 4 + out 1
  fill_holes         14: mask 1 + parent 4, parent 4 (flatten + face marks), parent 4 + out 1
  binary_erosion      2: mask 1 + out 1
  foreground_mask    13 (x 4 in each of three passes, mask 1), 45 with the clean-up (13 + 18 + 14)
The face-merge pass touches only tile faces and is left out.  ``share_of_floor`` = floor / measured time.  As context,
the host time of one ``scipy.ndimage.label`` call on the same mask is reported with the host's core count (scipy's
labelling is single-threaded); it is not a GPU number.  The card's name and power limit are read in the same run.
usage: python tools/bench_morphology.py [out.json] [seconds per window] [rounds]"""
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np
from scipy import ndimage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from mpgan import transforms as T  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_morphology.json")
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 0.2
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
if not torch.cuda.is_available():
    raise SystemExit("bench_morphology needs a B200")
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_BYTES_PER_S = 7.7e12
BYTES_PER_VOXEL = {"label": 21, "largest_component": 18, "fill_holes": 14, "binary_erosion": 2, "foreground_mask": 13,
                   "foreground_mask_cleaned": 45}


def calls_for(fn):
    """Warm up, and the number of calls that fill about ``seconds``."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return max(5, math.ceil(seconds * 1e3 / (e0.elapsed_time(e1) / 3)))


def window(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def timed(fn, voxels, name):
    n = calls_for(fn)
    ts = [window(fn, n) for _ in range(rounds)]
    ms = statistics.median(ts)
    floor_ms = voxels * BYTES_PER_VOXEL[name] / HBM_BYTES_PER_S * 1e3
    return {"ms": ms, "spread_ms": [min(ts), max(ts)], "calls_per_window": n, "floor_ms": floor_ms,
            "share_of_floor": floor_ms / ms, "bound": "memory"}


def head(shape, g):
    """A head-like fp32 volume on the device: gamma(4, 100) inside an ellipsoid, gamma(1, 10) outside."""
    grids = torch.meshgrid(*[torch.linspace(-1, 1, s, device=dev) for s in shape[-3:]], indexing="ij")
    inside = sum((q / 0.7) ** 2 for q in grids) < 1
    hi = torch.distributions.Gamma(4.0, 1 / 100.0).sample(shape).to(dev)
    lo = torch.distributions.Gamma(1.0, 1 / 10.0).sample(shape).to(dev)
    return torch.where(inside, hi, lo).contiguous()


def case(m, x=None):
    v = m.numel()
    res = {"voxels": v, "mask_fraction": float(m.float().mean())}
    res["label"] = timed(lambda: T.label(m), v, "label")
    res["components"] = T.label(m)[1].reshape(-1)[:4].tolist()
    res["largest_component"] = timed(lambda: T.largest_component(m), v, "largest_component")
    res["fill_holes"] = timed(lambda: T.fill_holes(m), v, "fill_holes")
    res["binary_erosion"] = timed(lambda: T.binary_erosion(m), v, "binary_erosion")
    if x is not None:
        res["foreground_mask"] = timed(lambda: T.foreground_mask(x), v, "foreground_mask")
        res["foreground_mask_cleaned"] = timed(
            lambda: T.foreground_mask(x, largest_component=True, fill_holes=True), v, "foreground_mask_cleaned")
    if m.dim() == 3:
        host = m.cpu().numpy()
        t0 = time.perf_counter()
        ndimage.label(host)
        res["scipy_label_host_s"] = time.perf_counter() - t0
        res["host_cores"] = os.cpu_count()
    return res


torch.manual_seed(0)
g = torch.Generator().manual_seed(0)
res = {}
x = head((128, 128, 128), g)
res["head_128cube"] = case(T.foreground_mask(x), x)
x = head((32, 128, 128, 128), g)
res["head_128cube_batch32"] = case(T.foreground_mask(x), x)
del x
torch.cuda.empty_cache()
x = head((256, 512, 512), g)
res["head_256x512x512"] = case(T.foreground_mask(x), x)
del x
torch.cuda.empty_cache()
r = torch.from_numpy(np.random.RandomState(1).rand(256, 512, 512) < 0.3116).to(dev)
res["percolation_256x512x512_p0.3116"] = case(r)
line = json.dumps({
    "metric": "label_ms_head_256x512x512", "value": res["head_256x512x512"]["label"]["ms"], "unit": "ms",
    "card": card, "hbm_bytes_per_s_floor": HBM_BYTES_PER_S, "seconds_per_window": seconds, "rounds": rounds,
    "cases": res})
print(line)
with open(out_path, "w") as f:
    f.write(line + "\n")
