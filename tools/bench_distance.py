"""Exact distance transform and mask agreement on the device: CUDA-event time per call, written as one JSON line to
the given path (default profiles/bench_distance.json) and printed.

Cases, all with head-shaped masks (``foreground_mask(x, largest_component=True, fill_holes=True)`` of a bright noisy
ellipsoid in a dark noisy field, paired with the same mask shifted by (2, -3, 1) voxels):
  1. one 128^3 pair;
  2. 32 such pairs in one call;
  3. one 256x512x512 pair (67 M voxels: every map exceeds the 126 MB L2).
Operations: ``distance_transform_edt`` of the truth mask and ``mask_agreement`` of the pair (unit spacing, HD95,
connectivity 1).  Each is timed over ``rounds`` windows of about ``seconds``; the median is reported.

Floor: both are bound by memory traffic, so the floor is the bytes per voxel the algorithm cannot avoid over 7.7 TB/s,
the B200's HBM3e bandwidth from the data sheet (at a 1000 W power limit), not a measured rate.  Bytes per voxel of one
image (rank 3), from the passes of csrc/distance.cu:
  distance_transform_edt  41: mask 1 + squared distances 8 (x pass), then read 8 + write 8 per y and z pass
  mask_agreement         101: two erosions 2 x (1 + 1); two transforms of surfaces 2 x 42 (pass 1 reads mask and
                              erosion); the reduction 4 (two masks, two erosions) + 1 (surface code); eight
                              radix-select levels x 1 (surface code); distance reads at surface voxels only, left out
The kernels move more than that (the envelope workspace, the int32 right-neighbour scan); DESIGN.md lists it.
``share_of_floor`` = floor / measured time.  As context, the host time of the scipy oracle on the same masks
(oracle/surface_distance.py: ``agreement`` at 128^3, one ``distance_transform_edt`` at 256x512x512) is reported with
the host's core count; it is not a GPU number.  The card's name and power limit are read in the same run.
usage: python tools/bench_distance.py [out.json] [seconds per window] [rounds]"""
import json
import math
import os
import statistics
import subprocess
import sys
import time

from scipy import ndimage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from mpgan import transforms as T  # noqa: E402
from oracle import surface_distance as osd  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_distance.json")
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 0.2
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
if not torch.cuda.is_available():
    raise SystemExit("bench_distance needs a B200")
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_BYTES_PER_S = 7.7e12
BYTES_PER_VOXEL = {"distance_transform_edt": 41, "mask_agreement": 101}


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


def head_masks(shape):
    """A head mask on the device and the same mask shifted by (2, -3, 1) voxels."""
    grids = torch.meshgrid(*[torch.linspace(-1, 1, s, device=dev) for s in shape[-3:]], indexing="ij")
    inside = sum((q / 0.7) ** 2 for q in grids) < 1
    hi = torch.distributions.Gamma(4.0, 1 / 100.0).sample(shape).to(dev)
    lo = torch.distributions.Gamma(1.0, 1 / 10.0).sample(shape).to(dev)
    truth = T.foreground_mask(torch.where(inside, hi, lo).contiguous(), largest_component=True, fill_holes=True)
    return torch.roll(truth, (2, -3, 1), dims=(-3, -2, -1)).contiguous(), truth


def case(pred, truth, host):
    v = truth.numel()
    res = {"voxels": v, "mask_fraction": float(truth.float().mean())}
    res["distance_transform_edt"] = timed(lambda: T.distance_transform_edt(truth), v, "distance_transform_edt")
    res["mask_agreement"] = timed(lambda: T.mask_agreement(pred, truth), v, "mask_agreement")
    r = T.mask_agreement(pred, truth)
    res["result"] = {k: r[k].reshape(-1)[0].item() for k in osd.KEYS}
    if host:
        p, t = pred.cpu().numpy(), truth.cpu().numpy()
        t0 = time.perf_counter()
        if host == "agreement":
            osd.agreement(p, t)
        else:
            ndimage.distance_transform_edt(~osd.surface(t))
        res[f"scipy_{host}_host_s"] = time.perf_counter() - t0
        res["host_cores"] = os.cpu_count()
    return res


torch.manual_seed(0)
res = {"pair_128cube": case(*head_masks((128, 128, 128)), "agreement"),
       "pair_128cube_batch32": case(*head_masks((32, 128, 128, 128)), None)}
torch.cuda.empty_cache()
res["pair_256x512x512"] = case(*head_masks((256, 512, 512)), "distance_transform_edt")
line = json.dumps({
    "metric": "mask_agreement_ms_pair_256x512x512", "value": res["pair_256x512x512"]["mask_agreement"]["ms"],
    "unit": "ms", "card": card, "hbm_bytes_per_s_floor": HBM_BYTES_PER_S, "seconds_per_window": seconds,
    "rounds": rounds, "cases": res})
print(line)
with open(out_path, "w") as f:
    f.write(line + "\n")
