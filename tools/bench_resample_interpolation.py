"""Nearest-neighbour and cubic B-spline resampling on the device: CUDA-event time per call after warm-up, written as
one JSON line to the given path (default profiles/bench_resample_interpolation.json) and printed.

Cases are tools/bench_resample.py's, so the figures sit beside linear resampling's:
  1. a 1 mm 256x256x176 oblique volume -> the 128^3 2 mm reference grid;
  2. 128^3 -> that native grid (the generated T2 back onto the scanner grid, where "bspline" replaces "linear");
  3. 256 slices of 512^2 at 0.5 mm -> 256^2 at 1 mm, rotated in plane.
Per case: ``resample(..., interpolation="nearest")`` on fp32 and on uint8, the coefficient pass
(``mpgan_bspline_coefficients`` on the source) and the B-spline evaluation (``mpgan_resample_bspline`` from those
coefficients), each timed on its own.  Algorithmic bytes: nearest reads the input and writes the output once (element
size each); coefficients read 4 B and write 8 B per source voxel; evaluation reads the 8 B coefficients once and writes
4 B per output voxel.  fp64 operations are counted from the arithmetic include/mpgan.h pins (rounded adds, multiplies,
divisions and floors; compares left out), not from the SASS.  The card's name and power limit are read in the same run.
usage: python tools/bench_resample_interpolation.py [out.json] [seconds per timing]"""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from mpgan import ops  # noqa: E402
from mpgan.transforms import ImageGeometry, reference_grid, resample, resample_map  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_resample_interpolation.json")
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 0.5
if not torch.cuda.is_available():
    raise SystemExit("bench_resample_interpolation needs a B200")
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_GBS = 7700.0            # data sheet, HGX B200 per GPU
FP64_OPS = 37e12 / 2        # data sheet, HGX B200 per GPU: 37 TFLOP/s FP64 counting an FMA as 2 -> fp64 operations/s
L2_MB = 126.0
# fp64 operations per voxel in the pinned arithmetic: continuous index 36 (rank 3) / 16 (rank 2); nearest + 1 add per
# axis; spline weights 16 per axis, then 7 per 4-tap sum (16 + 4 + 1 of them at rank 3, 4 + 1 at rank 2);
# coefficients 5 per voxel per axis (gain, causal multiply-add, anti-causal subtract-multiply)
FP64_PER_VOXEL = {"nearest": {3: 39, 2: 18}, "bspline": {3: 36 + 48 + 7 * 21, 2: 16 + 32 + 7 * 5},
                  "coefficients": {3: 15, 2: 10}}


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


def rates(ms, calls, nbytes, ops_count, input_bytes):
    return {"ms": ms, "calls": calls, "bytes": nbytes, "input_l2_resident": input_bytes / 1e6 < L2_MB,
            "algorithmic_gbs": nbytes / (ms * 1e-3) / 1e9, "frac_hbm_datasheet": nbytes / (ms * 1e-3) / 1e9 / HBM_GBS,
            "fp64_ops_per_s": ops_count / (ms * 1e-3), "frac_fp64_datasheet": ops_count / (ms * 1e-3) / FP64_OPS}


def rotation(axis, angle):
    a = np.asarray(axis, dtype=np.float64)
    a /= np.linalg.norm(a)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + math.sin(angle) * k + (1 - math.cos(angle)) * (k @ k)


def centred(size, spacing, direction):
    half = (np.asarray(size, dtype=np.float64) - 1) / 2 * np.asarray(spacing)
    return ImageGeometry(size, spacing, tuple(-(np.asarray(direction) @ half)), direction)


def case(x, source, target):
    rank = source.rank
    items = x.numel() // math.prod(source.shape)
    n_in, n_out = x.numel(), items * math.prod(target.shape)
    res = {"input_voxels": n_in, "output_voxels": n_out}
    for name, t in (("nearest_float32", x), ("nearest_uint8", x.clamp(0, 255).to(torch.uint8))):
        ms, calls = timed(lambda: resample(t, source, target, interpolation="nearest"))
        e = t.element_size()
        res[name] = rates(ms, calls, e * (n_in + n_out), n_out * FP64_PER_VOXEL["nearest"][rank], e * n_in)
    pad = (1,) * (3 - rank)
    coef = torch.empty(x.shape, dtype=torch.float64, device=dev)
    ms, calls = timed(lambda: ops.bspline_coefficients(x, items, rank, source.size + pad, coef))
    res["bspline_coefficients"] = rates(ms, calls, 12 * n_in, n_in * FP64_PER_VOXEL["coefficients"][rank], 4 * n_in)
    out = torch.empty((items,) + target.shape, dtype=torch.float32, device=dev)
    gmap = resample_map(source, target)
    ms, calls = timed(lambda: ops.resample_bspline(coef, items, rank, source.size + pad, target.size + pad, gmap, 0.0,
                                                   out))
    res["bspline_evaluation"] = rates(ms, calls, 8 * n_in + 4 * n_out, n_out * FP64_PER_VOXEL["bspline"][rank], 8 * n_in)
    ms, calls = timed(lambda: resample(x, source, target, interpolation="bspline"))
    res["bspline_resample_call"] = {"ms": ms, "calls": calls}
    return res


g = torch.Generator().manual_seed(0)
native = centred((256, 256, 176), (1.0, 1.0, 1.0), rotation((0.3, -0.5, 0.8), 0.35))
model_grid = reference_grid()
t1 = (torch.rand(native.shape, generator=g) * 1000).to(dev)
t2 = (torch.rand(model_grid.shape, generator=g) * 255).to(dev)
c = math.cos(0.4)
slices_src = centred((512, 512), (0.5, 0.5), np.array([[c, -math.sin(0.4)], [math.sin(0.4), c]]))
slices = (torch.rand((256, 1) + slices_src.shape, generator=g) * 255).to(dev)

res = {"native_1mm_256x256x176_to_reference_128cube": case(t1, native, model_grid),
       "reference_128cube_to_native_1mm_256x256x176": case(t2, model_grid, native),
       "slices_256x512x512_0.5mm_to_256x256_1mm_rotated": case(slices, slices_src, reference_grid(256, 256.0, rank=2))}
line = json.dumps({
    "metric": "resample_bspline_reference_128cube_to_native_1mm_ms",
    "value": res["reference_128cube_to_native_1mm_256x256x176"]["bspline_resample_call"]["ms"], "unit": "ms",
    "card": card, "hbm_peak_gbs": HBM_GBS, "fp64_peak_ops_per_s": FP64_OPS,
    "peak_source": "data sheet (HGX B200, per GPU)", "seconds_per_timing": seconds, "cases": res})
print(line)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    f.write(line + "\n")
