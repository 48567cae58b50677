"""Linear resampling on the device (mpgan.transforms.resample): CUDA-event time per call after warm-up, one JSON line.

Cases (the native-grid chain of INTEGRATION.md at production sizes):
  1. a 1 mm 256x256x176 oblique T1 -> the 128^3 2 mm reference grid (the step in front of the generator);
  2. 128^3 -> that native grid (the generated T2 back onto the scanner grid);
  3. 256 slices of 512^2 at 0.5 mm -> 256^2 at 1 mm, rotated in plane (the 2-D model's grid).
Next to them, in the same run, ``infer_volume`` of the reference-literal 3-D generator on one 128^3 volume, so
resampling's share of a native-grid inference is stated.  For each case: the time per call over enough calls to fill
about half a second, the algorithmic bytes (input read once, output written once) and the rate they imply, whether the
input fits the 126 MB L2 (repeated calls then read it from there), and the fp64 instruction rate against the data
sheet's, so the record says which of the two bounds the kernel.
usage: python tools/bench_resample.py [seconds per case]"""
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
import mpgan  # noqa: E402
from mpgan import inference  # noqa: E402
from mpgan.transforms import ImageGeometry, reference_grid, resample  # noqa: E402

seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 0.5
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_GBS = 7700.0            # data sheet, HGX B200 per GPU
FP64_OPS = 37e12 / 2        # data sheet, HGX B200 per GPU: 37 TFLOP/s FP64 counting an FMA as 2 -> fp64 instructions/s
L2_MB = 126.0
# DADD + DMUL + DSETP + FRND.F64 per output voxel in resample_linear_kernel's SASS (cuobjdump -sass of this build,
# CUDA 12.9; four voxels per thread): the rank-3 and rank-2 instances
FP64_PER_VOXEL = {3: 74.25, 2: 39.5}


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


def rotation(axis, angle):
    a = np.asarray(axis, dtype=np.float64)
    a /= np.linalg.norm(a)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + math.sin(angle) * k + (1 - math.cos(angle)) * (k @ k)


def centred(size, spacing, direction):
    half = (np.asarray(size, dtype=np.float64) - 1) / 2 * np.asarray(spacing)
    return ImageGeometry(size, spacing, tuple(-(np.asarray(direction) @ half)), direction)


def case(x, source, target):
    ms, calls = timed(lambda: resample(x, source, target))
    out_numel = x.numel() // math.prod(source.shape) * math.prod(target.shape)
    nbytes = 4 * (x.numel() + out_numel)
    ops = out_numel * FP64_PER_VOXEL[source.rank]
    return {"ms": ms, "calls": calls, "input_mb": 4 * x.numel() / 1e6, "output_mb": 4 * out_numel / 1e6,
            "input_l2_resident": 4 * x.numel() / 1e6 < L2_MB, "algorithmic_gbs": nbytes / (ms * 1e-3) / 1e9,
            "frac_hbm_datasheet": nbytes / (ms * 1e-3) / 1e9 / HBM_GBS,
            "fp64_instr_per_s": ops / (ms * 1e-3), "frac_fp64_datasheet": ops / (ms * 1e-3) / FP64_OPS}


g = torch.Generator().manual_seed(0)
torch.manual_seed(0)
native = centred((256, 256, 176), (1.0, 1.0, 1.0), rotation((0.3, -0.5, 0.8), 0.35))
model_grid = reference_grid()
t1 = (torch.rand(native.shape, generator=g) * 1000).to(dev)
t2 = (torch.rand(model_grid.shape, generator=g) * 2 - 1).to(dev)
c = math.cos(0.4)
slices_src = centred((512, 512), (0.5, 0.5), np.array([[c, -math.sin(0.4)], [math.sin(0.4), c]]))
slices = (torch.rand((256, 1) + slices_src.shape, generator=g) * 1000).to(dev)

res = {"native_1mm_256x256x176_to_reference_128cube": case(t1, native, model_grid),
       "reference_128cube_to_native_1mm_256x256x176": case(t2, model_grid, native),
       "slices_256x512x512_0.5mm_to_256x256_1mm_rotated": case(slices, slices_src,
                                                               reference_grid(256, 256.0, rank=2))}
del slices
torch.cuda.empty_cache()
m3 = mpgan.GAN(1, 128, 128, 128).cuda().freeze()
gg = inference.GraphedGenerator(m3, (1, 1, 128, 128, 128), dev)
ms_infer, calls = timed(lambda: inference.infer_volume(m3, t2[None, None], batch=1, graphed=gg))
ms_resample = (res["native_1mm_256x256x176_to_reference_128cube"]["ms"]
               + res["reference_128cube_to_native_1mm_256x256x176"]["ms"])
chain = {"infer_volume_128cube_ms": ms_infer, "calls": calls, "resample_both_ways_ms": ms_resample,
         "resample_share_of_native_grid_inference": ms_resample / (ms_resample + ms_infer)}
print(json.dumps({
    "metric": "resample_native_1mm_to_reference_128cube_ms", "value": res["native_1mm_256x256x176_to_reference_128cube"]["ms"],
    "unit": "ms", "card": card, "hbm_peak_gbs": HBM_GBS, "fp64_peak_instr_per_s": FP64_OPS,
    "peak_source": "data sheet (HGX B200, per GPU)", "precision_generator": mpgan.DEFAULT_PRECISION,
    "cases": res, "native_grid_inference": chain}))
