"""SSIM / PSNR on the device (mpgan.transforms.structural_similarity / peak_signal_noise_ratio): CUDA-event times after
warm-up, one JSON line.  Cases: BASELINE config 5's 256 x 512 x 512 volume (536 MB of fp32 inputs, more than L2) with the
uniform 7-tap and the Gaussian 11-tap window; the reference's literal 128^3 volume (L2-resident after the first pass);
the 256 per-slice 2-D SSIMs of the same 512^2 stack in one call; PSNR of the large volume; the fp64 numpy/scipy
oracle's host time on the 128^3 volume.
usage: python tools/bench_metrics.py [reps]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cross-modality-minipig-gan_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402
from mpgan import transforms as T  # noqa: E402
from oracle import metrics as om  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
if os.path.exists(peaks_path):
    hbm_gbs, hbm_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json"
else:
    hbm_gbs, hbm_src = 7700.0, "data sheet (HGX B200, per GPU)"
FP64_TFLOPS = 37.0   # data sheet, HGX B200 per GPU, dense FP64


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


def fp64_flop(shape, rank, win):
    """fp64 operations ssim_sums_kernel issues (FMA = 2): the w pass over the halo rows of each tile (products formed
    per tap: 10 per tap), the h and d passes (5 FMA per tap each) and ~20 for S, per interior voxel.  The tile height
    follows the host's shared-memory choice."""
    wd = win if rank == 3 else 1
    g = 8
    while g > 1 and (wd * 5 * 2 * 32 * g * 8 + 5 * (2 * g + win - 1) * 32 * 8 + 2 * (2 * g + win - 1) * (31 + win) * 4
                     > 226 * 1024):
        g //= 2
    th = 2 * g
    vox = 1
    for s in shape[len(shape) - rank:]:
        vox *= s - win + 1
    items = 1
    for s in shape[:len(shape) - rank]:
        items *= s
    per_vox = 10 * win * (th + win - 1) / th + 10 * win + 10 * wd + 20
    return items * vox * per_vox


def case(name, a, b, rank, **kw):
    ms, v = timed(lambda: T.structural_similarity(a, b, data_range=255.0, spatial_dims=rank, **kw), reps)
    win = 2 * int(3.5 * 1.5 + 0.5) + 1 if kw.get("gaussian_weights") else 7
    gbs = 2 * 4 * a.numel() / (ms * 1e-3) / 1e9
    fl = fp64_flop(tuple(a.shape), rank, win)
    return name, {"ms": ms, "mssim_mean": float(v.mean()), "gbs": gbs, "frac_hbm": gbs / hbm_gbs,
                  "fp64_tflops": fl / (ms * 1e-3) / 1e12, "frac_fp64_datasheet": fl / (ms * 1e-3) / 1e12 / FP64_TFLOPS}


g = torch.Generator().manual_seed(0)
truth = torch.round(torch.rand((256, 512, 512), generator=g) * 255).to(dev)
gen = torch.clamp(truth + torch.round(torch.randn((256, 512, 512), generator=g).to(dev) * 12), 0, 255)
t128, g128 = truth[:128, :128, :128].contiguous(), gen[:128, :128, :128].contiguous()
res = dict([
    case("vol_256x512x512_uniform7", gen, truth, 3),
    case("vol_256x512x512_gaussian11", gen, truth, 3, gaussian_weights=True),
    case("cube_128_uniform7_l2_resident", g128, t128, 3),
    case("cube_128_gaussian11_l2_resident", g128, t128, 3, gaussian_weights=True),
    case("slices_256x512x512_2d_uniform7", gen, truth, 2),
    case("slices_256x512x512_2d_gaussian11", gen, truth, 2, gaussian_weights=True),
])
ms_psnr, psnr = timed(lambda: T.peak_signal_noise_ratio(truth, gen, data_range=255.0), reps)
a_np, b_np = g128.cpu().double().numpy(), t128.cpu().double().numpy()
t0 = time.perf_counter()
ref = om.structural_similarity(a_np, b_np, data_range=255.0)
host_s = time.perf_counter() - t0
print(json.dumps({
    "metric": "ssim_ms_256x512x512_uniform7", "value": res["vol_256x512x512_uniform7"]["ms"], "unit": "ms",
    "card": card, "hbm_peak_gbs": hbm_gbs, "hbm_peak_source": hbm_src, "fp64_peak_tflops": FP64_TFLOPS,
    "fp64_peak_source": "data sheet (HGX B200, per GPU, dense)", "reps": reps,
    "cases": res,
    "psnr_ms_256x512x512": ms_psnr, "psnr_gbs": 2 * 4 * truth.numel() / (ms_psnr * 1e-3) / 1e9, "psnr_db": psnr,
    "oracle_host_s_128_uniform7": host_s,
    "cube_128_uniform7_abs_diff_vs_oracle": abs(res["cube_128_uniform7_l2_resident"]["mssim_mean"] - ref),
}))
