"""Rigid registration by Mattes mutual information on the device: CUDA-event time per ``register_rigid`` call after a
warm-up call, written as one JSON line to the given path (default profiles/bench_registration.json) and printed.

Cases (phantom T1 / T2 heads of oracle/registration.py, a 10 degree / 10 mm offset, the default pyramid (4, 2, 1),
sigmas (2, 1, 0), 100 iterations, 50 bins, the T1's > 0.05 mask):
  1. one 128^3 2 mm pair;
  2. 8 such pairs in one call;
  3. one 256x256x176 1 mm pair;
  4. per iteration at full resolution (shrink 1) of the 128^3 pair: pass 1 (histogram and -MI:
     ``mpgan_mattes_evaluate`` without the gradient) and pass 1 + pass 2 (with it); pass 2 is their difference.
Bytes are the least the passes must move from memory, per evaluation: the fixed samples (4 B) and the mask (1 B) of
every fixed voxel read, the moving image (4 B per voxel) and, for pass 2, its gradient (12 B per voxel), each once.
The share of the HBM bound is those bytes over the data sheet's 7.7 TB/s, over the measured time; the working sets of
these cases fit the 126 MB L2 except the 1 mm case's, so most of it is served from L2 and the share only says how far
the passes are from streaming their inputs once.  Whole calls also include the smoothing, range and step kernels.
The card's name and power limit are read in the same run.
usage: python tools/bench_registration.py [out.json]"""
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
from mpgan.transforms import ImageGeometry, _registration_plan, grid_center, register_rigid  # noqa: E402
from oracle import registration as orr  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bench_registration.json")
if not torch.cuda.is_available():
    raise SystemExit("bench_registration needs a B200")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
HBM_GBS = 7700.0   # data sheet, HGX B200 per GPU


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def pair(size, spacing, items):
    g = ImageGeometry(size, (spacing,) * 3, tuple(-n * spacing / 2 for n in size))
    c = grid_center(g)
    true = np.array([math.radians(6), math.radians(-5), math.radians(5), 6.0, -5.0, 6.0])
    f = torch.from_numpy(orr.phantom(g, "t1", edge_mm=1.5 * spacing)).cuda()
    m = torch.from_numpy(orr.phantom(g, "t2", true, c, edge_mm=1.5 * spacing)).cuda()
    f, m = f.expand((items,) + f.shape).contiguous(), m.expand((items,) + m.shape).contiguous()
    return g, f, m, f > 0.05


cases = {}
for name, size, spacing, items in (("pair_128cube_2mm", (128,) * 3, 2.0, 1), ("8_pairs_128cube_2mm", (128,) * 3, 2.0, 8),
                                   ("pair_256x256x176_1mm", (256, 256, 176), 1.0, 1)):
    g, f, m, mask = pair(size, spacing, items)
    tf = register_rigid(f, m, g, g, fixed_mask=mask)
    ms = timed(lambda: register_rigid(f, m, g, g, fixed_mask=mask), 3)
    # bytes of the metric passes if every level ran all 100 iterations (an item that stops early skips its passes, so
    # this bounds the call's bytes from above and its share of the HBM bound is an upper bound too)
    plan = _registration_plan(g, g, (4, 2, 1), (2.0, 1.0, 0.0), "geometry")
    nbytes = 0
    for lvl in plan["levels"]:
        s = lvl["shrink"]
        nfs = math.prod(math.ceil(n / s) for n in size)
        nm = math.prod(size)
        nbytes += 100 * items * (2 * (5 * nfs) + 2 * 4 * nm + 12 * nm)
    cases[name] = {"items": items, "ms": ms, "ms_per_pair": ms / items, "status": tf.status.cpu().tolist(),
                   "metric": tf.metric.cpu().tolist(), "bytes_metric_passes_all_iterations": nbytes,
                   "frac_hbm_datasheet": nbytes / (ms * 1e-3) / (HBM_GBS * 1e9)}

g, f, m, mask = pair((128,) * 3, 2.0, 1)
fsize = msize = tuple(g.size)
plan = _registration_plan(g, g, (1,), (0.0,), "geometry")
state = torch.empty(1, 96, dtype=torch.float64, device="cuda")
status = torch.empty(1, dtype=torch.int32, device="cuda")
hist = torch.empty(1, 50, 50, dtype=torch.int64, device="cuda")
metric = torch.empty(1, dtype=torch.float64, device="cuda")
ws = ops.mattes_workspace(1, fsize, msize, 50, "cuda")
mk = mask.view(torch.uint8)
ops.rigid_level(state, status, 1, 3, plan["base"], plan["center"], None, plan["t0"], True, 1.0)
ops.mattes_prepare(f, m, mk, 1, 3, fsize, msize, 1, 50, plan["base"][3:12], plan["min_scale"], state, status,
                   ws)
p1 = timed(lambda: ops.mattes_evaluate(f, m, mk, 1, 3, fsize, msize, 1, 50, False, True, state, status, hist, metric,
                                       ws), 200)
p12 = timed(lambda: ops.mattes_evaluate(f, m, mk, 1, 3, fsize, msize, 1, 50, True, True, state, status, hist, metric,
                                        ws), 200)
nf = math.prod(g.size)
b1, b2 = 5 * nf + 4 * nf, 5 * nf + 4 * nf + 12 * nf
cases["iteration_128cube_full_resolution"] = {
    "samples_in_mask": int(mask.sum()), "pass1_ms": p1, "pass1_bytes": b1,
    "pass1_frac_hbm_datasheet": b1 / (p1 * 1e-3) / (HBM_GBS * 1e9), "pass2_ms": p12 - p1, "pass2_bytes": b2,
    "pass2_frac_hbm_datasheet": b2 / ((p12 - p1) * 1e-3) / (HBM_GBS * 1e9), "pass1_plus_pass2_ms": p12}

res = {"metric": "register_rigid_128cube_2mm_pair_ms", "value": cases["pair_128cube_2mm"]["ms"], "unit": "ms",
       "card": card, "hbm_peak_gbs": HBM_GBS, "peak_source": "data sheet (HGX B200, per GPU)", "cases": cases}
line = json.dumps(res)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as fh:
    fh.write(line + "\n")
print(line)
