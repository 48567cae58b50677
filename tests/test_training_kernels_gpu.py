"""The non-convolution kernels of the training step, element-wise against fp64, at the edges of their own dispatch.

BatchNorm (csrc/bn.cu register kernels and csrc/bn_stream.cu streaming kernels), Linear, the losses, Adam and the layout
helpers.  Each case runs the ``ops`` entry points on buffers laid out like the conv-engine file's (inputs are channel
slices padded with 1024 and followed by one image of 1024; outputs, statistics and parameter gradients sit inside
sentinel-filled buffers) and compares every stored value with fp64 computed on the operands the kernel received.

Each stage is checked against fp64 recomputed from the kernel's OWN fp32 intermediates (the saved mean / invstd /
scale / shift, the fp64 sums), so the bounds stay a few roundings wide; each intermediate is checked on its own against
fp64 from the raw inputs.  Bounds are derived from the arithmetic (2^-24 per fp32 rounding, u_out for the store):

* statistics (fp64 throughout): P * 2^-52 * sum|x|;
* saved coefficients: one fp32 rounding of the fp64 formula of bn_finalize_kernel / bn_train_coeffs;
* y = act(fma(x, sc, sh)) (+ res): u_out * |ref| + 2^-23 * (|x sc| + |sh|) * max(1, |slope|) (+ 2^-23 * |a + res|);
* backward sums: L * 2^-23 * sum|term|, L the longest fp32 chain of the engine at that shape (``bn_chain``): pixels
  per thread from ``ew_grid`` plus the warp-shuffle levels for bn.cu, 2 * ceil(chunks / CTAs) plus the shuffle levels
  for bn_stream.cu -- never L = P, which at 40 MB would hide a whole 16 KB chunk;
* dx: u_out * |ref| + 12 * 2^-24 * (|sc g act'| + |k2| (|x| + |mean|) + |k3|), which covers both formulations
  (``k2 (x - mean) + k3`` in bn.cu, ``k2 x + kd`` in bn_stream.cu) and the fp32 roundings of k2 / k3 (at most 5 each)
  and of the two fmas.

The activation kink: both engines form z = fma(x, sc, sh) in fp32, a single rounding of the exact value, which never
changes its sign; the branch of act' is therefore decided exactly by z in fp64 and no tolerance is given at the kink.
Exact zeros of z are reached through ``bn_act_apply`` / ``bn_act_bwd`` / ``act_bwd`` with a given scale / shift.

Which engine runs inside one entry point is invisible from Python: each case names the predicates it satisfies (mirrors
of ``bn_stream_ok``, ``vec_ok``, ``ew_grid``, ``stream_smem`` and the ``linear_bwd`` split, checked on the CPU against
hand-computed values), and ``test_forced_engines_in_child_process`` reruns the GPU cases with MPGAN_BN_STREAM_MIN_MB=0
(every qualifying call streams, tiny shapes included) and with MPGAN_BN_STREAM_MIN_MB=1048576 and MPGAN_NO_LINEAR_TC=1
(the register kernels and the CUDA-core Linear at the production-size shapes).
"""
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BF, F32, F64 = torch.bfloat16, torch.float32, torch.float64
U = 2.0 ** -24                          # one fp32 rounding (relative)
U_OUT = {BF: 2.0 ** -8, F32: 2.0 ** -23}
FILL = 1024.0                           # input margins: any read of them is a large error
SENT = -320.0                           # output margins (exact in bf16): must be unchanged after the call
ACT_NONE, ACT_PRELU, ACT_LEAKY, ACT_TANH = 0, 1, 2, 3
ACT_NAMES = {ACT_NONE: "none", ACT_PRELU: "prelu", ACT_LEAKY: "leaky", ACT_TANH: "tanh"}
LEAKY, ALPHA = 0.2, 0.25
CHILD = "MPGAN_TRAIN_KERNELS_CHILD"     # "stream" / "register" in the forced-engine child runs
ENGINE_RUN = os.environ.get(CHILD, "default")
MIN_MB = int(os.environ.get("MPGAN_BN_STREAM_MIN_MB", "2"))
LINEAR_TC = os.environ.get("MPGAN_NO_LINEAR_TC", "0") != "1"
CHUNK = 16384                           # bn_stream.cu kChunkBytes


# ------------------------------------------------------------------------------------------------ the checker
def check_elementwise(got, ref, bound, what, names=None, locate=None):
    """Assert |got - ref| <= bound element-wise; on failure name the worst element (``locate(idx)`` adds the engine's
    chunk / block of it) and the count out of bounds.  Returns the largest |got - ref| / bound."""
    got, ref, bound = got.double(), ref.double(), bound.double()
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    ratio = torch.nan_to_num(ratio, nan=float("inf"))
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if worst > 1.0:
        idx = torch.unravel_index(torch.argmax(ratio), ratio.shape)
        idx = tuple(int(i) for i in idx)
        names = names or (["image"] + [f"p{i}" for i in range(ratio.dim() - 2)] + ["channel"])
        where = ", ".join(f"{k}={v}" for k, v in zip(names, idx))
        msg = f"{what}: |got - ref| / bound = {worst:.3g} at {where}"
        if locate is not None:
            msg += f", {locate(idx)}"
        msg += f" (got {float(got[idx]):.8g}, ref {float(ref[idx]):.8g}, bound {float(bound[idx]):.3g}); " \
               f"{int((ratio > 1).sum())} elements out of bounds"
        raise AssertionError(msg)
    return worst


# ------------------------------------------------------------------------------------------------ dispatch mirrors
def ceil_div(a, b):
    return -(-a // b)


def ew_grid(pixels, cv, blocks_per_sm, pix_per_thread, sms):
    """bn.cu ew_grid: blocks of 256 threads, gridDim * 256 a multiple of cv, at most 512 pixels per thread."""
    total = pixels * cv
    b = ceil_div(total, 256 * pix_per_thread)
    cap = max(sms * blocks_per_sm, ceil_div(total, 256 * 512))
    b = max(min(b, cap), 1)
    mult = cv // math.gcd(cv, 256)
    return ceil_div(b, mult) * mult


def vec_ok(ptr, ld):
    """bn.cu vec_ok (ptr: byte address or None)."""
    return ptr is None or (ptr % 16 == 0 and ld % 8 == 0)


def bn_stream_ok(dtype, in0, in1, out, ld0, ld1, ldo, pixels, C, act, min_mb=MIN_MB):
    if dtype != BF or C % 8 or C > 512:
        return False
    cv = C // 8
    if cv & (cv - 1):
        return False
    if ld0 != C or (in1 is not None and ld1 != C):
        return False
    if out is not None and (ldo < C or ldo % 8):
        return False
    if any(p is not None and p % 16 for p in (in0, in1, out)):
        return False
    if act == ACT_TANH:
        return False
    return pixels * C * 2 >= (min_mb << 20)


def stream_smem(C, nin):
    """bn_stream.cu stream_smem: (dynamic shared-memory bytes, ring stages) within 227 KB."""
    fixed = 128 + 2 * 6 * 8 + 4 * C * 4 + 512 * 16 * 4 + 64 + 256
    s = min((227 * 1024 - fixed) // (nin * CHUNK), 6)
    return fixed + s * nin * CHUNK, s


def stream_launch(pixels, C, nin, sms):
    """bn_stream.cu launch_stream: (grid, stages, chunks per CTA, chunks).  Two stages while a CTA walks <= 16 chunks."""
    nchunks = ceil_div(pixels * C * 2, CHUNK)
    per_cta = ceil_div(nchunks, sms)
    stages = stream_smem(C, nin)[1]
    if per_cta <= 16 and stages > 2:
        stages = 2
    grid = min(nchunks, sms)
    return grid, stages, ceil_div(nchunks, grid), nchunks


def reduce_branch(cv):
    """bn.cu group_reduce_to_global: warp shuffles (cv | 32), shared memory (256 % cv == 0), or per-thread atomics."""
    if cv <= 32 and 32 % cv == 0:
        return "warp"
    if 256 % cv == 0:
        return "block"
    return "global"


def linear_bwd_split(dtype, batch, k, j, aligned=True):
    """linear_loss_optim.cu mpgan_linear_bwd: (dx kernel, dw kernel)."""
    vec = dtype == BF and k % 8 == 0 and aligned and batch <= 65535 and j <= 65535
    if j * k <= 1024 and batch >= 512:
        return ("vec" if vec else "scalar"), "small"
    return ("vec" if vec else "scalar"), ("vec" if vec else "scalar")


def linear_tc_ok(dtype, b, j, k):
    """ops.linear_tc_ok for a contiguous input."""
    return LINEAR_TC and dtype == BF and b % 16 == 0 and b >= 256 and j % 16 == 0 and 16 <= j <= 512 and k % 256 == 0


def bn_chain(engine, mode, P, C, vec, sms):
    """Longest fp32 chain of one per-channel backward sum.  mode: "sums" (bwd_reduce: sum dz, sum dz xhat), "slope"
    (PReLU slope sum, all channels of a thread), "dbias" (bwd_apply column sums, then fp32 atomics)."""
    if engine == "stream":
        grid, _, per_cta, _ = stream_launch(P, C, 2, sms)
        cv = C // 8
        shuf = int(math.log2(32 // cv)) if cv <= 32 else 0
        if mode == "slope":
            return 16 * per_cta + 5            # 2 items x 8 channels per chunk, fp32 warp_sum
        if mode == "sums":
            return 2 * per_cta + shuf
        return 2 * per_cta + shuf + grid + 1   # + one fp32 atomic per CTA and the prior value
    V = 4 if vec else 1
    cv = C // V
    if mode == "dbias":
        grid = ew_grid(P, cv, 6 if vec else 8, 16, sms)
    else:
        grid = ew_grid(P, cv, 6 if vec else 8, 16 if vec else 32, sms)
    pstep = grid * 256 // cv
    ppt = ceil_div(P, pstep)
    if mode == "slope":
        return ppt * V                         # per-thread fp32, fp64 above
    br = reduce_branch(cv)
    shuf = int(math.log2(32 // cv)) if br == "warp" else 0
    if mode == "sums":
        return ppt + shuf
    atomics = grid if br != "global" else pstep
    return ppt + shuf + atomics + 1


# ------------------------------------------------------------------------------------------------ BatchNorm cases
class BnCase:
    """One BatchNorm layer: forward (bn_stats, then bn_train_apply or bn_finalize + bn_act_apply, or the eval-mode
    finalize), bn_act_apply with a given scale / shift that puts exact zeros on z, bn_act_bwd and (LeakyReLU / none)
    act_bwd.  layout: "contig" (ld = C, the streaming engine's input), "slice" (8-channel margins: vector path),
    "odd" (margins 1 / 2: ld % 8 != 0 and a one-element pointer offset, the scalar path).  out: the output's layout."""

    def __init__(self, C, shape, dtype=BF, act=ACT_LEAKY, res=False, layout="slice", out="slice", fused=True,
                 eval_mode=False, alpha_dev=False, ratio=False, seed=0):
        self.C, self.shape, self.dtype, self.act, self.res = C, tuple(shape), dtype, act, res
        self.layout, self.out, self.fused, self.eval, self.alpha_dev, self.ratio = layout, out, fused, eval_mode, alpha_dev, ratio
        self.seed = seed
        self.P = prod(self.shape)
        self.id = (f"C{C}-{'x'.join(map(str, self.shape))}-{'f32' if dtype == F32 else 'bf16'}-{ACT_NAMES[act]}"
                   f"{'_dev' if alpha_dev else ''}{'-res' if res else ''}-in_{layout}-out_{out}"
                   f"{'-eval' if eval_mode else ('-fused' if fused else '-finalize')}{'-mean300' if ratio else ''}")

    # nominal pointers (byte offsets of the views from 512-byte aligned allocations) for the predicates
    def _ptr(self, layout):
        return {"contig": 0, "slice": 8, "odd": 1}[layout] * (2 if self.dtype == BF else 4)

    def _ld(self, layout):
        return {"contig": self.C, "slice": self.C + 16, "odd": self.C + 3}[layout]

    def stream(self, which, min_mb=MIN_MB):
        x, lx, o, lo = self._ptr(self.layout), self._ld(self.layout), self._ptr(self.out), self._ld(self.out)
        if which == "fwd":
            return bn_stream_ok(self.dtype, x, x if self.res else None, o, lx, lx, lo, self.P, self.C, self.act, min_mb)
        if which == "reduce":
            return bn_stream_ok(self.dtype, x, x, None, lx, lx, 0, self.P, self.C, self.act, min_mb)
        return bn_stream_ok(self.dtype, x, x, o, lx, lx, lo, self.P, self.C, self.act, min_mb)

    def vec(self, which):
        ok = self.C % 8 == 0 and vec_ok(self._ptr(self.layout), self._ld(self.layout))
        if which != "reduce":
            ok = ok and vec_ok(self._ptr(self.out), self._ld(self.out))
        return ok

    def predicates(self, min_mb=MIN_MB):
        out = []
        for which in ("fwd", "reduce", "apply"):
            if self.stream(which, min_mb):
                grid, stages, per_cta, nch = stream_launch(self.P, self.C, 1 if which == "fwd" and not self.res else 2, 148)
                out.append(f"{which}:stream(cv={self.C // 8},stages={stages},chunks={nch})")
            else:
                v = self.vec(which)
                V = (8 if which == "fwd" else 4) if v else 1
                br = "" if which == "fwd" else f",{reduce_branch(self.C // V)}"
                out.append(f"{which}:register(V={V}{br})")
        return out


def prod(t):
    r = 1
    for v in t:
        r *= v
    return r


A = [ACT_PRELU, ACT_LEAKY, ACT_NONE, ACT_TANH]
BN_CASES = []
# every channel count of the networks and the odd ones the reduction's branches need, vector and scalar, bf16 and fp32
for i, C in enumerate([1, 3, 8, 16, 24, 32, 48, 64, 96, 128, 256, 512]):
    BN_CASES.append(BnCase(C, (2, 9, 13), BF, A[i % 4], res=i % 2 == 0, layout="slice", out="slice", fused=i % 3 != 0,
                           alpha_dev=i % 4 == 1 and i % 8 == 1, seed=i))
    BN_CASES.append(BnCase(C, (3, 7, 11), F32, A[(i + 1) % 4], res=i % 2 == 1, layout="odd" if i % 2 else "slice",
                           out="odd" if i % 3 == 0 else "slice", fused=i % 2 == 0, seed=100 + i))
    BN_CASES.append(BnCase(C, (1, 9, 13), BF, A[(i + 2) % 4], res=i % 3 == 0, layout="odd", out="slice", seed=200 + i))
BN_CASES += [
    BnCase(2304, (1, 5, 60), BF, ACT_LEAKY, layout="slice", seed=301),               # bn_stats: cv = 288 > 256 lanes
    BnCase(2304, (1, 3, 7), F32, ACT_PRELU, layout="slice", res=True, seed=302),
    # bn_stats blocks of 2048 pixels; ragged against the 2x / 4x-unrolled walks
    BnCase(16, (1, 1, 2047), BF, ACT_PRELU, res=True, seed=303),
    BnCase(16, (1, 1, 2048), BF, ACT_LEAKY, seed=304),
    BnCase(16, (1, 1, 2049), BF, ACT_NONE, res=True, seed=305),
    BnCase(3, (1, 1, 2049), F32, ACT_PRELU, layout="odd", seed=306),
    BnCase(64, (1, 37, 111), BF, ACT_PRELU, res=True, seed=307, ratio=True),
    BnCase(24, (3, 41, 67), BF, ACT_LEAKY, alpha_dev=True, seed=308),                 # V = 4: "global" branch, big grid
    BnCase(32, (3, 40, 64), F32, ACT_TANH, res=True, seed=309, ratio=True),
    # eval mode (running statistics)
    BnCase(16, (2, 9, 13), BF, ACT_PRELU, eval_mode=True, res=True, seed=310),
    BnCase(3, (2, 9, 13), F32, ACT_LEAKY, eval_mode=True, layout="odd", seed=311),
    BnCase(64, (2, 128, 128), BF, ACT_LEAKY, eval_mode=True, layout="contig", out="contig", seed=312),
    # contiguous, below 2 MB: register kernels by default, the streaming engine with MPGAN_BN_STREAM_MIN_MB=0
    BnCase(8, (1, 5, 7), BF, ACT_PRELU, layout="contig", out="contig", seed=313),
    BnCase(64, (1, 1, 2049), BF, ACT_LEAKY, res=True, layout="contig", out="slice", seed=314, ratio=True),
    BnCase(512, (1, 3, 5), BF, ACT_NONE, layout="contig", out="contig", seed=315),
    # streaming sizes: just above 2 MB (partial last chunk), one shape per cv = C / 8, 300:1 channels
    BnCase(64, (1, 1, 16385), BF, ACT_LEAKY, layout="contig", out="contig", seed=320),
    BnCase(8, (2, 400, 331), BF, ACT_PRELU, res=True, layout="contig", out="slice", seed=321, ratio=True),
    BnCase(16, (1, 331, 301), BF, ACT_LEAKY, alpha_dev=True, layout="contig", out="contig", seed=322),
    BnCase(32, (3, 97, 113), BF, ACT_NONE, res=True, layout="contig", out="contig", seed=323),
    BnCase(64, (2, 67, 131), BF, ACT_PRELU, layout="contig", out="slice", seed=324, ratio=True),
    BnCase(128, (1, 83, 103), BF, ACT_LEAKY, res=True, layout="contig", out="contig", seed=325, fused=False),
    BnCase(256, (1, 53, 79), BF, ACT_PRELU, layout="contig", out="slice", seed=326),
    BnCase(512, (1, 31, 67), BF, ACT_LEAKY, res=True, layout="contig", out="contig", seed=327, ratio=True),
    # above ~39 MB a CTA walks > 16 chunks and the ring has 5 (C = 512, two inputs) or 6 stages; nin = 1 forward
    BnCase(512, (1, 1, 40961), BF, ACT_LEAKY, res=True, layout="contig", out="slice", seed=330, ratio=True),
    BnCase(64, (1, 5, 65539), BF, ACT_PRELU, layout="contig", out="contig", seed=331, ratio=True),
]
_ids = [c.id for c in BN_CASES]
assert len(set(_ids)) == len(_ids), "duplicate BatchNorm case ids"


def bn_operands(c):
    g = torch.Generator(device="cpu").manual_seed(1000 + c.seed)

    def r(*shape, scale=1.0):
        return (torch.rand(shape, generator=g, dtype=F64) * 2 - 1) * scale

    n, C = c.shape, c.C
    x = r(*n, C) * 2 + 0.3
    if c.ratio and C > 1:       # |mean| : std = 300 : 1, the un-normalised hand-over between cascaded UNets
        x[..., 1] = 300.0 + r(*n) * math.sqrt(3)
    x = x.to(c.dtype)
    flat = x.view(-1, C)
    flat[::7, 0] = flat[0, 0]   # repeated value: bn_act_apply / bn_act_bwd below put z = 0 exactly there
    d = {"x": x, "dy": r(*n, C).to(c.dtype), "gamma": (r(C) + 1.5).float(), "beta": r(C).float(),
         "rm": r(C).float(), "rv": (r(C).abs() + 0.5).float(), "dg0": r(C).float(), "db0": r(C).float(),
         "dbias0": r(C).float(), "dalpha0": torch.tensor([0.125])}
    if c.res:
        d["res"] = r(*n, C).to(c.dtype)
    return d


def bn_slope(c):
    if c.act == ACT_PRELU:
        return ALPHA
    if c.act == ACT_LEAKY:
        return 0.3 if c.alpha_dev else LEAKY
    return 1.0


def act_ref(z, act, slope):
    if act in (ACT_PRELU, ACT_LEAKY):
        return torch.where(z > 0, z, slope * z)
    if act == ACT_TANH:
        return torch.tanh(z)
    return z


def act_grad_ref(z, act, slope):
    """act'(z) in fp64 and an absolute bound on the kernel's fp32 act' (tanh: 1 - t*t from a tanhf of 2 ulp)."""
    if act in (ACT_PRELU, ACT_LEAKY):
        return torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope)), torch.zeros_like(z)
    if act == ACT_TANH:
        t = torch.tanh(z)
        # |dt| <= 2 ulp(t) + (1 - t^2) 2^-24 |z|; |d(1 - t t)| <= 2 |t| |dt| + 2 roundings
        dt = 4 * U * t.abs() + (1 - t * t) * U * z.abs()
        return 1 - t * t, 2 * t.abs() * dt + 2 * U
    return torch.ones_like(z), torch.zeros_like(z)


# -------- references and bounds of each stage (all tensors fp64 on the caller's device, (P, C) views) --------
def check_stats(stats, x, what):
    x = x.double()
    P = x.shape[0]
    r1 = check_elementwise(stats[: x.shape[1]], x.sum(0), P * 2.0 ** -52 * x.abs().sum(0), what + " stats (sum)",
                           names=["channel"])
    r2 = check_elementwise(stats[x.shape[1]:], (x * x).sum(0), P * 2.0 ** -52 * (x * x).sum(0),
                           what + " stats (sum of squares)", names=["channel"])
    return max(r1, r2)


def coeffs_ref(stats, P, eps):
    """bn_finalize_kernel / bn_train_coeffs in fp64: mean, 1 / sqrt(var + eps) and bounds of their fp32 roundings."""
    C = stats.numel() // 2
    m = stats[:C] / P
    e2 = stats[C:] / P
    var = (e2 - m * m).clamp_min(0)
    eps32 = float(torch.tensor(eps, dtype=F32))
    inv = 1 / torch.sqrt(var + eps32)
    dvar = 4 * 2.0 ** -53 * (e2 + m * m)          # fp64 E[x^2] - mean^2, with or without a contracted fma
    return m, var, inv, U * m.abs(), U * inv + 0.5 * dvar / (var + eps32) * inv + 2.0 ** -50 * inv


def check_saved(saved, stats, P, gamma, beta, eps, what, train=True, rm=None, rv=None):
    """saved (4, C) fp32 = mean, invstd, scale, shift.  scale / shift against fp64 of the kernel's own mean / invstd."""
    mean, inv, sc, sh = (saved[i].double() for i in range(4))
    g, b = gamma.double(), beta.double()
    worst = 0.0
    if train:
        m, _, inv_ref, bm, bi = coeffs_ref(stats, P, eps)
        worst = max(worst, check_elementwise(mean, m, bm, what + " saved mean", names=["channel"]))
        worst = max(worst, check_elementwise(inv, inv_ref, bi, what + " saved invstd", names=["channel"]))
    else:       # evaluation: mean = running_mean; invstd = 1.f / sqrtf(running_var + eps): three roundings
        eps32 = float(torch.tensor(eps, dtype=F32))
        worst = max(worst, check_elementwise(mean, rm.double(), torch.zeros_like(mean), what + " eval mean",
                                             names=["channel"]))
        ref = 1 / torch.sqrt(rv.double() + eps32)
        worst = max(worst, check_elementwise(inv, ref, 3.01 * U * ref, what + " eval invstd", names=["channel"]))
    ref = g * inv
    worst = max(worst, check_elementwise(sc, ref, U * ref.abs(), what + " saved scale", names=["channel"]))
    ref = b - mean * sc
    worst = max(worst, check_elementwise(sh, ref, U * (ref.abs() + (mean * sc).abs()), what + " saved shift",
                                         names=["channel"]))
    return worst


def check_running(rm, rv, rm0, rv0, saved_mean, stats, P, mom, what):
    """running_mean = (1 - mom) rm + mom mean (the kernel's fp32 mean), running_var with the unbiased fp64 variance
    rounded to fp32 once; (1 - mom) is rounded once in fp32, then two products and one sum."""
    mom32 = float(torch.tensor(mom, dtype=F32))
    keep = float(torch.tensor(1.0, dtype=F32) - torch.tensor(mom32, dtype=F32))
    a, b = keep * rm0.double(), mom32 * saved_mean.double()
    w = check_elementwise(rm.double(), a + b, 2 * U * (a.abs() + b.abs()) + U * (a + b).abs(), what + " running_mean",
                          names=["channel"])
    _, var, _, _, _ = coeffs_ref(stats, P, 1e-5)
    unb = var * (P / (P - 1)) if P > 1 else var
    a, b = keep * rv0.double(), mom32 * unb
    return max(w, check_elementwise(rv.double(), a + b, 3 * U * (a.abs() + b.abs()) + U * (a + b).abs() + 2.0 ** -40 * b.abs(),
                                    what + " running_var", names=["channel"]))


def fwd_ref(x, sc, sh, act, slope, res, dtype):
    """y = act(fma(x, sc, sh)) (+ res) in fp64 and its bound."""
    z = x * sc + sh
    a = act_ref(z, act, slope)
    mag = (x * sc).abs() + sh.abs()
    bnd = 2 * U * mag * max(1.0, abs(slope))
    if act == ACT_TANH:
        bnd = 2 * U * mag + 4 * U * a.abs()          # tanhf: 2 ulp, plus the rounding of z through tanh' <= 1
    y = a
    if res is not None:
        y = a + res
        bnd = bnd + 2 * U * (a.abs() + res.abs())
    return y, U_OUT[dtype] * y.abs() + bnd


def bwd_sums_ref(dy, x, mean, inv, sc, sh, act, slope, engine="register"):
    """fp64 sums of dz, dz * xhat and the PReLU slope terms, and the magnitudes their bounds scale with.  bn.cu forms
    xhat = (x - mean) * invstd (relative roundings of xhat); bn_stream.cu forms fma(x, invstd, -mean * invstd), whose
    rounded -mean * invstd errs by 2^-24 |mean invstd| -- the whole difference at a channel with |mean| >> std."""
    z = x * sc + sh
    f, df = act_grad_ref(z, act, slope)
    gz = dy * f
    xh = (x - mean) * inv
    t1 = gz.abs() + dy.abs() * df
    t2 = t1 * (xh.abs() + ((mean * inv).abs() if engine == "stream" else 0))
    s3 = (dy * z.clamp_max(0)).sum() if act == ACT_PRELU else torch.zeros((), dtype=F64, device=x.device)
    return gz.sum(0), (gz * xh).sum(0), s3, t1.sum(0), t2.sum(0), (dy * z.clamp_max(0)).abs().sum()


def engine_locate(engine, P, C, vec, sms, shape, kind="apply"):
    """Where a (pixel, channel) element lives in the engine: its 16 KB chunk and CTA, or its register-kernel block
    (kind "fwd": bn_act_apply's grid, V = 8; "apply": bn_act_bwd_apply's, V = 4)."""
    def loc(idx):
        p, ch = idx[0], idx[1] if len(idx) > 1 else 0
        img = p // prod(shape[1:])
        if engine == "stream":
            grid, _, _, _ = stream_launch(P, C, 2, sms)
            k = (p * C + ch) * 2 // CHUNK
            return f"image {img}, 16 KB chunk {k} of {ceil_div(P * C * 2, CHUNK)} (CTA {k % grid} of {grid})"
        V = (8 if kind == "fwd" else 4) if vec else 1
        cv = C // V
        grid = ew_grid(P, cv, 8, 4, sms) if kind == "fwd" else ew_grid(P, cv, 6 if vec else 8, 16, sms)
        pstep = grid * 256 // cv
        return f"image {img}, block {((p % pstep) * cv + ch // V) // 256} of {grid}"
    return loc


def check_bwd(c, dy, x, mean, inv, sc, sh, sums, dx, dbias, dbias0, engine, vec_r, vec_a, sms, what, dtype):
    """sums[0..2C] (fp64) and dx / dbias of bn_act_bwd against fp64 from the kernel's own coefficients and sums."""
    P, C = x.shape
    slope = bn_slope(c)
    s1, s2, s3, t1, t2, t3 = bwd_sums_ref(dy, x, mean, inv, sc, sh, c.act, slope, engine)
    L = bn_chain(engine, "sums", P, C, vec_r, sms)
    w = check_elementwise(sums[:C], s1, (L + 1) * 2 * U * t1, what + " sum dz", names=["channel"])
    w = max(w, check_elementwise(sums[C:2 * C], s2, (L + 3) * 2 * U * t2, what + " sum dz*xhat", names=["channel"]))
    Ls = bn_chain(engine, "slope", P, C, vec_r, sms)
    w = max(w, check_elementwise(sums[2 * C:], s3.view(1), ((Ls + 2) * 2 * U * t3).view(1), what + " PReLU slope sum",
                                 names=["slot"]))
    # dx from the kernel's own fp64 sums, as the kernels form k2 / k3
    z = x * sc + sh
    f, df = act_grad_ref(z, c.act, slope)
    k2 = -sc * inv * (sums[C:2 * C] / P)
    k3 = -sc * (sums[:C] / P)
    ref = sc * dy * f + k2 * (x - mean) + k3
    mag = (sc * dy * f).abs() + k2.abs() * (x.abs() + mean.abs()) + k3.abs()
    bnd = U_OUT[dtype] * ref.abs() + 12 * U * mag + sc.abs() * dy.abs() * df
    loc = engine_locate(engine, P, C, vec_a, sms, c.shape)
    w = max(w, check_elementwise(dx, ref, bnd, what + " dx", names=["pixel", "channel"], locate=loc))
    Lb = bn_chain(engine, "dbias", P, C, vec_a, sms)
    ref = dbias0 + dx.sum(0)
    w = max(w, check_elementwise(dbias, ref, Lb * 2 * U * (dbias0.abs() + dx.abs().sum(0)), what + " dbias",
                                 names=["channel"]))
    return w


# ------------------------------------------------------------------------------------------------ CPU self-tests
def test_dispatch_mirrors_match_hand_computed_values():
    # ring stages from stream_smem's arithmetic: 5 for C >= 256 with two inputs, 6 otherwise
    assert stream_smem(512, 2)[1] == 5 and stream_smem(256, 2)[1] == 5
    assert stream_smem(128, 2)[1] == 6 and stream_smem(64, 2)[1] == 6 and stream_smem(512, 1)[1] == 6
    assert stream_smem(512, 2)[0] == 41504 + 5 * 2 * CHUNK
    # a CTA walks more than 16 chunks above 148 * 16 * 16 KB = 37 MiB: then the full ring
    assert stream_launch(40961, 512, 2, 148) == (148, 5, 18, 2561)
    assert stream_launch(5 * 65539, 64, 1, 148)[:2] == (148, 6)
    assert stream_launch(16385, 64, 2, 148) == (129, 2, 1, 129)          # 2 MB + one pixel: partial last chunk
    # ew_grid: 2049 pixels of 24 channels on the V = 4 path -> 6 blocks (a multiple of cv / gcd(cv, 256) = 3)
    assert ew_grid(2049, 6, 6, 16, 148) == 6
    assert ew_grid(4_000_000, 16, 6, 16, 148) == 888
    assert ew_grid(10 ** 9, 16, 6, 16, 148) == ceil_div(16 * 10 ** 9, 256 * 512)   # 512 pixels per thread at most
    assert ew_grid(1, 1, 8, 4, 148) == 1
    assert vec_ok(0x1000, 24) and not vec_ok(0x1002, 24) and not vec_ok(0x1000, 20) and vec_ok(None, 3)
    assert bn_stream_ok(BF, 0, None, 0, 64, 0, 64, 16384, 64, ACT_LEAKY, 2)          # exactly 2 MiB
    assert not bn_stream_ok(BF, 0, None, 0, 64, 0, 64, 16383, 64, ACT_LEAKY, 2)
    assert not bn_stream_ok(BF, 0, None, 0, 64, 0, 64, 16384, 64, ACT_TANH, 2)
    assert not bn_stream_ok(BF, 0, None, 0, 24, 0, 24, 10 ** 6, 24, ACT_LEAKY, 2)    # cv = 3
    assert not bn_stream_ok(BF, 0, None, 0, 1024, 0, 1024, 10 ** 6, 1024, ACT_LEAKY, 2)
    assert not bn_stream_ok(F32, 0, None, 0, 64, 0, 64, 10 ** 6, 64, ACT_LEAKY, 2)
    assert not bn_stream_ok(BF, 0, None, 0, 80, 0, 64, 10 ** 6, 64, ACT_LEAKY, 2)    # input slice
    assert bn_stream_ok(BF, 0, None, 16, 64, 0, 80, 10 ** 6, 64, ACT_LEAKY, 2)       # output slice
    assert not bn_stream_ok(BF, 0, None, 2, 64, 0, 80, 10 ** 6, 64, ACT_LEAKY, 2)
    assert bn_stream_ok(BF, 0, None, 0, 64, 0, 64, 1, 64, ACT_LEAKY, 0)
    assert [reduce_branch(v) for v in (1, 2, 4, 8, 16, 32, 64, 128, 256, 3, 6, 12, 24)] == \
        ["warp"] * 6 + ["block"] * 3 + ["global"] * 4
    assert linear_bwd_split(BF, 4, 4096, 8) == ("vec", "vec")
    assert linear_bwd_split(BF, 4, 4100, 8) == ("scalar", "scalar")
    assert linear_bwd_split(BF, 4, 4096, 8, aligned=False) == ("scalar", "scalar")
    assert linear_bwd_split(F32, 4, 4096, 8) == ("scalar", "scalar")
    assert linear_bwd_split(BF, 512, 64, 16) == ("vec", "small")
    assert linear_bwd_split(BF, 511, 64, 16) == ("vec", "vec")
    assert linear_bwd_split(BF, 4096, 1025, 1) == ("scalar", "scalar")
    # chains: bn.cu at 4 M pixels of 64 channels: 282 pixels per thread + 2 shuffle levels; the stream engine at 40 MB
    assert bn_chain("register", "sums", 4_000_000, 64, True, 148) == 282 + 1
    assert bn_chain("stream", "sums", 40961, 512, True, 148) == 2 * 18
    assert bn_chain("stream", "sums", 5 * 65539, 64, True, 148) == 2 * 18 + 2


def test_case_tables_cover_the_dispatch():
    pred = [p for c in BN_CASES for p in c.predicates(2)]
    for cv in (1, 2, 4, 8, 16, 32, 64):
        assert any(f"stream(cv={cv}," in p for p in pred), cv
    assert any("stages=5" in p for p in pred) and any("stages=6" in p for p in pred)
    assert any(p.startswith("fwd:stream") and "stages=6" in p for p in pred)
    for br in ("warp", "block", "global"):
        assert any(f"V=4,{br}" in p for p in pred) and any(f"V=1,{br}" in p for p in pred), br
    assert any("fwd:register(V=8" in p for p in pred) and any("fwd:register(V=1" in p for p in pred)
    # a partial last 16 KB chunk in a streamed case
    assert any(c.stream("apply", 2) and (c.P * c.C * 2) % CHUNK for c in BN_CASES)
    # with MPGAN_BN_STREAM_MIN_MB=0 the small contiguous cases stream too
    assert sum(c.stream("apply", 0) for c in BN_CASES) > sum(c.stream("apply", 2) for c in BN_CASES)


def test_references_agree_with_torch_batchnorm():
    """The fp64 forward / backward formulas against torch.nn.functional.batch_norm + autograd in fp64."""
    c = BnCase(16, (2, 5, 7), F32, ACT_PRELU, res=True)
    d = bn_operands(c)
    x = d["x"].double().view(-1, 16).requires_grad_(True)
    y = F.batch_norm(x, None, None, d["gamma"].double(), d["beta"].double(), training=True, eps=1e-5)
    y = F.prelu(y, torch.tensor([ALPHA], dtype=F64))
    dy = d["dy"].double().view(-1, 16)
    y.backward(dy)
    xd = x.detach()
    stats = torch.cat([xd.sum(0), (xd * xd).sum(0)])
    m, _, inv, _, _ = coeffs_ref(stats, x.shape[0], 1e-5)
    sc = d["gamma"].double() * inv
    sh = d["beta"].double() - m * sc
    yr, _ = fwd_ref(xd, sc, sh, ACT_PRELU, ALPHA, None, F32)
    assert torch.allclose(yr, y.detach(), rtol=1e-6, atol=1e-6)
    s1, s2, *_ = bwd_sums_ref(dy, xd, m, inv, sc, sh, ACT_PRELU, ALPHA)
    P = x.shape[0]
    dx = sc * dy * torch.where(xd * sc + sh > 0, 1.0, ALPHA) - sc * inv * (s2 / P) * (xd - m) - sc * s1 / P
    assert torch.allclose(dx, x.grad, rtol=1e-6, atol=1e-9)


def _model_bwd(c, d, engine="register", sms=148):
    """A correct backward on the CPU: fp32 arithmetic, one rounding per stored value, fp64 sums of fp32 terms."""
    x, dy = d["x"].double().view(-1, c.C), d["dy"].double().view(-1, c.C)
    P = x.shape[0]
    stats = torch.cat([x.sum(0), (x * x).sum(0)])
    m, _, inv, _, _ = coeffs_ref(stats, P, 1e-5)
    mean, inv = m.float().double(), inv.float().double()
    sc = (d["gamma"].double() * inv).float().double()
    sh = (d["beta"].double() - mean * sc).float().double()
    z = (x * sc + sh).float().double()
    slope = bn_slope(c)
    f = torch.where(z > 0, 1.0, slope)
    gz = dy * f
    sums = torch.cat([gz.sum(0), (gz * ((x - mean) * inv).float().double()).sum(0),
                      ((dy * z.clamp_max(0)).sum() if c.act == ACT_PRELU else torch.zeros(())).view(1)])
    k2 = (-sc * inv * (sums[c.C:2 * c.C] / P)).float().double()
    k3 = (-sc * (sums[:c.C] / P)).float().double()
    dx = (sc * gz + k2 * (x - mean) + k3).to(c.dtype).double()
    dbias = d["dbias0"].double() + dx.sum(0)
    return x, dy, mean, inv, sc, sh, sums, dx, dbias


BWD_SELF = BnCase(16, (1, 1, 4099), BF, ACT_PRELU, layout="slice", seed=7)
STREAM_SELF = BnCase(64, (1, 5, 65539), BF, ACT_LEAKY, layout="contig", out="contig", seed=8)


@pytest.mark.parametrize("c", [BWD_SELF, STREAM_SELF, BN_CASES[3], BN_CASES[4], BN_CASES[1]], ids=lambda c: c.id)
def test_checker_accepts_correct_bn_model(c):
    d = bn_operands(c)
    x, dy, mean, inv, sc, sh, sums, dx, dbias = _model_bwd(c, d)
    engine = "stream" if c.stream("reduce", 2) else "register"
    assert check_bwd(c, dy, x, mean, inv, sc, sh, sums, dx, dbias, d["dbias0"].double(), engine, c.vec("reduce"),
                     c.vec("apply"), 148, c.id, c.dtype) <= 1.0
    y, bnd = fwd_ref(x, sc, sh, c.act, bn_slope(c), None, c.dtype)
    model = act_ref((x * sc + sh).float().double(), c.act, bn_slope(c)).to(c.dtype)
    assert check_elementwise(model, y, bnd, c.id + " y", names=["pixel", "channel"]) <= 1.0


def test_checker_rejects_scale_off_by_4_ulp():
    c = next(c for c in BN_CASES if c.C == 16)
    d = bn_operands(c)
    x = d["x"].double().view(-1, c.C)
    stats = torch.cat([x.sum(0), (x * x).sum(0)])
    m, _, inv, _, _ = coeffs_ref(stats, x.shape[0], 1e-5)
    sc = (d["gamma"].double() * inv.float().double()).float()
    saved = torch.stack([m.float(), inv.float(), sc, (d["beta"].double() - m.float().double() * sc.double()).float()])
    assert check_saved(saved, stats, x.shape[0], d["gamma"], d["beta"], 1e-5, c.id) <= 1.0
    bad = saved.clone()
    bad[2, 5] = (bad[2, 5].view(torch.int32) + 4).view(F32)
    with pytest.raises(AssertionError, match="saved scale: .* at channel=5"):
        check_saved(bad, stats, x.shape[0], d["gamma"], d["beta"], 1e-5, c.id)


def test_checker_rejects_residual_missing_on_last_pixel():
    c = BnCase(16, (2, 9, 13), BF, ACT_LEAKY, res=True)
    d = bn_operands(c)
    x, res = d["x"].double().view(-1, 16), d["res"].double().view(-1, 16)
    sc, sh = torch.linspace(0.5, 2, 16, dtype=F64), torch.linspace(-1, 1, 16, dtype=F64)
    y, bnd = fwd_ref(x, sc, sh, c.act, LEAKY, res, BF)
    model = (act_ref((x * sc + sh).float().double(), c.act, LEAKY) + res).to(BF)
    assert check_elementwise(model, y, bnd, "y", names=["pixel", "channel"]) <= 1.0
    model[-1] = act_ref((x[-1] * sc + sh).float().double(), c.act, LEAKY).to(BF)
    with pytest.raises(AssertionError, match=f"pixel={x.shape[0] - 1}, .*block"):
        check_elementwise(model, y, bnd, "y", names=["pixel", "channel"],
                          locate=engine_locate("register", x.shape[0], 16, True, 148, c.shape))


def test_checker_rejects_missing_last_chunk_of_40mb_stream():
    """At 5 x 65 539 pixels of 64 channels (40 MB) the per-CTA chain bound (18 chunks) sees one missing 16 KB chunk."""
    c = STREAM_SELF
    d = bn_operands(c)
    x, dy, mean, inv, sc, sh, sums, dx, dbias = _model_bwd(c, d)
    P = x.shape[0]
    per_chunk = CHUNK // (2 * c.C)
    last = slice((ceil_div(P * c.C * 2, CHUNK) - 1) * per_chunk, P)
    gz = dy[last] * torch.where(x[last] * sc + sh > 0, 1.0, LEAKY)
    bad = sums.clone()
    bad[:c.C] -= gz.sum(0)
    bad[c.C:2 * c.C] -= (gz * (x[last] - mean) * inv).sum(0)
    with pytest.raises(AssertionError, match="sum dz.* at channel="):
        check_bwd(c, dy, x, mean, inv, sc, sh, bad, dx, dbias, d["dbias0"].double(), "stream", True, True, 148, c.id, BF)


def test_checker_rejects_last_cta_partial_missing_from_dbias():
    c = BWD_SELF
    d = bn_operands(c)
    x, dy, mean, inv, sc, sh, sums, dx, dbias = _model_bwd(c, d)
    P, C = x.shape
    cv = C // 4
    grid = ew_grid(P, cv, 6, 16, 148)
    pstep = grid * 256 // cv
    tid = (torch.arange(P).view(-1, 1) % pstep) * cv + torch.arange(C).view(1, -1) // 4
    mine = (tid // 256) == grid - 1
    bad = dbias - (dx * mine).sum(0)
    with pytest.raises(AssertionError, match="dbias: .* at channel="):
        check_bwd(c, dy, x, mean, inv, sc, sh, sums, dx, bad, d["dbias0"].double(), "register", True, True, 148, c.id, BF)


def test_checker_rejects_wrong_side_of_prelu_kink():
    c = BWD_SELF
    d = bn_operands(c)
    x, dy, mean, inv, sc, sh, sums, dx, dbias = _model_bwd(c, d)
    z = x * sc + sh
    y, bnd = fwd_ref(x, sc, sh, ACT_PRELU, ALPHA, None, BF)
    model = act_ref(z.float().double(), ACT_PRELU, ALPHA).to(BF)
    i = int(torch.argmin(z))
    p, ch = i // c.C, i % c.C
    model[p, ch] = z[p, ch].to(BF)            # the identity branch for one negative z
    with pytest.raises(AssertionError, match=f"pixel={p}, channel={ch}, .*block"):
        check_elementwise(model, y, bnd, "y", names=["pixel", "channel"],
                          locate=engine_locate("register", x.shape[0], c.C, True, 148, c.shape))
    bad = dx.clone()
    bad[p, ch] = (sc[ch] * dy[p, ch] + (-sc[ch] * inv[ch] * sums[c.C + ch] / x.shape[0]) * (x[p, ch] - mean[ch])
                  - sc[ch] * sums[ch] / x.shape[0]).to(BF).double()
    with pytest.raises(AssertionError, match=f"dx: .* pixel={p}, channel={ch}"):
        check_bwd(c, dy, x, mean, inv, sc, sh, sums, bad, dbias, d["dbias0"].double(), "register", True, True, 148, c.id, BF)


# ------------------------------------------------------------------------------------------------ Linear / loss / Adam
LIN_FWD = [(3, 4095, 5), (3, 4096, 5), (4, 4097, 8), (2, 3 * 4096 + 1, 6)]


def linear_fwd_chain(k):
    """16 products per thread (fmaf), block_sum (two 5-level warp sums), the bias, one fp32 atomic per 4096-chunk."""
    return 16 + 10 + 1 + ceil_div(k, 4096)


def linear_fwd_ref(x, w, b):
    x, w, b = x.double(), w.double(), b.double()
    return x @ w.t() + b, x.abs() @ w.abs().t() + b.abs()


def _lin_operands(bsz, k, j, dtype, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    r = (lambda *s: (torch.rand(s, generator=g, dtype=F64) * 2 - 1))
    return r(bsz, k).to(dtype), r(j, k).to(dtype), r(j).float(), r(bsz, j).float(), r(j, k).float(), r(j).float()


def test_checker_rejects_wrong_last_partial_k_chunk():
    bsz, k, j = LIN_FWD[3]
    x, w, b, *_ = _lin_operands(bsz, k, j, F32, 5)
    ref, S = linear_fwd_ref(x, w, b)
    bnd = linear_fwd_chain(k) * 2 * U * S
    model = (x.float() @ w.float().t() + b).double()
    assert check_elementwise(model, ref, bnd, "linear_fwd", names=["batch", "j"]) <= 1.0
    bad = model - (x[:, -1:].double() @ w[:, -1:].double().t())          # the last chunk (one element) dropped
    with pytest.raises(AssertionError, match="linear_fwd: .* at batch="):
        check_elementwise(bad, ref, bnd, "linear_fwd", names=["batch", "j"])


def adam_ref_state(step, lr, b1, b2):
    """state[1], state[2] in fp64 from the fp32 lr / betas, as adam_prep_kernel computes them before rounding."""
    lr, b1, b2 = (float(torch.tensor(v, dtype=F32)) for v in (lr, b1, b2))
    return lr / (1 - b1 ** step), math.sqrt(1 - b2 ** step)


def adam_check(p0, g, m0, v0, p, m, v, state, b1, b2, eps, what):
    """One Adam step against fp64 of the kernel's own m / v / state (and of the previous p, m, v)."""
    b1, b2, eps = (float(torch.tensor(t, dtype=F32)) for t in (b1, b2, eps))
    p0, g, m0, v0, p, m, v = (t.double() for t in (p0, g, m0, v0, p, m, v))
    c1, c2 = 1 - b1, 1 - b2                     # exact in fp32 (Sterbenz) for betas in [0.5, 1)
    ref = m0 + (g - m0) * c1
    w = check_elementwise(m, ref, 2 * U * (g - m0).abs() * c1 + U * ref.abs(), what + " m", names=["element"])
    ref = v0 * b2 + c2 * g * g
    w = max(w, check_elementwise(v, ref, 2 * U * (v0 * b2).abs() + 4 * U * c2 * g * g + U * ref.abs(), what + " v",
                                 names=["element"]))
    step, bc2 = float(state[1]), float(state[2])
    q = m / (torch.sqrt(v) / bc2 + eps)
    ref = p0 - step * q
    # sqrt, / bc2, + eps: 3 roundings of the denominator; the quotient, the product and the difference: 3 more
    return max(w, check_elementwise(p, ref, 6.01 * U * (step * q).abs() + U * ref.abs(), what + " p", names=["element"]))


def check_adam_state(state, step, lr, b1, b2, what):
    s1, s2 = adam_ref_state(step, lr, b1, b2)
    assert int(state[0:1].view(torch.int32)) == step, f"{what}: step counter {int(state[0:1].view(torch.int32))} != {step}"
    check_elementwise(state[1:3].double(), torch.tensor([s1, s2], dtype=F64, device=state.device),
                      torch.tensor([U * s1, U * s2], dtype=F64, device=state.device) * 2, what + " bias corrections",
                      names=["state slot"])


def _adam_model(p, g, m, v, step_size, bc2, b1, b2, eps):
    c1, c2 = 1 - torch.tensor(b1, dtype=F32), 1 - torch.tensor(b2, dtype=F32)
    mi = m + (g - m) * c1
    vi = v * torch.tensor(b2, dtype=F32) + c2 * g * g
    pi = p - torch.tensor(step_size, dtype=F32) * (mi / (torch.sqrt(vi) / torch.tensor(bc2, dtype=F32) + eps))
    return pi, mi, vi


def test_checker_rejects_adam_with_t_minus_1_bias_correction():
    lr, b1, b2, eps = 5e-4, 0.5, 0.999, 1e-8
    g = torch.Generator(device="cpu").manual_seed(3)
    p, m, v = torch.rand(300, generator=g), torch.zeros(300), torch.zeros(300)
    for step in range(1, 6):
        gr = torch.rand(300, generator=g) - 0.5
        s1, s2 = adam_ref_state(step, lr, b1, b2)
        state = torch.tensor([0.0, s1, s2])
        state[0:1].view(torch.int32)[0] = step
        pn, mn, vn = _adam_model(p, gr, m, v, float(torch.tensor(s1, dtype=F32)), float(torch.tensor(s2, dtype=F32)), b1, b2, eps)
        check_adam_state(state.float(), step, lr, b1, b2, "adam")
        assert adam_check(p, gr, m, v, pn, mn, vn, state, b1, b2, eps, "adam") <= 1.0
        if step == 3:
            b1s, b2s = adam_ref_state(step - 1, lr, b1, b2)
            bad = torch.tensor([state[0], b1s, b2s]).float()
            bad[0:1].view(torch.int32)[0] = step
            with pytest.raises(AssertionError, match="bias corrections"):
                check_adam_state(bad, step, lr, b1, b2, "adam")
        p, m, v = pn, mn, vn


def l1_grad_ref(a, b, weight, n, gscale, da0, dtype):
    """Bit-exact: g = gscale * (weight / (float)n) in fp32, da = (+-g or 0) (+ prior da) rounded once to the dtype."""
    w = torch.tensor(weight, dtype=F32) / torch.tensor(float(n), dtype=F32)
    gg = (torch.tensor(gscale, dtype=F32) if gscale is not None else torch.tensor(1.0, dtype=F32)) * w
    d = a.float() - b.float()
    v = torch.where(d > 0, gg, torch.where(d < 0, -gg, torch.zeros((), dtype=F32)))
    if da0 is not None:
        v = v + da0.float()
    return v.to(dtype)


def test_checker_rejects_l1_tail_skipped():
    n = 8 * 37 + 7                               # n % V = V - 1 for bf16
    g = torch.Generator(device="cpu").manual_seed(4)
    a, b = (torch.rand(n, generator=g) - 0.5).to(BF), (torch.rand(n, generator=g) - 0.5).to(BF)
    da0 = (torch.rand(n, generator=g) - 0.5).to(BF)
    ref = l1_grad_ref(a, b, 0.7, n, None, da0, BF)
    got = ref.clone()
    got[n - n % 8:] = da0[n - n % 8:]             # the scalar tail never ran
    assert torch.equal(ref, l1_grad_ref(a, b, 0.7, n, None, da0, BF))
    with pytest.raises(AssertionError, match=f"element={n - 1}|element={n - 2}|element={n - 7}"):
        check_elementwise(got, ref, torch.zeros(n, dtype=F64), "l1 gradient", names=["element"])


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture
def routes(monkeypatch):
    """The ``what`` name of every C entry point ``ops`` calls (ops.check is called once per entry point)."""
    from mpgan import ops
    calls = []
    real = ops.check

    def record(rc, what):
        calls.append(what)
        real(rc, what)

    monkeypatch.setattr(ops, "check", record)
    return calls


class Guards:
    """Device buffers whose margins hold a sentinel that the kernels must leave unchanged."""

    def __init__(self):
        self.keep = []

    def vec(self, host, lo=8, hi=8, dtype=None):
        host = host.to(dtype) if dtype is not None else host
        big = torch.full((lo + host.numel() + hi,), SENT, dtype=host.dtype, device="cuda")
        view = big[lo:lo + host.numel()].view(host.shape)
        view.copy_(host.cuda())
        self.keep.append((big, (slice(lo, lo + host.numel()),), "vector"))
        return view

    def act_out(self, shape, C, dtype, layout):
        lo, hi = {"contig": (0, 0), "slice": (8, 8), "odd": (1, 2)}[layout]
        big = torch.full((shape[0] + 1,) + tuple(shape[1:]) + (lo + C + hi,), SENT, dtype=dtype, device="cuda")
        self.keep.append((big, (slice(0, shape[0]),) + (slice(None),) * (len(shape) - 1) + (slice(lo, lo + C),), "act"))
        return big[:shape[0], ..., lo:lo + C]

    def intact(self, what):
        for big, inner, kind in self.keep:
            mask = torch.ones(big.shape, dtype=torch.bool, device=big.device)
            mask[inner] = False
            outside = big[mask]
            assert torch.all(outside == SENT), \
                f"{what}: {int((outside != SENT).sum())} {kind} elements outside the output view were written"


def act_in(host, layout):
    """Input activation: a view in a buffer of FILL with channel margins per layout and one trailing image."""
    lo, hi = {"contig": (0, 0), "slice": (8, 8), "odd": (1, 2)}[layout]
    n, C = host.shape[0], host.shape[-1]
    big = torch.full((n + 1,) + tuple(host.shape[1:-1]) + (lo + C + hi,), FILL, dtype=host.dtype, device="cuda")
    view = big[:n, ..., lo:lo + C]
    view.copy_(host.cuda())
    return view


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def report(family, name, worst):
    print(f"[train-kernel] {ENGINE_RUN} {family} {name} max|err|/bound {worst:.4f}")


def _flat(t):
    return t.reshape(-1, t.shape[-1]).double()


# ------------------------------------------------------------------------------------------------ GPU: BatchNorm
@pytest.mark.gpu
@pytest.mark.parametrize("c", BN_CASES, ids=lambda c: c.id)
def test_batchnorm_elementwise(c, routes):
    from mpgan import ops
    nsm = sms()
    d = bn_operands(c)
    G = Guards()
    C, P, dt = c.C, c.P, c.dtype
    x, dy = act_in(d["x"], c.layout), act_in(d["dy"], c.layout)
    res = act_in(d["res"], c.layout) if c.res else None
    y = G.act_out(c.shape, C, dt, c.out)
    bn = SimpleNamespace(num_features=C, eps=1e-5, momentum=0.1, weight=G.vec(d["gamma"]), bias=G.vec(d["beta"]),
                         running_mean=G.vec(d["rm"]), running_var=G.vec(d["rv"]),
                         num_batches_tracked=G.vec(torch.tensor([7]), dtype=torch.int64))
    stats = G.vec(torch.zeros(2 * C, dtype=F64))
    saved = G.vec(torch.zeros(4, C))
    alpha = G.vec(torch.tensor([ALPHA if c.act == ACT_PRELU else 0.3])) if (c.act == ACT_PRELU or c.alpha_dev) else None
    slope = bn_slope(c)
    # the engine each entry point takes: the mirrors on the actual pointers agree with the case's nominal predicates
    pr = dict(zip(("fwd", "reduce", "apply"), c.predicates(MIN_MB)))
    assert bn_stream_ok(dt, x.data_ptr(), res.data_ptr() if c.res else None, y.data_ptr(), ops.ld(x),
                        ops.ld(res) if c.res else 0, ops.ld(y), P, C, c.act) == c.stream("fwd"), pr
    assert vec_ok(x.data_ptr(), ops.ld(x)) == vec_ok(c._ptr(c.layout), c._ld(c.layout))
    assert vec_ok(y.data_ptr(), ops.ld(y)) == vec_ok(c._ptr(c.out), c._ld(c.out))
    xs = _flat(x.float())
    worst = {}

    # ---- forward
    routes.clear()
    if c.eval:
        ops.bn_finalize(None, P, bn, False, saved[0], saved[1], saved[2], saved[3])
        ops.bn_act_apply(x, saved[2], saved[3], c.act, alpha, LEAKY, res, y)
        torch.cuda.synchronize()
        assert tuple(routes) == ("bn_finalize", "bn_act_apply"), routes
        worst["saved"] = check_saved(saved, None, P, d["gamma"].cuda(), d["beta"].cuda(), 1e-5, c.id, train=False,
                                     rm=d["rm"].cuda(), rv=d["rv"].cuda())
        assert torch.equal(bn.running_mean.cpu(), d["rm"]) and torch.equal(bn.running_var.cpu(), d["rv"])
        assert int(bn.num_batches_tracked) == 7, "eval mode counted a batch"
    else:
        ops.bn_stats(x, stats)
        if c.fused:
            ops.bn_train_apply(x, stats, bn, saved, c.act, alpha, LEAKY, res, y)
        else:
            ops.bn_finalize(stats, P, bn, True, saved[0], saved[1], saved[2], saved[3])
            ops.bn_act_apply(x, saved[2], saved[3], c.act, alpha, LEAKY, res, y)
        torch.cuda.synchronize()
        assert tuple(routes) == (("bn_stats", "bn_train_apply") if c.fused else
                                 ("bn_stats", "bn_finalize", "bn_act_apply")), routes
        worst["stats"] = check_stats(stats.double(), xs, c.id)
        worst["saved"] = check_saved(saved, stats.double(), P, d["gamma"].cuda(), d["beta"].cuda(), 1e-5, c.id)
        worst["running"] = check_running(bn.running_mean, bn.running_var, d["rm"].cuda(), d["rv"].cuda(), saved[0],
                                         stats.double(), P, 0.1, c.id)
        assert int(bn.num_batches_tracked) == 8, f"{c.id}: num_batches_tracked {int(bn.num_batches_tracked)} != 8"
    sc, sh = saved[2].double(), saved[3].double()
    eng_f = "stream" if c.stream("fwd") else "register"
    loc = engine_locate(eng_f, P, C, c.vec("fwd"), nsm, c.shape, "fwd")
    ref, bnd = fwd_ref(xs, sc, sh, c.act, slope, _flat(res.float()) if c.res else None, dt)
    worst["y"] = check_elementwise(_flat(y.float()), ref, bnd, c.id + " y", names=["pixel", "channel"], locate=loc)

    # ---- bn_act_apply with a given scale / shift: z = 0 exactly where channel 0 repeats its first value
    k_sc = saved[2].clone()
    k_sh = saved[3].clone()
    k_sc[0] = 0.5
    k_sh[0] = -0.5 * float(xs[0, 0])
    y2 = G.act_out(c.shape, C, dt, c.out)
    routes.clear()
    ops.bn_act_apply(x, k_sc, k_sh, c.act, alpha, LEAKY, res, y2)
    torch.cuda.synchronize()
    assert tuple(routes) == ("bn_act_apply",)
    assert int((xs[:, 0] * 0.5 - 0.5 * float(xs[0, 0]) == 0).sum()) >= 1
    ref, bnd = fwd_ref(xs, k_sc.double(), k_sh.double(), c.act, slope, _flat(res.float()) if c.res else None, dt)
    worst["y(kink)"] = check_elementwise(_flat(y2.float()), ref, bnd, c.id + " y at z = 0", names=["pixel", "channel"],
                                         locate=loc)

    # ---- backward, with the kinked coefficients so that act' is taken at z = 0 exactly
    sums = G.vec(torch.zeros(2 * C + 1, dtype=F64))
    dg, db, dbias = G.vec(d["dg0"]), G.vec(d["db0"]), G.vec(d["dbias0"])
    da = G.vec(d["dalpha0"]) if c.act == ACT_PRELU else None
    dx = G.act_out(c.shape, C, dt, c.out)
    mean, inv = saved[0].clone(), saved[1].clone()
    routes.clear()
    ops.bn_act_bwd(dy, x, mean, inv, k_sc, k_sh, c.act, alpha, LEAKY, sums, dg, db, da, dx, dbias=dbias)
    torch.cuda.synchronize()
    assert tuple(routes) == ("bn_act_bwd_reduce", "bn_act_bwd_apply"), routes
    eng_b = "stream" if c.stream("reduce") else "register"
    assert c.stream("apply") == c.stream("reduce"), "dx takes the engine of the reduction in every table case"
    sd = sums.double()
    worst["bwd"] = check_bwd(c, _flat(dy.float()), xs, mean.double(), inv.double(), k_sc.double(), k_sh.double(), sd,
                             _flat(dx.float()), dbias.double(), d["dbias0"].cuda().double(),
                             eng_b, c.vec("reduce"), c.vec("apply"), nsm, c.id, dt)
    for name, got, g0, s in (("dbeta", db, d["db0"], sd[:C]),
                             ("dgamma", dg, d["dg0"], sd[C:2 * C])):
        ref = g0.cuda().double() + s
        worst[name] = check_elementwise(got.double(), ref, U * (s.abs() + ref.abs()), c.id + " " + name,
                                        names=["channel"])
    if da is not None:
        ref = d["dalpha0"].cuda().double() + sd[2 * C:]
        worst["dalpha"] = check_elementwise(da.double(), ref, U * (sd[2 * C:].abs() + ref.abs()), c.id + " dalpha",
                                            names=["slot"])

    # ---- act_bwd: dx = dy * act'(z) on a saved pre-activation (exact zeros of z are in it)
    if c.act in (ACT_LEAKY, ACT_NONE) and not c.alpha_dev:
        z = act_in(torch.where(d["x"] == d["x"].view(-1, C)[0, 0], torch.zeros((), dtype=dt), d["x"]), c.layout)
        dx2 = G.act_out(c.shape, C, dt, c.out)
        routes.clear()
        ops.act_bwd(dy, z, c.act, LEAKY, dx2)
        torch.cuda.synchronize()
        assert tuple(routes) == ("act_bwd",)
        zz = _flat(z.float())
        f = torch.where(zz > 0, 1.0, LEAKY if c.act == ACT_LEAKY else 1.0)
        ref = _flat(dy.float()) * f
        worst["act_bwd"] = check_elementwise(_flat(dx2.float()), ref, U_OUT[dt] * ref.abs() + 2 * U * ref.abs(),
                                             c.id + " act_bwd", names=["pixel", "channel"])
    G.intact(c.id)
    report("batchnorm", f"{c.id} [{' '.join(pr.values())}]",
           max(worst.values()))


# ------------------------------------------------------------------------------------------------ GPU: Linear
@pytest.mark.gpu
@pytest.mark.parametrize("bsz,k,j", LIN_FWD)
@pytest.mark.parametrize("dtype", [F32, BF])
def test_linear_fwd_elementwise(bsz, k, j, dtype, routes):
    from mpgan import ops
    x, w, b, *_ = _lin_operands(bsz, k, j, dtype, 11 + k)
    G = Guards()
    y = G.vec(torch.zeros(bsz, j))
    routes.clear()
    ops.linear_fwd(x.cuda(), w.cuda(), b.cuda(), y)
    torch.cuda.synchronize()
    assert tuple(routes) == ("linear_fwd",)
    ref, S = linear_fwd_ref(x.cuda(), w.cuda(), b.cuda())
    worst = check_elementwise(y.double(), ref, linear_fwd_chain(k) * 2 * U * S, f"linear_fwd {bsz}x{k}x{j}",
                              names=["batch", "j"])
    G.intact("linear_fwd")
    report("linear_fwd", f"{bsz}x{k}x{j}-{dtype}", worst)


# batch, K, J, dtype, aligned: vector / scalar dx and dw, linear_dw_small on both sides of batch 512 and J*K 1024
LIN_BWD = [(4, 4096, 8, BF, True), (3, 4100, 5, BF, True), (3, 4096, 5, BF, False), (3, 1000, 7, F32, True),
           (512, 64, 16, BF, True), (511, 64, 16, BF, True), (512, 1025, 1, BF, False), (600, 1024, 1, F32, True),
           (4096, 64, 1, BF, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("bsz,k,j,dtype,aligned", LIN_BWD)
def test_linear_bwd_elementwise(bsz, k, j, dtype, aligned, routes):
    from mpgan import ops
    x, w, _, dy, dw0, db0 = _lin_operands(bsz, k, j, dtype, 21 + k)
    G = Guards()
    off = 0 if aligned else 1
    xb = torch.full((bsz * k + 8,), FILL, dtype=dtype, device="cuda")
    xv = xb[off:off + bsz * k].view(bsz, k)
    xv.copy_(x.cuda())
    wv = w.cuda()
    dyv = dy.cuda()
    dx = G.vec(torch.zeros(bsz, k, dtype=dtype), lo=8 + off)
    dw = G.vec(dw0, lo=8 + (0 if aligned else 1))
    db = G.vec(db0)
    routes.clear()
    ops.linear_bwd(xv, wv, dyv, dx, dw, db)
    torch.cuda.synchronize()
    assert tuple(routes) == ("linear_bwd",)
    split = linear_bwd_split(dtype, bsz, k, j, aligned)
    xd, wd, dyd = xv.double(), wv.double(), dyv.double()
    ref = dyd @ wd
    w1 = check_elementwise(dx.double(), ref, U_OUT[dtype] * ref.abs() + (j + 1) * 2 * U * (dyd.abs() @ wd.abs()),
                           f"linear_bwd dx ({split[0]})", names=["batch", "k"])
    rows = 64 if split[1] == "small" else bsz
    L = rows + ceil_div(bsz, rows) + 1          # fp32 chain per thread, then fp32 atomics per 64-row block (small)
    ref = dw0.cuda().double() + dyd.t() @ xd
    w2 = check_elementwise(dw.double(), ref, L * 2 * U * (dw0.cuda().double().abs() + dyd.abs().t() @ xd.abs()),
                           f"linear_bwd dw ({split[1]})", names=["j", "k"])
    ref = db0.cuda().double() + dyd.sum(0)
    w3 = check_elementwise(db.double(), ref, L * 2 * U * (db0.cuda().double().abs() + dyd.abs().sum(0)),
                           "linear_bwd db", names=["j"])
    G.intact("linear_bwd")
    report("linear_bwd", f"{bsz}x{k}x{j}-{dtype}-{'aligned' if aligned else 'offset'} [{split}]", max(w1, w2, w3))


LIN_TC = [(256, 256, 16), (256, 32768, 512), (1040, 256, 512), (1040, 32768, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("bsz,k,j", LIN_TC)
def test_linear_tc_elementwise(bsz, k, j, routes):
    """linear_tc_fwd / linear_tc_bwd at the linear_tc_ok edges (with MPGAN_NO_LINEAR_TC=1: the CUDA-core Linear)."""
    from mpgan import ops
    x, w, b, dz, dw0, db0 = _lin_operands(bsz, k, j, BF, 31 + k + j)
    xc, wc, bc, dzc = x.cuda(), w.cuda(), b.cuda(), dz.cuda()
    tc = linear_tc_ok(BF, bsz, j, k)
    assert ops.linear_tc_ok(xc, j, k) == tc
    G = Guards()
    routes.clear()
    if tc:
        z = ops.linear_tc_fwd(xc, wc, bc)
        assert tuple(routes) == ("linear_tc_fwd", "cast"), routes
    else:
        z = ops.linear_fwd(xc, wc, bc, torch.zeros(bsz, j, device="cuda"))
        assert tuple(routes) == ("linear_fwd",), routes
    torch.cuda.synchronize()
    ref, S = linear_fwd_ref(xc, wc, bc)
    u = U_OUT[BF] if tc else 0.0                # the tcgen05 path stores z in bf16
    w1 = check_elementwise(z.double(), ref, u * ref.abs() + (k + 1) * 2 * U * S, f"linear z {bsz}x{k}x{j}",
                           names=["batch", "j"])
    dx = G.vec(torch.zeros(bsz, k, dtype=BF))
    dw, db = G.vec(dw0), G.vec(db0)
    routes.clear()
    if tc:
        ops.linear_tc_bwd(xc, wc, dzc, dx, dw, db)
        assert tuple(routes) == ("cast", "weight_transpose", "linear_tc_dx", "linear_tc_dw", "colsum"), routes
        dzd = dz.to(BF).cuda().double()         # dz is rounded to bf16 for the tensor cores
    else:
        ops.linear_bwd(xc, wc, dzc, dx, dw, db)
        assert tuple(routes) == ("linear_bwd",), routes
        dzd = dzc.double()
    torch.cuda.synchronize()
    xd, wd = xc.double(), wc.double()
    ref = dzd @ wd
    w2 = check_elementwise(dx.double(), ref, U_OUT[BF] * ref.abs() + (j + 1) * 2 * U * (dzd.abs() @ wd.abs()),
                           "linear dx", names=["batch", "k"])
    ref = dw0.cuda().double() + dzd.t() @ xd
    w3 = check_elementwise(dw.double(), ref, (bsz + 2) * 2 * U * (dw0.cuda().double().abs() + dzd.abs().t() @ xd.abs()),
                           "linear dw", names=["j", "k"])
    ref = db0.cuda().double() + dzd.sum(0)
    w4 = check_elementwise(db.double(), ref, (bsz + 2) * 2 * U * (db0.cuda().double().abs() + dzd.abs().sum(0)),
                           "linear db", names=["j"])
    G.intact("linear tc")
    report("linear_tc", f"{bsz}x{k}x{j} [{'tcgen05' if tc else 'cuda-core'}]", max(w1, w2, w3, w4))


# ------------------------------------------------------------------------------------------------ GPU: losses
@pytest.mark.gpu
def test_sigmoid_bce_elementwise(routes):
    from mpgan import ops
    z = torch.cat([torch.linspace(-200, 200, 4090), torch.tensor([-88.7, -88.8, 0.0, 88.7, 16.7, 17.0])]).float()
    n = z.numel()
    G = Guards()
    p = G.vec(torch.zeros(n))
    ops.sigmoid_fwd(z.cuda(), p)
    torch.cuda.synchronize()
    zd = z.cuda().double()
    ref = 1 / (1 + torch.exp(-zd))
    # expf 2 ulp, 1 + e and the division one rounding each; below 2^-126 the quotient is subnormal (expf overflows
    # beyond -88.7): an absolute 2^-126
    worst = check_elementwise(p.double(), ref, 6 * U * ref + torch.where(ref < 2.0 ** -126, 2.0 ** -126, 0.0),
                              "sigmoid_fwd", names=["element"])
    assert float(p[0]) == 0.0 and float(p[4089]) == 1.0          # both BCE clamps below are reached
    dp = G.vec(torch.linspace(-3, 3, n))
    dz = G.vec(torch.zeros(n))
    ops.sigmoid_bwd(dp, p, dz)
    torch.cuda.synchronize()
    pd, dpd = p.double(), dp.double()
    ref = dpd * pd * (1 - pd)
    worst = max(worst, check_elementwise(dz.double(), ref, 3 * U * ref.abs() + 2.0 ** -149, "sigmoid_bwd",
                                         names=["element"]))
    for tval in (0.0, float(torch.tensor(0.9, dtype=F32)), 1.0):      # the fp32 target the kernel receives
        for m in (n, 1000, 7):
            pm, t = p[:m], torch.full((m,), tval, device="cuda")
            loss = G.vec(torch.tensor([0.375]))
            ops.bce_fwd(pm, t, 0.75, loss)
            torch.cuda.synchronize()
            pdm = pm.double()
            lp = torch.log(pdm).clamp_min(-100)
            lq = torch.log1p(-pdm).clamp_min(-100)
            term = (tval - 1) * lq - tval * lp
            mag = (abs(tval - 1) * lq.abs() + tval * lp.abs()).sum()
            L = ceil_div(m, 256) + 10 + 4               # per-thread fp32 chain, block_sum, the two logs' roundings
            ref = 0.375 + 0.75 * term.sum() / m
            bnd = L * 2 * U * 0.75 * mag / m + 2 * U * (abs(float(ref)) + 0.375)
            worst = max(worst, check_elementwise(loss.double(), ref.view(1), bnd.view(1), f"bce_fwd t={tval} n={m}",
                                                 names=["slot"]))
            gs = G.vec(torch.tensor([1.5]))
            dpr = G.vec(torch.zeros(m))
            ops.bce_bwd(pm, t, 0.75, gs, dpr)
            torch.cuda.synchronize()
            den = torch.clamp_min(pdm * (1 - pdm), float(torch.tensor(1e-12, dtype=F32)))
            ref = 1.5 * 0.75 / m * (pdm - tval) / den
            # 7 roundings; a subnormal numerator g (p - t) rounds absolutely (2^-149), and the division amplifies it
            bnd = 8 * U * ref.abs() + 2.0 ** -149 / den
            worst = max(worst, check_elementwise(dpr.double(), ref, bnd, f"bce_bwd t={tval} n={m}",
                                                 names=["element"]))
    G.intact("sigmoid / bce")
    report("loss", "sigmoid+bce", worst)


L1_CASES = [(n, dtype, off) for dtype in (F32, BF) for n in (8 * 1000, 8 * 1000 + 1, 8 * 1000 + 7, 4 * 999 + 3, 5)
            for off in (0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,off", L1_CASES)
def test_l1_elementwise(n, dtype, off, routes):
    """l1_fwd, l1_bwd, l1_fwd_bwd (loss only, gradient only, both, accumulate, device gscale, fp64 slot) / LazyL1.
    off = 1: one element past a 16-byte boundary, the scalar fall-back of l1_fwd_bwd."""
    from mpgan import ops
    g = torch.Generator(device="cpu").manual_seed(n + off)
    a = ((torch.rand(n, generator=g) - 0.5) * 4).to(dtype)
    b = ((torch.rand(n, generator=g) - 0.5) * 4).to(dtype)
    b[::5] = a[::5]                                               # d = 0: gradient 0
    da0 = (torch.rand(n, generator=g) - 0.5).to(dtype)
    G = Guards()

    def put(t):
        big = torch.full((n + 16,), FILL, dtype=dtype, device="cuda")
        v = big[8 + off:8 + off + n]
        v.copy_(t.cuda())
        return v

    av, bv = put(a), put(b)
    ad, bd = av.double(), bv.double()
    s = (ad - bd).abs().sum()
    sab = s
    worst = 0.0
    nv = 4 if dtype == F32 else 8
    # loss: fp32 per thread, block_sum, one fp32 atomic per block (<= 148 * 16 blocks), weight / n rounded
    nsm = sms()
    L = ceil_div(n, 256) + 10 + nsm * 16 + 3
    loss = G.vec(torch.tensor([0.5]))
    ops.l1_fwd(av, bv, 0.7, loss)
    torch.cuda.synchronize()
    ref = 0.5 + 0.7 * s / n
    worst = max(worst, check_elementwise(loss.double(), ref.view(1), (L * 2 * U * (0.7 * sab / n + 0.5)).view(1),
                                         "l1_fwd", names=["slot"]))
    for accumulate in (False, True):
        da = G.vec(da0, lo=8 + off)
        ops.l1_bwd(av, bv, 0.7, None, da, accumulate)
        torch.cuda.synchronize()
        ref = l1_grad_ref(av.cpu(), bv.cpu(), 0.7, n, None, da0 if accumulate else None, dtype)
        worst = max(worst, check_elementwise(da.cpu(), ref, torch.zeros(n, dtype=F64), f"l1_bwd acc={accumulate}",
                                             names=["element"]))
    gs = G.vec(torch.tensor([1.25]))
    for loss_kind in (None, F32, F64):
        for grad in ("none", "set", "acc"):
            if loss_kind is None and grad == "none":
                continue
            start = 1e6 if loss_kind == F64 else 0.5
            lt = G.vec(torch.tensor([start], dtype=loss_kind)) if loss_kind is not None else None
            da = G.vec(da0, lo=8 + off) if grad != "none" else None
            routes.clear()
            if grad == "acc" and lt is not None:
                ops.LazyL1(av, bv, 0.7, lt).add_to(da)
            else:
                ops.l1_fwd_bwd(av, bv, 0.7, lt, da, grad == "acc", gscale=gs if grad == "set" else None)
            torch.cuda.synchronize()
            assert tuple(routes) == ("l1_fwd_bwd",)
            what = f"l1_fwd_bwd loss={loss_kind} grad={grad} vec={'yes' if off == 0 else 'no'} n%V={n % nv}"
            if lt is not None:
                ref = start + 0.7 * s / n
                # the fp64 slot: per-block fp32 partials, added in fp64 to a total of 1e6 (2^-52 per block)
                bnd = L * 2 * U * 0.7 * sab / n + (nsm * 8 * 2.0 ** -52 * abs(float(ref)) if loss_kind == F64 else
                                                   L * 2 * U * start)
                worst = max(worst, check_elementwise(lt.double(), ref.view(1), torch.as_tensor(bnd).view(1),
                                                     what + " loss", names=["slot"]))
            if da is not None:
                ref = l1_grad_ref(av.cpu(), bv.cpu(), 0.7, n, 1.25 if grad == "set" else None,
                                  da0 if grad == "acc" else None, dtype)
                worst = max(worst, check_elementwise(da.cpu(), ref, torch.zeros(n, dtype=F64), what + " gradient",
                                                     names=["element"]))
    G.intact("l1")
    report("l1", f"n{n}-{dtype}-off{off}", worst)


@pytest.mark.gpu
@pytest.mark.parametrize("ti,to", [(F32, F32), (F32, BF), (BF, F32), (BF, BF)])
def test_tanh_elementwise(ti, to):
    from mpgan import ops
    n = 3001
    x = torch.cat([torch.linspace(-12, 12, n - 3), torch.tensor([0.0, 1e-20, -1e-30])]).to(ti)
    G = Guards()
    y = G.vec(torch.zeros(n, dtype=to))
    ops.tanh_fwd(x.cuda(), y)
    torch.cuda.synchronize()
    ref = torch.tanh(x.cuda().double())
    worst = check_elementwise(y.double(), ref, U_OUT[to] * ref.abs() + 4 * U * ref.abs(), f"tanh_fwd {ti}->{to}",
                              names=["element"])
    if ti == to:
        dy = torch.linspace(-2, 2, n).to(ti).cuda()
        yv = y.clone()
        dx = G.vec(torch.zeros(n, dtype=ti))
        ops.tanh_bwd(dy, yv, dx)
        torch.cuda.synchronize()
        t, g = yv.double(), dy.double()
        ref = g * (1 - t * t)
        bnd = U_OUT[ti] * ref.abs() + 2 * U * g.abs() * (t * t + (1 - t * t).abs()) + U * ref.abs()
        worst = max(worst, check_elementwise(dx.double(), ref, bnd, f"tanh_bwd {ti}", names=["element"]))
    G.intact("tanh")
    report("tanh", f"{ti}->{to}", worst)


# ------------------------------------------------------------------------------------------------ GPU: Adam
@pytest.mark.gpu
@pytest.mark.parametrize("n", [255, 256, 257, 256 * 40 - 1, 256 * 40 + 1])
def test_adam_elementwise(n, routes):
    from mpgan import ops
    lr, b1, b2, eps = 5e-4, 0.5, 0.999, 1e-8
    g = torch.Generator(device="cpu").manual_seed(n)
    G = Guards()
    p = G.vec(torch.rand(n, generator=g) - 0.5)
    m, v = G.vec(torch.zeros(n)), G.vec(torch.zeros(n))
    state = G.vec(torch.zeros(4))
    shadow = G.vec(torch.zeros(n, dtype=BF))
    scale = torch.logspace(-8, 4, n, dtype=F64).float()            # gradients from 1e-8 to 1e4
    worst = 0.0
    for step in list(range(1, 6)) + [10000]:
        if step == 10000:                                          # a state advanced to step 10^4
            state[0:1].view(torch.int32).fill_(9999)
        gr = ((torch.rand(n, generator=g) - 0.5) * 2 * scale).cuda()
        gr[::17] = 0                                               # g = 0; with v = 0 the denominator is eps
        p0, m0, v0 = p.clone(), m.clone(), v.clone()
        routes.clear()
        ops.adam_step(p, gr, m, v, lr, b1, b2, eps, state, shadow)
        torch.cuda.synchronize()
        assert tuple(routes) == ("adam_step",)
        check_adam_state(state, step, lr, b1, b2, f"adam n={n} step={step}")
        worst = max(worst, adam_check(p0, gr, m0, v0, p, m, v, state, b1, b2, eps, f"adam n={n} step={step}"))
        assert torch.equal(shadow, p.to(BF)), f"adam n={n} step={step}: bf16 shadow is not rn(p)"
    G.intact("adam")
    report("adam", f"n{n}", worst)


# ------------------------------------------------------------------------------------------------ GPU: bit-exact helpers
@pytest.mark.gpu
@pytest.mark.parametrize("ti,to", [(F32, F32), (F32, BF), (BF, F32), (BF, BF)])
@pytest.mark.parametrize("layout", ["slice", "odd"])
def test_add_copy_cast_transpose_permute_bit_exact(ti, to, layout, routes):
    from mpgan import ops
    g = torch.Generator(device="cpu").manual_seed(5)
    C = 24
    a = ((torch.rand(2, 9, 7, C, generator=g) - 0.5) * 8).to(ti)
    b = ((torch.rand(2, 9, 7, C, generator=g) - 0.5) * 8).to(ti)
    G = Guards()
    av, bv = act_in(a, layout), act_in(b, "slice" if layout == "odd" else "contig")
    for with_b in (True, False):
        out = G.act_out(a.shape[:-1], C, to, layout)
        routes.clear()
        ops.add_copy(av, bv if with_b else None, out)
        torch.cuda.synchronize()
        assert tuple(routes) == ("add_copy",)
        ref = ((a.float() + b.float()) if with_b else a.float()).to(to)
        assert torch.equal(out.cpu(), ref), f"add_copy {ti}->{to} {layout} b={with_b}"
    src = a.reshape(-1)
    dst = G.vec(torch.zeros(src.numel(), dtype=to))
    ops.cast(src.cuda(), dst)
    torch.cuda.synchronize()
    assert torch.equal(dst.cpu(), src.to(to))
    cy, taps, cx = 5, 9, 7
    w = a.reshape(-1)[: cy * taps * cx].view(cy, taps, cx)
    wt = G.vec(torch.zeros(cy * taps * cx, dtype=to))
    ops.weight_transpose(w.cuda(), wt, cy, taps, cx)
    torch.cuda.synchronize()
    assert torch.equal(wt.cpu().view(cx, taps, cy), w.permute(2, 1, 0).to(to))
    rows, S = 3, 37
    s = a.reshape(-1)[: rows * C * S]
    d1 = G.vec(torch.zeros(rows * C * S, dtype=to))
    ops.permute_flatten(s.cuda(), d1, rows, C, S, True)
    torch.cuda.synchronize()
    assert torch.equal(d1.cpu().view(rows, S, C), s.view(rows, C, S).permute(0, 2, 1).to(to))
    prior = b.reshape(-1)[: rows * C * S].to(to)
    d2 = G.vec(prior)
    ops.permute_flatten(s.cuda(), d2, rows, C, S, False, accumulate=True)
    torch.cuda.synchronize()
    ref = (s.view(rows, S, C).permute(0, 2, 1).float() + prior.view(rows, C, S).float()).to(to)
    assert torch.equal(d2.cpu().view(rows, C, S), ref)
    G.intact("layout helpers")


@pytest.mark.gpu
def test_weight_transpose_batch_bit_exact():
    from mpgan import ops
    g = torch.Generator(device="cpu").manual_seed(6)
    shapes = [(16, 9, 32), (1, 27, 64), (128, 1, 3), (7, 16, 5)]
    srcs = [(torch.rand(s, generator=g) - 0.5).to(BF).cuda() for s in shapes]
    G = Guards()
    dsts = [G.vec(torch.zeros(prod(s), dtype=BF)) for s in shapes]
    table = torch.tensor([[sv.data_ptr(), dv.data_ptr(), *s] for sv, dv, s in zip(srcs, dsts, shapes)],
                         dtype=torch.int64, device="cuda")
    ops.weight_transpose_batch(table, len(shapes), max(prod(s) for s in shapes))
    torch.cuda.synchronize()
    for sv, dv, s in zip(srcs, dsts, shapes):
        assert torch.equal(dv.view(s[2], s[1], s[0]), sv.permute(2, 1, 0))
    G.intact("weight_transpose_batch")


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [2, 3])
@pytest.mark.parametrize("dtype", [F32, BF])
def test_patches_bit_exact(rank, dtype):
    """patch_gather is a copy; patch_scatter_add sums the covering patches in sample order in fp32 onto a prior dvol."""
    from mpgan import ops
    b, ns, roi, C = 2, 5, 6, 3
    sp = (13, 11) if rank == 2 else (9, 8, 10)
    g = torch.Generator(device="cpu").manual_seed(rank)
    vol = (torch.rand((b,) + sp + (C,), generator=g) - 0.5).to(dtype)
    o = torch.stack([torch.randint(0, s - roi + 1, (b, ns), generator=g) for s in sp], dim=-1)
    o[0, 1] = o[0, 0]                                              # overlapping patches
    od = o.reshape(-1, rank).to(torch.int32).cuda()
    out = ops.patch_gather(vol.cuda(), od, ns, roi)
    torch.cuda.synchronize()
    dp = (torch.rand(out.shape, generator=g) - 0.5).to(dtype)
    dvol0 = (torch.rand(vol.shape, generator=g) - 0.5).to(dtype)
    ref = dvol0.float().clone()
    for bi in range(b):
        for si in range(ns):
            sl = tuple(slice(int(v), int(v) + roi) for v in o[bi, si])
            assert torch.equal(out[bi * ns + si].cpu(), vol[bi][sl])
            ref[bi][sl] += dp[bi * ns + si].float()
    dvol = dvol0.cuda()
    ops.patch_scatter_add(dp.cuda(), od, ns, roi, dvol)
    torch.cuda.synchronize()
    assert torch.equal(dvol.cpu(), ref.to(dtype))
    report("patches", f"rank{rank}-{dtype}", 0.0)


# ------------------------------------------------------------------------------------------------ forced engines
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["stream", "register"])
def test_forced_engines_in_child_process(engine):
    """The GPU cases again with every qualifying BatchNorm call on the streaming engine (MPGAN_BN_STREAM_MIN_MB=0,
    read once per process, hence a child), or with every call on the register kernels and the CUDA-core Linear."""
    if ENGINE_RUN != "default":
        pytest.skip("this is a child run")
    env = dict(os.environ, **{CHILD: engine})
    if engine == "stream":
        env["MPGAN_BN_STREAM_MIN_MB"] = "0"
        sel = "batchnorm"
    else:
        env["MPGAN_BN_STREAM_MIN_MB"] = "1048576"
        env["MPGAN_NO_LINEAR_TC"] = "1"
        sel = "batchnorm or linear"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
        ["-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider", "-rA", "-s"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    lines = [l[l.index("[train-kernel]"):] for l in r.stdout.splitlines() if "[train-kernel]" in l]
    print("\n".join(lines))
    assert r.returncode == 0, f"{engine} run failed:\n" + r.stdout[-6000:] + r.stderr[-3000:]
    assert lines and all(f"[train-kernel] {engine} " in l for l in lines)
    if engine == "stream":
        assert any("fwd:stream" in l and "C8-1x5x7" in l for l in lines), "tiny contiguous case did not stream"
    else:
        assert not any(":stream" in l for l in lines)
