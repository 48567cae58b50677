"""The generator's inference path, element-wise against fp64: the BatchNorm fold, the fused eval-mode layers and the
fused UNet tail, plus a captured generator graph that must follow its weights.

* ``Runtime.folded``: bf16 weights ``w32 * gamma / sqrt(running_var + eps)`` along the layer's output axis (the cx axis
  of a ConvTranspose, transposed to [cx][taps][cy]) and an fp32 bias.  The weights are checked bit for bit against the
  same fp32 arithmetic; the bias within a few fp32 roundings of fp64; the fused layer against the module's eval-mode
  definition ``prelu(bn_eval(conv(x, w32) + b)) (+ res)`` in fp64, within the kernel's bound plus one bf16 rounding of
  the folded weights, ``2^-8 * sum|w scale x|``.
* ``c1_conv_act`` (conv_c1_fast.cu fprop_run_kernel with a slope) and ``tc_conv_act`` (the tap-GEMM / halo epilogues):
  ``u_out |ref| + K 2^-23 S max(1, |slope|) + 2^-24 |slope acc|``, K the taps times reduced channels plus the bias
  (and the residual), S the same sum over |operands|.
* ``c1_tail_fwd_kernel`` (bn.cu): ``z = fmaf(c, sc, sh)`` is one rounding of the exact value, so the PReLU branch is
  decided exactly by z in fp64 and no tolerance is given at the kink; h is rounded to bf16 after the slope multiply
  (``2^-8 |h| + 2^-23 |z| max(1, |slope|)``); the conv is a 10-term fp32 chain (bias + 9 fmas) rounded to bf16 before
  the residual add and rounded again (``2^-8 |y| + 2^-8 |a| + 10 2^-23 S``), checked against fp64 of the STORED h.
  The saved mean / invstd / scale / shift and the running statistics are checked against fp64 of the statistics.
* ``c1_tail_bwd_reduce_kernel``: dh has the same two bf16 roundings (9-term chain); the three sums are checked against
  fp64 over the kernel's own stored dh with ``(L + 3) 2^-23 sum|term|``, L the longest per-thread fp32 chain: runs per
  thread (from a mirror of the launch with the device's SM count) times the run length -- never L = P, which would hide
  a missing CTA at production size.  ``bn_act_bwd_apply`` with C = 1 is checked from the kernel's own sums.

Inputs sit in buffers padded with 1024 (a read outside the operand is a large error), outputs and every statistic in
sentinel-filled buffers whose margins are asserted after each call.  ``routes`` records the ``ops`` entry points of each
case.  ``test_unfused_routes_in_child_process`` re-runs the GPU cases with MPGAN_NO_EVAL_FUSION, MPGAN_NO_TAIL_FUSION
and MPGAN_NO_C1ACT set: ``ops.conv_act`` then declines the one-channel layers, the generator runs BatchNorm apply +
convolution + add, and the same fp64 references and bounds apply.
"""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BF, F32, F64 = torch.bfloat16, torch.float32, torch.float64
U = 2.0 ** -24                          # one fp32 rounding (relative)
U_ACC = 2.0 ** -23                      # per term of an fp32 chain
U_OUT = {BF: 2.0 ** -8, F32: 2.0 ** -23}
FILL = 1024.0                           # input margins: any read of them is a large error
SENT = -320.0                           # output margins (exact in bf16): must be unchanged after the call
ACT_PRELU = 1
MOM, EPS = 0.1, 1e-5
SWITCHES = ("MPGAN_NO_EVAL_FUSION", "MPGAN_NO_TAIL_FUSION", "MPGAN_NO_C1ACT")
CHILD = "MPGAN_INFERENCE_KERNELS_CHILD"
FALLBACK = os.environ.get(CHILD) == "1"
KTHREADS = 256


# ------------------------------------------------------------------------------------------------ the checker
def check_elementwise(got, ref, bound, what, names=None, locate=None):
    """Assert |got - ref| <= bound element-wise; on failure name the worst element (``locate(idx)`` adds the run / tile /
    CTA that owns it) and the count out of bounds.  Returns the largest |got - ref| / bound."""
    got, ref, bound = got.double(), ref.double(), bound.double()
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    ratio = torch.nan_to_num(ratio, nan=float("inf"))
    worst = float(ratio.max()) if ratio.numel() else 0.0
    if worst > 1.0:
        idx = tuple(int(i) for i in torch.unravel_index(torch.argmax(ratio), ratio.shape))
        names = names or (["image"] + [f"p{i}" for i in range(ratio.dim() - 2)] + ["channel"])
        msg = f"{what}: |got - ref| / bound = {worst:.3g} at " + ", ".join(f"{k}={v}" for k, v in zip(names, idx))
        if locate is not None:
            msg += f", {locate(idx)}"
        msg += f" (got {float(got[idx]):.8g}, ref {float(ref[idx]):.8g}, bound {float(bound[idx]):.3g}); " \
               f"{int((ratio > 1).sum())} elements out of bounds"
        raise AssertionError(msg)
    return worst


def ceil_div(a, b):
    return -(-a // b)


def prod(t):
    r = 1
    for v in t:
        r *= v
    return r


def report(family, name, worst):
    print(f"[inference-kernel] {'unfused' if FALLBACK else 'default'} {family} {name} max|err|/bound {worst:.4f}")


def _rnd(shape, seed, dtype, scale=1.0, lo=-1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return ((torch.rand(shape, generator=g, dtype=F64) * (1 - lo) + lo) * scale).to(dtype)


# ------------------------------------------------------------------------------------------------ dispatch mirrors
def tail_fwd_launch(n, H, W, aligned, sms):
    """bn.cu mpgan_c1_tail_fwd: (RUN, runs, blocks, runs per thread).  RUN 8 when W % 8 == 0 and c, y, h are 16-byte
    aligned; ceil(runs / 256) blocks capped at num_sms * 16."""
    run = 8 if W % 8 == 0 and aligned else 4
    runs = n * H * ceil_div(W, run)
    blocks = min(ceil_div(runs, KTHREADS), sms * 16)
    return run, runs, blocks, ceil_div(runs, blocks * KTHREADS)


def tail_bwd_launch(n, H, W, aligned, sms):
    """bn.cu mpgan_c1_tail_bwd_reduce: RUN 8 when W % 8 == 0 and dy is 16-byte aligned; ceil(runs / 512) blocks capped
    at num_sms * 8."""
    run = 8 if W % 8 == 0 and aligned else 4
    runs = n * H * ceil_div(W, run)
    blocks = min(ceil_div(runs, 2 * KTHREADS), sms * 8)
    return run, runs, blocks, ceil_div(runs, blocks * KTHREADS)


def run_cta(n, H, W, run, blocks):
    """CTA that owns each pixel of an (n, H, W) image under the grid-stride loop (run r -> thread r % (blocks * 256))."""
    wq = ceil_div(W, run)
    q = torch.arange(W) // run
    r = (torch.arange(n * H).view(n, H, 1) * wq + q.view(1, 1, W))
    return (r % (blocks * KTHREADS)) // KTHREADS


def c1act_covered(cy, s, xw, dtype, y_aligned=True, ldy_ok=True):
    """conv_c1_fast.cu c1f_fprop with a slope: the run-based kernel only.  8 | cy with cy / 8 dividing 32, an aligned
    output (16 bytes, pixel stride % 8 == 0), and stride 1, or stride 2 on a bf16 image with 8 | width (vector windows)."""
    cv = cy // 8
    if cy % 8 or not (y_aligned and ldy_ok) or cv > 32 or 32 % cv:
        return False
    vec = dtype == BF and xw % 8 == 0
    return s == 1 or vec


def bwd_apply_chain(P, sms):
    """bn.cu bn_act_bwd_apply for C = 1 (scalar kernel, ew_grid(P, 1, 8, 16)): pixels per thread, the block's fp32
    column sum and one fp32 atomic per CTA onto the prior value."""
    b = ceil_div(P, 256 * 16)
    cap = max(sms * 8, ceil_div(P, 256 * 512))
    grid = max(min(b, cap), 1)
    return ceil_div(P, grid * 256) + 8 + grid + 1


# ------------------------------------------------------------------------------------------------ fp64 references
def prelu(z, slope):
    return torch.where(z > 0, z, slope * z)


def fold_expected(w32, gamma, var, eps, transposed, cy, taps, cx):
    """Runtime.folded's arithmetic on the CPU, fp32: scale = gamma / sqrt(var + eps), bf16(w32 * scale) along the output
    axis (cy of a conv; cx of a ConvTranspose, then transposed to [cx][taps][cy])."""
    scale = gamma.float() / torch.sqrt(var.float() + eps)
    w3 = w32.float().reshape(cy, taps, cx)
    if transposed:
        return (w3 * scale.view(1, 1, -1)).permute(2, 1, 0).contiguous().to(BF), scale
    return (w3 * scale.view(-1, 1, 1)).contiguous().to(BF), scale


def check_fold(wf, bf, w32, b0, gamma, beta, mean, var, eps, transposed, cy, taps, cx, what):
    exp, scale = fold_expected(w32, gamma, var, eps, transposed, cy, taps, cx)
    assert wf.shape == exp.shape, f"{what}: folded weights of shape {tuple(wf.shape)}, expected {tuple(exp.shape)}"
    bad = (wf.view(torch.int16) != exp.view(torch.int16))
    if bool(bad.any()):
        i = tuple(int(v) for v in bad.nonzero()[0])
        names = ("cx", "tap", "cy") if transposed else ("cy", "tap", "cx")
        raise AssertionError(f"{what}: folded weight differs from bf16(w32 * scale) at "
                             + ", ".join(f"{k}={v}" for k, v in zip(names, i))
                             + f" (got {float(wf[i]):.6g}, expected {float(exp[i]):.6g}); {int(bad.sum())} elements")
    sc64 = gamma.double() / torch.sqrt(var.double() + float(torch.tensor(eps, dtype=F32)))
    ref = (b0.double() - mean.double()) * sc64 + beta.double()
    # scale: 3 roundings (add, sqrt, divide); (b - mean) * scale + beta: 3 more
    bnd = 8 * U * ((b0.double() - mean.double()).abs() * sc64.abs() + beta.double().abs()) + 2.0 ** -60
    return check_elementwise(bf.cpu(), ref, bnd, what + " folded bias", names=["channel"])


def tail_fwd_ref_h(c, sc, sh, slope):
    """h = prelu(c * sc + sh) in fp64 from the saved fp32 scale / shift, and its bound."""
    z = c.double() * sc + sh
    h = prelu(z, slope)
    return h, U_OUT[BF] * h.abs() + 2 * U * z.abs() * max(1.0, abs(slope)), z


def stencil(img, w9, flip=False):
    """3x3 zero-padded correlation of (n, H, W) with w9[t] (t = 3 * row + col); flip: w9[8 - t] (the transposed conv)."""
    k = w9.double().view(3, 3)
    if flip:
        k = k.flip(0, 1)
    return F.conv2d(img.double().unsqueeze(1), k.view(1, 1, 3, 3), padding=1).squeeze(1)


def tail_fwd_ref_y(h, w9, b):
    """y = bf16(a) + h with a = conv3x3(h) + b, from the stored h."""
    a = stencil(h, w9) + b
    S = stencil(h.abs(), w9.abs()) + abs(b)
    y = a + h.double()
    return y, U_OUT[BF] * (y.abs() + a.abs()) + 10 * U_ACC * S + 2 * U * (a.abs() + h.double().abs())


def coeffs_ref(stats, P, eps):
    """bn_train_coeffs in fp64: mean, 1 / sqrt(var + eps) and bounds of their fp32 roundings."""
    m = stats[0] / P
    e2 = stats[1] / P
    var = (e2 - m * m).clamp_min(0)
    eps32 = float(torch.tensor(eps, dtype=F32))
    inv = 1 / torch.sqrt(var + eps32)
    dvar = 4 * 2.0 ** -53 * (e2 + m * m)
    return m, var, inv, U * m.abs(), U * inv + 0.5 * dvar / (var + eps32) * inv + 2.0 ** -50 * inv


def check_saved(saved, stats, P, gamma, beta, what):
    mean, inv, sc, sh = (saved[i].double() for i in range(4))
    m, _, inv_ref, bm, bi = coeffs_ref(stats, P, EPS)
    w = check_elementwise(mean.view(1), m.view(1), bm.view(1), what + " saved mean", names=["channel"])
    w = max(w, check_elementwise(inv.view(1), inv_ref.view(1), bi.view(1), what + " saved invstd", names=["channel"]))
    ref = gamma.double() * inv
    w = max(w, check_elementwise(sc.view(1), ref.view(1), (U * ref.abs()).view(1), what + " saved scale",
                                 names=["channel"]))
    ref = beta.double() - mean * sc
    return max(w, check_elementwise(sh.view(1), ref.view(1), (U * (ref.abs() + (mean * sc).abs())).view(1),
                                    what + " saved shift", names=["channel"]))


def check_running(rm, rv, rm0, rv0, saved_mean, stats, P, what):
    mom32 = float(torch.tensor(MOM, dtype=F32))
    keep = float(torch.tensor(1.0, dtype=F32) - torch.tensor(mom32, dtype=F32))
    a, b = keep * rm0.double(), mom32 * saved_mean.double()
    w = check_elementwise(rm.double().view(1), (a + b).view(1), (2 * U * (a.abs() + b.abs()) + U * (a + b).abs()).view(1),
                          what + " running_mean", names=["channel"])
    _, var, _, _, _ = coeffs_ref(stats, P, EPS)
    unb = var * (P / (P - 1)) if P > 1 else var
    a, b = keep * rv0.double(), mom32 * unb
    bnd = 3 * U * (a.abs() + b.abs()) + U * (a + b).abs() + 2.0 ** -40 * b.abs()
    return max(w, check_elementwise(rv.double().view(1), (a + b).view(1), bnd.view(1), what + " running_var",
                                    names=["channel"]))


def check_nbt(nbt, nbt0, what, blocks):
    assert int(nbt) == int(nbt0) + 1, \
        f"{what}: num_batches_tracked went from {int(nbt0)} to {int(nbt)} with {blocks} CTAs in the grid, expected +1"


def check_eval_untouched(before, after, what):
    """Evaluation mode: every BatchNorm / saved buffer other than the scale / shift inputs is left as it was."""
    for k in before:
        b, a = before[k], after[k]
        assert torch.equal(b, a), f"{what}: evaluation mode changed {k} from {b.tolist()} to {a.tolist()}"


def tail_bwd_ref(dy, c, dh, w9, mean, inv, sc, sh, slope, L):
    """dh = bf16(bf16(conv3x3^T(dy)) + dy) and the three sums over the STORED dh and c; returns references and bounds."""
    acc = stencil(dy, w9, flip=True)
    S = stencil(dy.abs(), w9.abs(), flip=True)
    dh_ref = acc + dy.double()
    dh_bnd = U_OUT[BF] * (dh_ref.abs() + acc.abs()) + 9 * U_ACC * S + 2 * U * (acc.abs() + dy.double().abs())
    g, cv = dh.double(), c.double()
    z = cv * sc + sh
    gz = g * torch.where(z > 0, 1.0, slope)
    xh = (cv - mean) * inv
    s = torch.stack([gz.sum(), (gz * xh).sum(), (g * z.clamp_max(0)).sum()])
    t = torch.stack([gz.abs().sum(), (gz * xh).abs().sum(), (g * z.clamp_max(0)).abs().sum()])
    return dh_ref, dh_bnd, s, (L + 3) * U_ACC * t + 2.0 ** -60


# ------------------------------------------------------------------------------------------------ case tables
class TailCase:
    """One call of the fused tail on an (n, H, W) one-channel image.  c_off: element offset of c in its buffer (1: two
    bytes off 16, the 4-pixel variant at any width).  mode: "train" (statistics given) or "eval"."""

    def __init__(self, n, H, W, mode, c_off=0, seed=0, kink=False, note=""):
        self.n, self.H, self.W, self.mode, self.c_off, self.seed, self.kink = n, H, W, mode, c_off, seed, kink
        self.id = f"{mode}-{n}x{H}x{W}" + (f"-off{c_off}" if c_off else "") + ("-kink" if kink else "") + note

    def launch(self, sms):
        return tail_fwd_launch(self.n, self.H, self.W, self.c_off == 0, sms)


GRID_SMS = 148       # the table's grid-stride shapes loop at >= 148 SMs; the GPU cases assert it with the real count
_TAIL_SHAPES = ([(2, 5, w, 0) for w in (8, 16, 24, 520)]                              # <8>
                + [(2, 5, w, 0) for w in (1, 2, 3, 4, 5, 7, 9, 13)] + [(2, 5, 16, 1)]  # <4>
                + [(1, 1, 24, 0), (3, 1, 13, 0), (1, 7, 16, 0), (3, 6, 9, 0)]         # H = 1, n in {1, 3}
                + [(16, 512, 512, 0), (16, 512, 513, 0)])                             # production; <4> grid stride
TAIL_FWD = ([TailCase(n, h, w, "train", o, seed=i) for i, (n, h, w, o) in enumerate(_TAIL_SHAPES)]
            + [TailCase(n, h, w, "eval", o, seed=100 + i, kink=(i % 3 == 0)) for i, (n, h, w, o) in enumerate(_TAIL_SHAPES)]
            + [TailCase(24, 512, 512, "train", seed=50, note="-gridstride")])
TAIL_BWD = ([TailCase(n, h, w, "bwd", o, seed=200 + i, kink=(i % 2 == 0)) for i, (n, h, w, o) in
             enumerate([(2, 5, 8, 0), (2, 5, 520, 0), (2, 5, 13, 0), (2, 5, 16, 1), (3, 1, 7, 0), (1, 7, 1, 0),
                        (16, 512, 512, 0)])]
            + [TailCase(20, 512, 512, "bwd", seed=300, kink=True, note="-gridstride")])


def tail_operands(c):
    """Host operands of a tail case: c (bf16), asymmetric taps, bias, slope, BatchNorm parameters and statistics."""
    cimg = _rnd((c.n, c.H, c.W), c.seed + 1, BF, 3.0, lo=-0.6)
    if c.kink:
        cimg.view(-1)[:: 5] = 0.0
    w9 = torch.tensor([0.75, -0.5, 0.125, 0.3125, 1.25, -0.875, -0.0625, 0.5625, 0.25], dtype=F64)
    w9 = (w9 * (1 + 0.1 * _rnd((9,), c.seed + 2, F64))).to(BF)
    d = {"c": cimg, "w9": w9, "bias": torch.tensor([0.3125], dtype=F32), "slope": torch.tensor([(0.25, -0.5, 1.5, 0.0)[c.seed % 4]]),
         "gamma": torch.tensor([1.375], dtype=F32), "beta": torch.tensor([-0.25], dtype=F32),
         "rm": torch.tensor([0.125], dtype=F32), "rv": torch.tensor([0.75], dtype=F32),
         "nbt": torch.tensor([7], dtype=torch.int64)}
    v = cimg.double()
    d["stats"] = torch.stack([v.sum(), (v * v).sum()])
    if c.mode in ("eval", "bwd"):     # scale / shift inputs (eval) or the saved coefficients (bwd)
        sc = torch.tensor([0.8125], dtype=F32)
        sh = torch.tensor([0.0 if c.kink else -0.3], dtype=F32)
        d["saved"] = torch.cat([torch.tensor([0.0625, 1.0625], dtype=F32), sc, sh])
    if c.mode == "bwd":
        d["dy"] = _rnd((c.n, c.H, c.W), c.seed + 3, BF, 2.0, lo=-0.5)
        d["dparam0"] = torch.tensor([0.5, -0.25, 0.125, 0.75], dtype=F32)    # dgamma, dbeta, dalpha, dbias
    return d


class C1Case:
    """One ``c1_conv_act`` call: (n, H, W) one-channel bf16 (or fp32) input, 3x3 kernel to cy channels."""

    def __init__(self, cy, s, p, n, H, W, dtype=BF, w_off=0, slope=0.25, y_misalign=None, seed=0, kink=False, x_off=0):
        self.cy, self.s, self.p, self.n, self.H, self.W, self.dtype = cy, s, p, n, H, W, dtype
        self.w_off, self.slope, self.y_misalign, self.seed, self.kink, self.x_off = w_off, slope, y_misalign, seed, kink, x_off
        self.ys = ((H + 2 * p - 3) // s + 1, (W + 2 * p - 3) // s + 1)
        self.covered = c1act_covered(cy, s, W, dtype, y_misalign != "base", y_misalign != "stride") and \
            (dtype == BF or s == 1) and (x_off == 0 or s == 1)
        self.id = (f"cy{cy}-s{s}p{p}-{n}x{H}x{W}-y{self.ys[1]}" + ("-f32" if dtype == F32 else "") +
                   (f"-woff{w_off}" if w_off else "") + (f"-xoff{x_off}" if x_off else "") + f"-slope{slope}" +
                   (f"-y{y_misalign}" if y_misalign else "") + ("-kink" if kink else ""))


def _c1_cases():
    cases, i = [], 0
    slopes = (0.25, 0.0, -0.5, 1.5)
    for cy in (8, 16, 32, 64, 128, 256):
        # stride 1 (RUN 8): output widths 7 / 8 / 9 / 24 (pad 1: yw = W) and 6 / 22 (pad 0); W % 8 == 0 -> vector windows
        for (p, W, n, H) in ((1, 7, 2, 3), (1, 8, 3, 1), (1, 9, 2, 4), (1, 24, 2, 5), (0, 8, 2, 4), (0, 24, 1, 5)):
            cases.append(C1Case(cy, 1, p, n, H, W, slope=slopes[i % 4], seed=i, kink=(i % 5 == 0))); i += 1
        # stride 2 (RUN 4, vector windows need 8 | W): output widths 3 / 4 / 8 / 12 / 19 / 20
        for (p, W, n, H) in ((0, 8, 2, 5), (1, 8, 2, 5), (1, 16, 3, 4), (1, 24, 2, 1), (0, 40, 2, 6), (1, 40, 2, 7)):
            cases.append(C1Case(cy, 2, p, n, H, W, slope=slopes[i % 4], seed=i, kink=(i % 5 == 0))); i += 1
    cases += [C1Case(32, 1, 1, 2, 5, 24, w_off=1, seed=90),                      # weights 2 bytes off 16: scalar loads
              C1Case(16, 2, 1, 2, 5, 16, w_off=1, seed=91),
              C1Case(64, 1, 1, 2, 5, 16, x_off=1, seed=92),                      # x 2 bytes off 16: scalar windows
              C1Case(32, 1, 1, 2, 5, 24, dtype=F32, seed=93),                    # fp32 through the C entry point
              C1Case(16, 1, 0, 2, 6, 9, dtype=F32, slope=-0.5, seed=94),
              C1Case(32, 2, 1, 2, 5, 24, dtype=F32, seed=95)]                   # fp32 stride 2: not covered
    # not covered: cy in {24, 48, 512}, stride 2 with W % 8 != 0, a misaligned output base or pixel stride
    cases += [C1Case(24, 1, 1, 2, 5, 16, seed=96), C1Case(48, 1, 1, 2, 5, 16, seed=97),
              C1Case(512, 1, 1, 1, 3, 8, seed=98), C1Case(16, 2, 1, 2, 5, 18, seed=99),
              C1Case(32, 1, 1, 2, 5, 16, y_misalign="base", seed=100), C1Case(32, 1, 1, 2, 5, 16, y_misalign="stride", seed=101)]
    return cases


C1_CASES = _c1_cases()


def tapgemm_tile(ow, oh, od, nimg, r3, npix=128):
    """conv_tc.cu choose_tile: the tw x th (x td) x tn tile the tap-GEMM kernel covers its output grid with."""
    def ilog2(v):
        l = 0
        while (1 << l) < v:
            l += 1
        return l
    best, bl = 1e300, (0, 0, 0)
    for lw in range(6):
        for lh in range(6):
            for ld in range(5 if r3 else 1):
                ln = ilog2(npix) - lw - lh - ld
                if ln < 0 or ln > 4:
                    continue
                tw, th, td, tn = 1 << lw, 1 << lh, 1 << ld, 1 << ln
                work = float(-(-ow // tw) * tw) * (-(-oh // th) * th) * (-(-od // td) * td) * (-(-nimg // tn) * tn)
                work *= 1.0 + 0.02 * ln + 0.01 * (5 - lw) + 0.005 * ld
                if work < best:
                    best, bl = work, (lw, lh, ld)
    return bl


class TcCase:
    """One ``tc_conv_act`` call.  op "act": X (cx) -> Y (cy); "actT": the ConvTranspose Y (cy) -> X (cx).  og: the
    output grid; res: None, "fused" or "unaligned" (must come back as None)."""

    def __init__(self, op, rank, n, cx, cy, og, k=3, s=1, p=1, res=None, seed=0, slope=0.25):
        self.op, self.rank, self.n, self.cx, self.cy, self.og = op, rank, n, cx, cy, tuple(og)
        self.k, self.s, self.p, self.res, self.seed, self.slope = k, s, p, res, seed, slope
        self.taps = k ** rank
        if op == "act":
            self.ys = self.og
            self.xs = tuple((v - 1) * s - 2 * p + k for v in self.og)      # the smallest X giving og
        else:
            self.xs = self.og
            self.ys = tuple((v + 2 * p - k) // s + 1 for v in self.og)
        self.K = (cx if op == "act" else cy) * self.taps + 1 + (1 if res else 0)
        self.id = f"{op}-r{rank}-n{n}-{cx}x{cy}-{'x'.join(map(str, self.og))}-k{k}s{s}p{p}" + (f"-res_{res}" if res else "")


def _tc_cases():
    lw, lh, ld = tapgemm_tile(8, 8, 8, 1, True)
    t = (1 << ld, 1 << lh, 1 << lw)
    grids = [tuple(max(v - 1, 1) for v in t), t, tuple(v + 1 for v in t)]
    cases, i = [], 0
    # the 3-D generator's eval layers (channels 16 / 32 / 64 / 128) on the tap-GEMM R3 epilogue
    for (cx, cy, s, res) in ((16, 16, 1, "fused"), (16, 32, 2, None), (32, 32, 1, "fused"), (32, 64, 2, "fused"),
                             (64, 128, 1, None), (128, 128, 1, "fused")):
        for g in grids:
            cases.append(TcCase("act", 3, 1 + i % 2, cx, cy, g, s=s, res=res, seed=i)); i += 1
    for (cx, cy, s, res) in ((32, 192, 2, None), (16, 64, 2, "fused"), (32, 32, 1, "fused")):
        for g in grids:
            cases.append(TcCase("actT", 3, 1 + i % 2, cx, cy, g, s=s, res=res, seed=i)); i += 1
    # rank-2 tap-GEMM act / actT at the N widths the conv-engine file's four cases miss (16, 32, 256, 512; 1x1 and k4)
    cases += [TcCase("act", 2, 3, 64, 16, (17, 23), k=1, p=0, res="fused", seed=60),
              TcCase("act", 2, 2, 32, 32, (15, 17), k=4, s=2, p=1, seed=61, slope=-0.5),
              TcCase("act", 2, 2, 64, 256, (9, 17), k=1, p=0, seed=62, slope=1.5),
              TcCase("act", 2, 1, 32, 512, (9, 11), k=1, p=0, res="fused", seed=63),
              TcCase("actT", 2, 2, 16, 64, (18, 30), k=4, s=2, p=1, res="fused", seed=64),
              TcCase("actT", 2, 2, 256, 64, (14, 10), k=4, s=2, p=1, seed=65, slope=0.0),
              TcCase("act", 3, 1, 32, 32, t, res="unaligned", seed=66),
              TcCase("act", 2, 2, 64, 16, (17, 23), k=1, p=0, res="unaligned", seed=67)]
    return cases


TC_CASES = _tc_cases()


# ------------------------------------------------------------------------------------------------ conv references
def _nc(t):
    return t.permute((0, t.dim() - 1) + tuple(range(1, t.dim() - 1)))


def _ncl(t):
    return t.permute((0,) + tuple(range(2, t.dim())) + (1,))


def _w_nc(w, rank, k):
    return w.reshape(w.shape[0], *((k,) * rank), w.shape[2]).permute((0, rank + 1) + tuple(range(1, rank + 1)))


def conv_ref(c, x, w, b, res, slope, absolute=False):
    """prelu(conv + b) (+ res) in fp64, channels-last; ``absolute``: the same on |operands| without the activation."""
    f = (lambda t: None if t is None else (t.double().abs() if absolute else t.double()))
    x, w, b, res = f(x), f(w), f(b), f(res)
    conv = F.conv2d if c.rank == 2 else F.conv3d
    if c.op == "act":
        a = _ncl(conv(_nc(x), _w_nc(w, c.rank, c.k), None, stride=c.s, padding=c.p))
    else:
        gin = torch.nn.grad.conv2d_input if c.rank == 2 else torch.nn.grad.conv3d_input
        a = _ncl(gin((x.shape[0], c.cx) + c.xs, _w_nc(w, c.rank, c.k), _nc(x), stride=c.s, padding=c.p))
    a = a + b
    out = a if absolute else prelu(a, slope)
    if res is not None:
        out = out + res
    return out, a


def act_bound(c, x, w, b, res, slope):
    ref, a = conv_ref(c, x, w, b, res, slope)
    S, _ = conv_ref(c, x, w, b, res, slope, absolute=True)
    dtype = x.dtype
    bnd = U_OUT[dtype] * ref.abs() + c.K * U_ACC * S * max(1.0, abs(slope)) + U * (slope * a).abs()
    return ref, bnd


def c1_locate(c):
    run = 8 if c.s == 1 else 4
    return lambda idx: f"run {idx[2] // run} of row {idx[1]} (w0 = {idx[2] // run * run}), channel group {idx[-1] // 8}"


def tc_locate(c):
    og = c.og if c.rank == 3 else (1,) + c.og
    lw, lh, ld = tapgemm_tile(og[2], og[1], og[0], c.n, c.rank == 3)
    tile = ((1 << ld,) if c.rank == 3 else ()) + (1 << lh, 1 << lw)
    return lambda idx: f"tile {tuple(p // t for p, t in zip(idx[1:-1], tile))} of {tile}"


def c1_as_case(c):
    class _C:
        op, rank, k, s, p, cx = "act", 2, 3, c.s, c.p, 1
        K = 10
    _C.s, _C.p, _C.xs = c.s, c.p, (c.H, c.W)
    return _C


def c1_operands(c):
    x = _rnd((c.n, c.H, c.W, 1), c.seed + 1, c.dtype)
    w = _rnd((c.cy, 9, 1), c.seed + 2, c.dtype, 0.7)
    b = _rnd((c.cy,), c.seed + 3, F32, 0.5)
    if c.kink:       # exact zeros of conv + bias: a zero image row band and zero bias in half the channels
        x[:, : max(1, c.H // 2)] = 0
        b[::2] = 0
    return {"x": x, "w": w, "b": b, "slope": torch.tensor([c.slope])}


def tc_operands(c):
    cin = c.cx if c.op == "act" else c.cy
    cout = c.cy if c.op == "act" else c.cx
    isp = c.xs if c.op == "act" else c.ys
    d = {"x": _rnd((c.n,) + isp + (cin,), c.seed + 1, BF), "w": _rnd((c.cy, c.taps, c.cx), c.seed + 2, BF),
         "b": _rnd((cout,), c.seed + 3, F32), "slope": torch.tensor([c.slope])}
    if c.res:
        d["res"] = _rnd((c.n,) + c.og + (cout,), c.seed + 4, BF)
    return d


# ------------------------------------------------------------------------------------------------ CPU models
def model_tail_fwd(c, d, sms=GRID_SMS, fault=None):
    """The tail forward in fp32 with the kernel's rounding points; returns (saved, h, y, rm, rv, nbt)."""
    P = c.n * c.H * c.W
    cv = d["c"].float()
    if c.mode == "train":
        st = d["stats"]
        m = st[0] / P
        var = max(float(st[1] / P - m * m), 0.0)
        mean = torch.tensor(float(m), dtype=F32)
        inv = torch.tensor(1.0 / math.sqrt(var + float(torch.tensor(EPS, dtype=F32))), dtype=F32)
        sc = d["gamma"][0] * inv
        sh = d["beta"][0] - mean * sc
        rm = (1 - torch.tensor(MOM, dtype=F32)) * d["rm"] + torch.tensor(MOM, dtype=F32) * mean
        unb = var * P / (P - 1) if P > 1 else var
        rv = (1 - torch.tensor(MOM, dtype=F32)) * d["rv"] + torch.tensor(MOM, dtype=F32) * torch.tensor(unb, dtype=F32)
        saved = torch.stack([mean, inv, sc.reshape(()), sh.reshape(())])
        nbt = d["nbt"] + (c.launch(sms)[2] if fault == "nbt_per_cta" else 1)
    else:
        saved = d["saved"].clone()
        sc, sh = saved[2], saved[3]
        rm, rv = d["rm"].clone(), d["rv"].clone()
        nbt = d["nbt"] + (1 if fault == "eval_nbt" else 0)
        if fault == "eval_running_mean":
            rm = rm + 0.01
    z = (cv.double() * sc.double() + sh.double()).float()
    h = torch.where(z > 0, z, d["slope"][0] * z).to(BF)
    a = (torch.tensor(0.0, dtype=F64) + stencil(h, d["w9"]) + float(d["bias"][0])).float().to(BF)
    y = (a.float() + h.float()).to(BF)
    if fault == "skip_tail_columns":          # the last W % 4 (or 3) columns of every row left unwritten
        k = c.W % 4 or 3
        y[..., c.W - k:] = 0
    return saved, h, y, rm, rv, nbt


def model_tail_bwd(c, d, sms=GRID_SMS, fault=None):
    """dh = bf16(bf16(acc) + dy) and the three fp64 sums of fp32 per-thread partials; returns (dh, sums3)."""
    w9 = d["w9"]
    acc = stencil(d["dy"], w9, flip=(fault != "unflipped")).float().to(BF)
    dh = (acc.float() + d["dy"].float()).to(BF)
    mean, inv, sc, sh = (float(v) for v in d["saved"])
    slope = float(d["slope"][0])
    g, cv = dh.double(), d["c"].double()
    z = (cv * sc + sh).float().double()
    pos = (z >= 0) if fault == "z_lt_0" else (z > 0)
    gz = g * torch.where(pos, 1.0, slope)
    xh = ((cv - mean).float() * inv).float().double()
    s = torch.stack([gz.sum(), (gz * xh).sum(), (g * z.clamp_max(0)).sum()])
    if fault == "last_cta_missing":
        run, _, blocks, _ = tail_bwd_launch(c.n, c.H, c.W, c.c_off == 0, sms)
        keep = run_cta(c.n, c.H, c.W, run, blocks) != blocks - 1
        s = torch.stack([gz[keep].sum(), (gz * xh)[keep].sum(), (g * z.clamp_max(0))[keep].sum()])
    return dh, s


def model_c1(c, d, fault=None):
    f = {k: v.float() for k, v in d.items()}
    x = _nc(f["x"])
    w = f["w"].reshape(c.cy, 1, 3, 3)
    a = F.conv2d(x, w, None if fault == "bias_after_act" else f["b"], stride=c.s, padding=c.p)
    out = prelu(a, f["slope"][0])
    if fault == "bias_after_act":
        out = out + f["b"].view(1, -1, 1, 1)
    return _ncl(out).to(c.dtype)


# ------------------------------------------------------------------------------------------------ shared checks
def check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, sms, dev="cpu"):
    """In order: saved coefficients, running statistics, num_batches_tracked, h from the saved scale / shift, y from
    the stored h.  Returns the largest err / bound."""
    P = c.n * c.H * c.W
    run, runs, blocks, per = c.launch(sms)
    w = 0.0
    if c.mode == "train":
        st = d["stats"].to(dev)
        w = check_saved(saved.to(dev), st, P, d["gamma"].to(dev)[0], d["beta"].to(dev)[0], c.id)
        w = max(w, check_running(rm.to(dev)[0], rv.to(dev)[0], d["rm"].to(dev)[0], d["rv"].to(dev)[0],
                                 saved.to(dev)[0], st, P, c.id))
        check_nbt(nbt[0], d["nbt"][0], c.id, blocks)
    else:
        check_eval_untouched({"running_mean": d["rm"], "running_var": d["rv"], "num_batches_tracked": d["nbt"],
                              "scale / shift": d["saved"][2:]},
                             {"running_mean": rm.cpu(), "running_var": rv.cpu(), "num_batches_tracked": nbt.cpu(),
                              "scale / shift": saved[2:].cpu()}, c.id)
    sc, sh = float(saved[2]), float(saved[3])
    slope = float(d["slope"][0])
    names = ["image", "row", "column"]
    loc = (lambda idx: f"run {idx[2] // run} (RUN {run}) of row {idx[1]}, CTA "
                       f"{((idx[0] * c.H + idx[1]) * ceil_div(c.W, run) + idx[2] // run) % (blocks * KTHREADS) // KTHREADS}"
                       f" of {blocks}")
    href, hb, _ = tail_fwd_ref_h(d["c"].to(dev), sc, sh, slope)
    if h is not None:
        w = max(w, check_elementwise(h.to(dev), href, hb, c.id + " h", names=names, locate=loc))
        hs = h.to(dev)
    else:
        hs = href.to(BF)
    yref, yb = tail_fwd_ref_y(hs, d["w9"].to(dev), float(d["bias"][0]))
    return max(w, check_elementwise(y.to(dev), yref, yb, c.id + " y", names=names, locate=loc))


def check_tail_bwd(c, d, dh, sums, sms, dev="cpu"):
    run, runs, blocks, per = tail_bwd_launch(c.n, c.H, c.W, c.c_off == 0, sms)
    L = per * run
    mean, inv, sc, sh = (float(v) for v in d["saved"])
    dh_ref, dh_bnd, s, sb = tail_bwd_ref(d["dy"].to(dev), d["c"].to(dev), dh.to(dev), d["w9"].to(dev), mean, inv, sc, sh,
                                         float(d["slope"][0]), L)
    loc = (lambda idx: f"run {idx[2] // run} (RUN {run}) of row {idx[1]}")
    w = check_elementwise(dh.to(dev), dh_ref, dh_bnd, c.id + " dh", names=["image", "row", "column"], locate=loc)
    return max(w, check_elementwise(sums.to(dev), s, sb, c.id + f" sums3 (L = {L}, {blocks} CTAs)", names=["slot"]))


# ------------------------------------------------------------------------------------------------ CPU self-tests
def test_dispatch_mirrors_match_hand_computed_values():
    assert tail_fwd_launch(2, 5, 8, True, 148) == (8, 10, 1, 1)
    assert tail_fwd_launch(2, 5, 16, False, 148) == (4, 40, 1, 1)
    assert tail_fwd_launch(16, 512, 512, True, 148) == (8, 524288, 2048, 1)       # 2048 <= 148 * 16 = 2368
    assert tail_fwd_launch(16, 512, 513, True, 148) == (4, 1056768, 2368, 2)      # capped: threads loop
    assert tail_fwd_launch(24, 512, 512, True, 148) == (8, 786432, 2368, 2)
    assert tail_bwd_launch(10, 512, 512, True, 148) == (8, 327680, 640, 2)        # two runs per thread by design
    assert tail_bwd_launch(20, 512, 512, True, 148) == (8, 655360, 1184, 3)       # capped at 148 * 8: threads loop
    assert tail_bwd_launch(2, 5, 13, True, 148) == (4, 40, 1, 1)
    cta = run_cta(1, 2, 9, 4, 1)
    assert cta.tolist() == [[[0] * 9, [0] * 9]]
    assert c1act_covered(256, 1, 7, BF) and not c1act_covered(512, 1, 8, BF) and not c1act_covered(24, 1, 8, BF)
    assert c1act_covered(16, 2, 16, BF) and not c1act_covered(16, 2, 18, BF) and not c1act_covered(16, 2, 16, F32)
    assert c1act_covered(16, 1, 9, F32) and not c1act_covered(32, 1, 8, BF, y_aligned=False)
    assert tapgemm_tile(8, 8, 8, 1, True) == (3, 3, 1)


def test_case_tables_cover_the_dispatch():
    fwd = {(c.launch(GRID_SMS)[0], c.mode) for c in TAIL_FWD}
    assert fwd == {(8, "train"), (4, "train"), (8, "eval"), (4, "eval")}
    assert any(c.launch(GRID_SMS)[3] > 1 and c.launch(GRID_SMS)[0] == 4 for c in TAIL_FWD)
    assert any(c.launch(GRID_SMS)[3] > 1 and c.launch(GRID_SMS)[0] == 8 for c in TAIL_FWD)
    assert any(tail_bwd_launch(c.n, c.H, c.W, c.c_off == 0, GRID_SMS)[2] == GRID_SMS * 8 for c in TAIL_BWD)
    assert {tail_bwd_launch(c.n, c.H, c.W, c.c_off == 0, GRID_SMS)[0] for c in TAIL_BWD} == {4, 8}
    cov = [c for c in C1_CASES if c.covered]
    for cy in (8, 16, 32, 64, 128, 256):
        for s, run in ((1, 8), (2, 4)):
            yws = {c.ys[1] for c in cov if c.cy == cy and c.s == s}
            assert {run - 1, run} <= yws and any(v > run and v % run for v in yws), (cy, s, yws)
    assert {c.cy for c in C1_CASES if not c.covered} >= {24, 48, 512}
    r3 = [c for c in TC_CASES if c.rank == 3 and c.res != "unaligned"]
    assert {(c.op, c.s, bool(c.res)) for c in r3} >= {("act", 1, True), ("act", 2, False), ("act", 2, True),
                                                     ("actT", 2, False), ("actT", 2, True)}


@pytest.mark.parametrize("c", TAIL_FWD, ids=lambda c: c.id)
def test_checker_accepts_correct_tail_fwd_model(c):
    if c.n * c.H * c.W > (1 << 22) + (1 << 20):
        pytest.skip("the grid-stride shape's model is the production one, larger")
    d = tail_operands(c)
    saved, h, y, rm, rv, nbt = model_tail_fwd(c, d)
    assert check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, GRID_SMS) <= 1.0


@pytest.mark.parametrize("c", TAIL_BWD, ids=lambda c: c.id)
def test_checker_accepts_correct_tail_bwd_model(c):
    d = tail_operands(c)
    dh, s = model_tail_bwd(c, d)
    assert check_tail_bwd(c, d, dh, s, GRID_SMS) <= 1.0


@pytest.mark.parametrize("c", [c for c in C1_CASES if c.covered], ids=lambda c: c.id)
def test_checker_accepts_correct_c1_act_model(c):
    d = c1_operands(c)
    ref, bnd = act_bound(c1_as_case(c), d["x"], d["w"], d["b"], None, c.slope)
    assert check_elementwise(model_c1(c, d), ref, bnd, c.id) <= 1.0


@pytest.mark.parametrize("c", [c for c in TC_CASES if c.res != "unaligned"], ids=lambda c: c.id)
def test_checker_accepts_correct_tc_act_model(c):
    d = tc_operands(c)
    f = {k: v.float() for k, v in d.items()}
    ref32, _ = conv_ref(c, f["x"].float(), f["w"], f["b"], f.get("res"), c.slope)
    ref, bnd = act_bound(c, d["x"], d["w"], d["b"], d.get("res"), c.slope)
    assert check_elementwise(ref32.float().to(BF), ref, bnd, c.id) <= 1.0


def test_checker_rejects_fold_along_cy_of_a_conv_transpose():
    cy, taps, cx = 24, 9, 16          # ConvTranspose(cy -> cx): the output channels are the cx axis
    w32 = _rnd((cy * taps * cx,), 1, F32)
    gamma, var = _rnd((cx,), 2, F32, 2.0), _rnd((cx,), 3, F32, 1.0, lo=0.0) + 1e-3
    good, _ = fold_expected(w32, gamma, var, EPS, True, cy, taps, cx)
    b0, beta, mean = _rnd((cx,), 4, F32), _rnd((cx,), 5, F32), _rnd((cx,), 6, F32)
    sc = gamma / torch.sqrt(var + EPS)
    bf = (b0 - mean) * sc + beta
    check_fold(good, bf, w32, b0, gamma, beta, mean, var, EPS, True, cy, taps, cx, "convT fold")
    # the fault: scale indexed by cy (the first cx of the per-channel scales broadcast along the wrong axis)
    sc_cy = torch.cat([sc, sc])[:cy]
    bad = (w32.view(cy, taps, cx) * sc_cy.view(-1, 1, 1)).permute(2, 1, 0).contiguous().to(BF)
    with pytest.raises(AssertionError, match="cx=.*tap=.*cy="):
        check_fold(bad, bf, w32, b0, gamma, beta, mean, var, EPS, True, cy, taps, cx, "convT fold")


def test_checker_rejects_skipped_last_columns_of_a_4_pixel_row():
    c = next(c for c in TAIL_FWD if c.mode == "train" and c.W == 13)
    d = tail_operands(c)
    saved, h, y, rm, rv, nbt = model_tail_fwd(c, d, fault="skip_tail_columns")
    with pytest.raises(AssertionError, match=r"y: .*column=1[0-2], run 3 \(RUN 4\)"):
        check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, GRID_SMS)


@pytest.mark.parametrize("fault", ["eval_nbt", "eval_running_mean"])
def test_checker_rejects_eval_mode_touching_running_statistics(fault):
    c = next(c for c in TAIL_FWD if c.mode == "eval")
    d = tail_operands(c)
    saved, h, y, rm, rv, nbt = model_tail_fwd(c, d)
    assert check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, GRID_SMS) <= 1.0
    saved, h, y, rm, rv, nbt = model_tail_fwd(c, d, fault=fault)
    with pytest.raises(AssertionError, match="evaluation mode changed"):
        check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, GRID_SMS)


def test_checker_rejects_num_batches_tracked_added_per_cta():
    c = next(c for c in TAIL_FWD if c.mode == "train" and (c.n, c.H, c.W) == (16, 512, 512))
    d = tail_operands(c)
    d["c"] = d["c"][:, :64]        # the model only needs nbt: keep the CPU work small
    c2 = TailCase(16, 64, 512, "train")
    saved, h, y, rm, rv, nbt = model_tail_fwd(c2, dict(d, stats=torch.stack([d["c"].double().sum(),
                                                                              (d["c"].double() ** 2).sum()])),
                                              fault="nbt_per_cta")
    with pytest.raises(AssertionError, match=r"num_batches_tracked went from 7 to 263 with 256 CTAs"):
        check_nbt(nbt[0], d["nbt"][0], c2.id, c2.launch(GRID_SMS)[2])


def test_checker_rejects_unflipped_taps_in_the_backward():
    c = TAIL_BWD[0]
    d = tail_operands(c)
    dh, s = model_tail_bwd(c, d, fault="unflipped")
    with pytest.raises(AssertionError, match="dh: .*run"):
        check_tail_bwd(c, d, dh, s, GRID_SMS)


def test_checker_rejects_sums_without_the_last_cta_at_the_grid_stride_shape():
    c = next(c for c in TAIL_BWD if "gridstride" in c.id)
    assert tail_bwd_launch(c.n, c.H, c.W, True, GRID_SMS)[3] > 1
    d = tail_operands(c)
    dh, s = model_tail_bwd(c, d, fault="last_cta_missing")
    with pytest.raises(AssertionError, match="sums3"):
        check_tail_bwd(c, d, dh, s, GRID_SMS)


def test_checker_rejects_prelu_branch_on_z_lt_0():
    c = next(c for c in TAIL_BWD if c.kink and d_has_zero_z(c))
    d = tail_operands(c)
    dh, s = model_tail_bwd(c, d, fault="z_lt_0")
    with pytest.raises(AssertionError, match="sums3"):
        check_tail_bwd(c, d, dh, s, GRID_SMS)


def d_has_zero_z(c):
    d = tail_operands(c)
    return float(d["saved"][3]) == 0.0 and bool((d["c"] == 0).any()) and float(d["slope"][0]) != 1.0


def test_checker_rejects_bias_added_after_the_activation():
    c = next(c for c in C1_CASES if c.covered and c.slope == -0.5 and not c.kink)
    d = c1_operands(c)
    ref, bnd = act_bound(c1_as_case(c), d["x"], d["w"], d["b"], None, c.slope)
    with pytest.raises(AssertionError, match="channel=.*run"):
        check_elementwise(model_c1(c, d, fault="bias_after_act"), ref, bnd, c.id, locate=c1_locate(c))


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture
def routes(monkeypatch):
    """The ``what`` name of every C entry point ``ops`` calls (ops.check is called once per entry point), plus
    ``c1_conv_act`` (``ops.conv_act`` checks its return code only when it is neither 0 nor -2): "c1_conv_act" for a
    launch, "c1_conv_act:-2" for a layer reported as not covered."""
    from mpgan import _lib, ops
    calls = []
    real = ops.check

    def record(rc, what):
        calls.append(what)
        real(rc, what)

    lib = _lib.load()
    real_c1 = lib.mpgan_c1_conv_act

    def c1(*a):
        rc = real_c1(*a)
        if rc in (0, -2):
            calls.append("c1_conv_act" if rc == 0 else "c1_conv_act:-2")
        return rc

    monkeypatch.setattr(ops, "check", record)
    monkeypatch.setattr(lib, "mpgan_c1_conv_act", c1)
    return calls


class Guards:
    """Device buffers whose margins hold a sentinel that the kernels must leave unchanged."""

    def __init__(self):
        self.keep = []

    def vec(self, host, lo=8, hi=8):
        big = torch.full((lo + host.numel() + hi,), SENT, dtype=host.dtype, device="cuda")
        view = big[lo:lo + host.numel()].view(host.shape)
        view.copy_(host.cuda())
        self.keep.append((big, (slice(lo, lo + host.numel()),)))
        return view

    def sentinel_only(self, n, dtype):
        big = torch.full((n + 16,), SENT, dtype=dtype, device="cuda")
        self.keep.append((big, (slice(0, 0),)))
        return big[8:8 + n]

    def img(self, shape, dtype, off=0):
        n = prod(shape)
        big = torch.full((8 + off + n + 64,), SENT, dtype=dtype, device="cuda")
        self.keep.append((big, (slice(8 + off, 8 + off + n),)))
        return big[8 + off:8 + off + n].view(shape)

    def intact(self, what):
        for big, inner in self.keep:
            mask = torch.ones(big.shape, dtype=torch.bool, device=big.device)
            mask[inner] = False
            outside = big[mask]
            assert torch.all(outside == SENT), \
                f"{what}: {int((outside != SENT).sum())} elements outside the output views were written"


def filled_img(host, off=0):
    """A device copy of ``host`` at element offset ``off`` of a buffer of FILL with one trailing image of FILL."""
    n = host.numel()
    big = torch.full((off + n + prod(host.shape[1:]) + 64,), FILL, dtype=host.dtype, device="cuda")
    v = big[off:off + n].view(host.shape)
    v.copy_(host.cuda())
    return v


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def run_tail_fwd(c, d, G, want_h=True):
    from mpgan import _lib
    lib = _lib.require_device()
    n, H, W = c.n, c.H, c.W
    cimg = filled_img(d["c"], c.c_off)
    h = G.img((n, H, W), BF, c.c_off) if want_h else None
    y = G.img((n, H, W), BF, c.c_off)
    w9, bias, slope = G.vec(d["w9"]), G.vec(d["bias"]), G.vec(d["slope"].float())
    gamma, beta = G.vec(d["gamma"]), G.vec(d["beta"])
    if c.mode == "train":
        stats = G.vec(d["stats"])
        rm, rv, nbt = G.vec(d["rm"]), G.vec(d["rv"]), G.vec(d["nbt"])
        saved = [G.vec(torch.zeros(1, dtype=F32)) for _ in range(4)]
    else:
        stats = None
        rm, rv = G.sentinel_only(1, F32), G.sentinel_only(1, F32)
        nbt = G.sentinel_only(1, torch.int64)
        saved = [G.sentinel_only(1, F32), G.sentinel_only(1, F32), G.vec(d["saved"][2:3]), G.vec(d["saved"][3:4])]
    rc = lib.mpgan_c1_tail_fwd(_p(cimg), n, H, W, _p(stats), _p(gamma), _p(beta), EPS, MOM, _p(rm), _p(rv), _p(nbt),
                               _p(saved[0]), _p(saved[1]), _p(saved[2]), _p(saved[3]), _p(slope), _p(w9), _p(bias), _p(h),
                               _p(y), _stream())
    assert rc == 0, f"{c.id}: c1_tail_fwd returned {rc}"
    torch.cuda.synchronize()
    if c.mode == "eval":      # the untouched buffers read as their original values for check_eval_untouched
        for t in (rm, rv, nbt, saved[0], saved[1]):
            assert torch.all(t == SENT), f"{c.id}: evaluation mode wrote a BatchNorm / saved buffer"
        rm_out, rv_out, nbt_out = d["rm"].clone(), d["rv"].clone(), d["nbt"].clone()
    else:
        rm_out, rv_out, nbt_out = rm.cpu(), rv.cpu(), nbt.cpu()
    sv = torch.cat([s.cpu() for s in saved])
    return sv, (h.clone() if h is not None else None), y.clone(), rm_out, rv_out, nbt_out


# ------------------------------------------------------------------------------------------------ GPU: the UNet tail
@pytest.mark.gpu
@pytest.mark.parametrize("c", TAIL_FWD, ids=lambda c: c.id)
def test_tail_fwd_elementwise(c, routes):
    nsm = sms()
    d = tail_operands(c)
    G = Guards()
    saved, h, y, rm, rv, nbt = run_tail_fwd(c, d, G)
    G.intact(c.id)
    if "gridstride" in c.id or (c.W == 513):
        assert c.launch(nsm)[3] > 1, f"{c.id}: no grid-stride loop at {nsm} SMs"
    w = check_tail_fwd(c, d, saved, h, y, rm, rv, nbt, nsm, dev="cuda")
    # without h_out: y identical (training mode moves the running statistics again: fresh copies)
    G2 = Guards()
    _, h2, y2, _, _, _ = run_tail_fwd(c, d, G2, want_h=False)
    G2.intact(c.id + " (no h_out)")
    assert h2 is None and torch.equal(y2, y), f"{c.id}: y differs when h is not stored"
    report("c1_tail_fwd", c.id, w)


@pytest.mark.gpu
@pytest.mark.parametrize("c", TAIL_BWD, ids=lambda c: c.id)
def test_tail_bwd_elementwise(c, routes):
    from mpgan import _lib, ops
    lib = _lib.require_device()
    nsm = sms()
    d = tail_operands(c)
    G = Guards()
    n, H, W = c.n, c.H, c.W
    dy = filled_img(d["dy"], c.c_off)
    cimg = filled_img(d["c"], 0)
    sv = [G.vec(d["saved"][i:i + 1]) for i in range(4)]
    slope, w9 = G.vec(d["slope"].float()), G.vec(d["w9"])
    dh = G.img((n, H, W), BF)
    sums = G.vec(torch.zeros(3, dtype=F64))
    rc = lib.mpgan_c1_tail_bwd_reduce(_p(dy), _p(cimg), n, H, W, _p(sv[0]), _p(sv[1]), _p(sv[2]), _p(sv[3]), _p(slope),
                                      _p(w9), _p(dh), _p(sums), _stream())
    assert rc == 0
    dp = [G.vec(d["dparam0"][i:i + 1]) for i in range(4)]
    dc = G.img((n, H, W), BF)
    rc = lib.mpgan_bn_act_bwd_apply(ops.dt(dh), _p(dh), 1, _p(cimg), 1, n * H * W, 1, _p(sv[0]), _p(sv[1]),
                                    _p(sv[2]), _p(sv[3]), ACT_PRELU, _p(slope), 0.0, _p(sums), _p(dp[0]), _p(dp[1]),
                                    _p(dp[2]), _p(dp[3]), _p(dc), 1, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    G.intact(c.id)
    if "gridstride" in c.id:
        assert tail_bwd_launch(n, H, W, True, nsm)[3] > 1, f"{c.id}: no grid-stride loop at {nsm} SMs"
    w = check_tail_bwd(c, d, dh, sums, nsm, dev="cuda")
    w = max(w, check_dc(c, d, dh, cimg, sums, dc, dp, nsm))
    report("c1_tail_bwd", c.id, w)


def check_dc(c, d, dh, cimg, sums, dc, dp, nsm):
    """bn_act_bwd_apply with C = 1 from the kernel's own sums: dc = sc g act'(z) + k2 (c - mean) + k3, and the
    parameter gradients accumulated onto their starting values."""
    P = c.n * c.H * c.W
    mean, inv, sc, sh = (float(v) for v in d["saved"])
    slope = float(d["slope"][0])
    s = sums.double()
    g, cv = dh.double(), cimg.double()
    z = cv * sc + sh
    f = torch.where(z > 0, 1.0, slope)
    k2 = -sc * inv * (s[1] / P)
    k3 = -sc * (s[0] / P)
    ref = sc * g * f + k2 * (cv - mean) + k3
    mag = (sc * g * f).abs() + k2.abs() * (cv.abs() + abs(mean)) + k3.abs()
    w = check_elementwise(dc, ref, U_OUT[BF] * ref.abs() + 12 * U * mag, c.id + " dc", names=["image", "row", "column"])
    d0 = d["dparam0"].double().cuda()
    for i, (name, src) in enumerate((("dgamma", s[1]), ("dbeta", s[0]), ("dalpha", s[2]))):
        r = d0[i] + src
        w = max(w, check_elementwise(dp[i].view(1), r.view(1), (2 * U * (d0[i].abs() + src.abs())).view(1),
                                     c.id + " " + name, names=["slot"]))
    dcs = dc.double()
    L = bwd_apply_chain(P, nsm)
    r = d0[3] + dcs.sum()
    return max(w, check_elementwise(dp[3].view(1), r.view(1), (L * U_ACC * (d0[3].abs() + dcs.abs().sum())).view(1),
                                    c.id + " dbias", names=["slot"]))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [c for c in TAIL_FWD if c.n * c.H * c.W < (1 << 20)], ids=lambda c: c.id)
def test_unfused_tail_route_elementwise(c, routes):
    """The route the generator takes without the fused tail: bn_act_apply (PReLU) -> 1 -> 1 conv -> add_copy, against
    the same fp64 references (scale / shift given, as in evaluation mode)."""
    from mpgan import ops
    d = tail_operands(TailCase(c.n, c.H, c.W, "eval", seed=c.seed, kink=c.kink))
    cimg = filled_img(d["c"]).view(c.n, c.H, c.W, 1)
    G = Guards()
    sc, sh = G.vec(d["saved"][2:3]), G.vec(d["saved"][3:4])
    slope = G.vec(d["slope"].float())
    h = G.img((c.n, c.H, c.W, 1), BF)
    routes.clear()
    ops.bn_act_apply(cimg, sc, sh, ACT_PRELU, slope, 0.0, None, h)
    spec = ops.ConvSpec(2, 1, 1, 3, 1, 1)
    a, _ = ops.conv_fprop(spec, h, d["w9"].cuda().view(1, 9, 1), d["bias"].cuda())
    y = G.img((c.n, c.H, c.W, 1), BF)
    ops.add_copy(a, h, y)
    torch.cuda.synchronize()
    G.intact(c.id)
    assert routes[0] == "bn_act_apply" and routes[-1] == "add_copy", routes
    href, hb, _ = tail_fwd_ref_h(d["c"].cuda(), float(d["saved"][2]), float(d["saved"][3]), float(d["slope"][0]))
    w = check_elementwise(h.view(c.n, c.H, c.W), href, hb, c.id + " h (bn_act_apply)", names=["image", "row", "column"])
    yref, yb = tail_fwd_ref_y(h.view(c.n, c.H, c.W), d["w9"].cuda(), float(d["bias"][0]))
    w = max(w, check_elementwise(y.view(c.n, c.H, c.W), yref, yb, c.id + " y (conv + add_copy)",
                                 names=["image", "row", "column"]))
    report("unfused_tail", c.id, w)


# ------------------------------------------------------------------------------------------------ GPU: c1_conv_act
@pytest.mark.gpu
@pytest.mark.parametrize("c", C1_CASES, ids=lambda c: c.id)
def test_c1_conv_act_elementwise(c, routes):
    from mpgan import _lib, ops
    lib = _lib.require_device()
    d = c1_operands(c)
    spec = ops.ConvSpec(2, 1, c.cy, 3, c.s, c.p)
    x = filled_img(d["x"], c.x_off)
    wbig = torch.full((c.cy * 9 + 16,), FILL, dtype=c.dtype, device="cuda")
    w = wbig[8 + c.w_off:8 + c.w_off + c.cy * 9].view(c.cy, 9, 1)
    w.copy_(d["w"].cuda())
    b, slope = d["b"].cuda(), d["slope"].float().cuda()
    lo, hi = {None: (8, 8), "base": (1, 15), "stride": (8, 3)}[c.y_misalign]
    bigo = torch.full((c.n + 1,) + c.ys + (lo + c.cy + hi,), SENT, dtype=c.dtype, device="cuda")
    out = bigo[:c.n, ..., lo:lo + c.cy]
    G = Guards()
    G.keep.append((bigo, (slice(0, c.n), slice(None), slice(None), slice(lo, lo + c.cy))))
    routes.clear()
    if c.dtype == F32:     # fp32 through the C entry point (ops.conv_act takes bf16 only)
        g = spec.geom(c.n, (c.H, c.W), c.ys)
        rc = lib.mpgan_c1_conv_act(ctypes.byref(g), ops.dt(x), _p(x), 1, _p(w), _p(b), _p(slope), _p(out), out.stride(-2),
                                   _stream())
        assert rc == (0 if c.covered else -2), f"{c.id}: mpgan_c1_conv_act returned {rc}"
        r = out if rc == 0 else None
    else:
        r = ops.conv_act(spec, x, w, b, slope, out=out)
    torch.cuda.synchronize()
    G.intact(c.id)
    covered = c.covered and (not FALLBACK or c.dtype == F32)     # the C entry point does not read MPGAN_NO_C1ACT
    ref, bnd = act_bound(c1_as_case(c), d["x"], d["w"], d["b"], None, c.slope)
    if covered:
        assert r is not None and routes == ["c1_conv_act"], f"{c.id}: route {routes}"
        wst = check_elementwise(out, ref.cuda(), bnd.cuda(), c.id, locate=c1_locate(c))
        report("c1_conv_act", c.id, wst)
        return
    assert r is None, f"{c.id}: the layer is not covered, conv_act must return None"
    assert all(v == "c1_conv_act:-2" for v in routes), f"{c.id}: launches although not covered: {routes}"
    assert torch.all(out == SENT), f"{c.id}: a declined call wrote its output"
    if c.dtype == F32:
        return
    # the unfused route: convolution (stored, rounded), then bn_act_apply with scale 1 / shift 0
    a, _ = ops.conv_fprop(spec, x, w, b)
    one, zero = torch.ones(c.cy, device="cuda"), torch.zeros(c.cy, device="cuda")
    y = ops.bn_act_apply(a, one, zero, ACT_PRELU, slope, 0.0, None, torch.empty_like(a))
    _, acc = conv_ref(c1_as_case(c), d["x"], d["w"], d["b"], None, c.slope)
    wst = check_elementwise(y, ref.cuda(), bnd.cuda() + U_OUT[BF] * acc.abs().cuda() * max(1.0, abs(c.slope)),
                            c.id + " (unfused)", locate=c1_locate(c))
    report("c1_conv_act_unfused", c.id, wst)


# ------------------------------------------------------------------------------------------------ GPU: tc_conv_act
@pytest.mark.gpu
@pytest.mark.parametrize("c", TC_CASES, ids=lambda c: c.id)
def test_tc_conv_act_elementwise(c, routes):
    from mpgan import ops
    d = tc_operands(c)
    cin = c.cx if c.op == "act" else c.cy
    cout = c.cy if c.op == "act" else c.cx
    big = torch.full((c.n + 1,) + d["x"].shape[1:-1] + (8 + cin + 8,), FILL, dtype=BF, device="cuda")
    x = big[:c.n, ..., 8:8 + cin]
    x.copy_(d["x"].cuda())
    w = d["w"].cuda()
    b, slope = d["b"].cuda(), d["slope"].float().cuda()
    res = None
    if c.res:
        lo, hi = (8, 8) if c.res == "fused" else (1, 2)
        rb = torch.full((c.n + 1,) + c.og + (lo + cout + hi,), FILL, dtype=BF, device="cuda")
        res = rb[:c.n, ..., lo:lo + cout]
        res.copy_(d["res"].cuda())
    bigo = torch.full((c.n + 1,) + c.og + (16 + cout + 16,), SENT, dtype=BF, device="cuda")
    out = bigo[:c.n, ..., 16:16 + cout]
    G = Guards()
    G.keep.append((bigo, (slice(0, c.n),) + (slice(None),) * c.rank + (slice(16, 16 + cout),)))
    if c.op == "act":
        spec = ops.ConvSpec(c.rank, c.cx, c.cy, c.k, c.s, c.p)
        routes.clear()
        r = ops.conv_act(spec, x, w, b, slope, res=res, out=out)
    else:
        wt = torch.empty(w.numel(), dtype=BF, device="cuda")
        ops.weight_transpose(w, wt, c.cy, c.taps, c.cx)
        spec = ops.ConvSpec(c.rank, c.cx, c.cy, c.k, c.s, c.p, transposed=True,
                            output_padding=c.xs[0] - ((c.ys[0] - 1) * c.s - 2 * c.p + c.k))
        routes.clear()
        r = ops.conv_act(spec, x, wt, b, slope, res=res, out=out)
    torch.cuda.synchronize()
    G.intact(c.id)
    if c.res == "unaligned":
        assert r is None and routes == [], f"{c.id}: an unaligned residual must be declined, got route {routes}"
        assert torch.all(out == SENT)
        return
    assert r is not None and routes == ["tc_conv_act"], f"{c.id}: route {routes}"
    ref, bnd = act_bound(c, d["x"], d["w"], d["b"], d.get("res"), c.slope)
    wst = check_elementwise(out, ref.cuda(), bnd.cuda(), c.id, locate=tc_locate(c))
    report("tc_conv_act", c.id, wst)


# ------------------------------------------------------------------------------------------------ GPU: the fold
def _gen_with_distinct_bn(rank, seed=0):
    """A bf16 CasNetGenerator (one UNet) whose every BatchNorm has its own per-channel gamma / beta / statistics,
    with a channel of running_var ~1e-6, one of gamma = 0 and a 1e3 spread between channels."""
    import mpgan
    torch.manual_seed(seed)
    shape = (1,) + (32,) * rank
    gen = mpgan.CasNetGenerator(shape, n_unet_blocks=1, dims=rank, precision="bf16")
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for m in gen.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                C = m.num_features
                spread = torch.logspace(-1.5, 1.5, C, dtype=F64)[torch.randperm(C, generator=g)]
                m.weight.copy_((0.5 + torch.rand(C, generator=g, dtype=F64)) * spread.sqrt())
                m.bias.copy_(torch.rand(C, generator=g, dtype=F64) - 0.5)
                m.running_mean.copy_((torch.rand(C, generator=g, dtype=F64) - 0.5) * 0.2)
                m.running_var.copy_(spread * (0.5 + torch.rand(C, generator=g, dtype=F64)) * 1e-2)
                m.running_var[0] = 1e-6
                if C > 1:
                    m.weight[C - 1] = 0.0
    gen.cuda()
    gen.eval()
    return gen


def _fused_convs(gen):
    from mpgan.nets import Convolution
    return [m for m in gen.modules() if isinstance(m, Convolution) and not m.conv_only]


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [2, 3])
def test_fold_bit_exact_and_layer_against_eval_definition(rank, routes):
    from mpgan import ops
    gen = _gen_with_distinct_bn(rank)
    x = _rnd((1, 1) + (32,) * rank, 5, F32).cuda()
    with torch.no_grad():
        gen.run_forward(x, save=False, need_wgrad=False)
    rt = gen.runtime
    worst, n_layers, declined = 0.0, 0, []
    for i, m in enumerate(_fused_convs(gen)):
        rec = rt.rec[m.conv]
        sp = rec.spec
        wf, bf = rt.folded(m.conv, m.norm)
        bn = m.norm
        b0 = m.conv.bias.detach()
        what = f"r{rank} layer {i} ({'ConvT' if sp.transposed else 'Conv'} {sp.cx}x{sp.cy} s{sp.stride[0]})"
        worst = max(worst, check_fold(wf.cpu(), bf.cpu(), rec.w32.cpu(), b0.cpu(), bn.weight.detach().cpu(),
                                      bn.bias.detach().cpu(), bn.running_mean.cpu(), bn.running_var.cpu(), bn.eps,
                                      sp.transposed, sp.cy, sp.taps, sp.cx, what))
        # the fused layer against the module's eval-mode definition, fp64 from the fp32 master weights
        cin, cout = (sp.cy, sp.cx) if sp.transposed else (sp.cx, sp.cy)
        isp = (5, 6, 7) if rank == 3 else (9, 16)      # 8 | width: the stride-2 first layer takes c1_conv_act
        xin = _rnd((2,) + isp + (cin,), 10 + i, BF)
        routes.clear()
        y = ops.conv_act(sp, xin.cuda().contiguous(), wf, bf, m.act.weight.detach(), res=None)
        if y is None:
            declined.append((sp.cx, sp.cy, sp.transposed))
            continue
        n_layers += 1
        c = TcCase("actT" if sp.transposed else "act", rank, 2, sp.cx, sp.cy,
                   sp.x_of_y(isp) if sp.transposed else sp.y_of_x(isp), k=sp.k[0], s=sp.stride[0], p=sp.pad[0])
        # first the kernel on its own operands (the folded bf16 weights and fp32 bias), then the eval definition
        wk = wf.view(sp.cx, sp.taps, sp.cy).permute(2, 1, 0) if sp.transposed else wf.view(sp.cy, sp.taps, sp.cx)
        kref, kbnd = act_bound(c, xin, wk.cpu(), bf.cpu(), None, float(m.act.weight))
        worst = max(worst, check_elementwise(y.cpu(), kref, kbnd, what + " fused layer vs its folded operands"))
        w32 = rec.w32.view(sp.cy, sp.taps, sp.cx).double().cpu()
        sc64 = bn.weight.detach().double().cpu() / torch.sqrt(bn.running_var.double().cpu() + bn.eps)
        slope = float(m.act.weight)
        _, a = conv_ref(c, xin, w32, b0.double().cpu(), None, slope)     # conv + b (pre-activation, exact)
        z = (a - bn.running_mean.double().cpu()) * sc64 + bn.bias.detach().double().cpu()
        ref = prelu(z, slope)
        wsc = (w32 * (sc64.view(1, 1, -1) if sp.transposed else sc64.view(-1, 1, 1))).abs()
        S, _ = conv_ref(c, xin, wsc, bf.abs().double().cpu(), None, 1.0, absolute=True)
        bnd = U_OUT[BF] * ref.abs() + (c.K + 8) * U_ACC * S * max(1.0, abs(slope)) + U_OUT[BF] * S * max(1.0, abs(slope))
        if sp.cx == 1 and not sp.transposed and not FALLBACK:
            assert routes == ["c1_conv_act"], f"{what}: route {routes}"
        else:
            assert routes == ["tc_conv_act"], f"{what}: route {routes}"
        worst = max(worst, check_elementwise(y.cpu(), ref, bnd, what + " fused layer vs eval definition"))
    # the top ConvTranspose (32 -> 1) has one output channel: no tcgen05 tile; its fold is unused (the fused tail or
    # the unfused BatchNorm runs it).  Rank 3 has no one-channel fused kernel; MPGAN_NO_C1ACT removes rank 2's.
    expected_declined = [(1, 32, True)] + ([(1, 16, False)] if rank == 3 or FALLBACK else [])
    assert sorted(declined) == sorted(expected_declined), f"rank {rank}: layers conv_act declines: {declined}"
    report("fold", f"r{rank}", worst)
    print(f"[inference-kernel] fold r{rank}: {n_layers} fused layers checked, declined {declined}")


@pytest.mark.gpu
def test_fold_cache_refreshes_in_place():
    gen = _gen_with_distinct_bn(2, seed=3)
    x = _rnd((1, 1, 32, 32), 5, F32).cuda()
    with torch.no_grad():
        gen.run_forward(x, save=False, need_wgrad=False)
    rt = gen.runtime
    m = _fused_convs(gen)[2]
    wf, bf = rt.folded(m.conv, m.norm)
    wf2, bf2 = rt.folded(m.conv, m.norm)
    assert wf2 is wf and bf2 is bf, "a second call must return the cached tensors"
    ptrs = (wf.data_ptr(), bf.data_ptr())
    old = wf.clone()
    with torch.no_grad():
        m.norm.running_var.mul_(4.0)
    wf3, bf3 = rt.folded(m.conv, m.norm)
    assert (wf3.data_ptr(), bf3.data_ptr()) == ptrs and not torch.equal(wf3, old)
    sp = rt.rec[m.conv].spec
    check_fold(wf3.cpu(), bf3.cpu(), rt.rec[m.conv].w32.cpu(), m.conv.bias.detach().cpu(), m.norm.weight.detach().cpu(),
               m.norm.bias.detach().cpu(), m.norm.running_mean.cpu(), m.norm.running_var.cpu(), m.norm.eps,
               sp.transposed, sp.cy, sp.taps, sp.cx, "after a running_var edit")
    other = _gen_with_distinct_bn(2, seed=9)
    gen.load_state_dict({k: v.cpu() for k, v in other.state_dict().items()})
    wf4, bf4 = rt.folded(m.conv, m.norm)
    assert (wf4.data_ptr(), bf4.data_ptr()) == ptrs
    check_fold(wf4.cpu(), bf4.cpu(), rt.rec[m.conv].w32.cpu(), m.conv.bias.detach().cpu(), m.norm.weight.detach().cpu(),
               m.norm.bias.detach().cpu(), m.norm.running_mean.cpu(), m.norm.running_var.cpu(), m.norm.eps,
               sp.transposed, sp.cy, sp.taps, sp.cx, "after load_state_dict")


# ------------------------------------------------------------------------------------------------ GPU: routes
def _route_multiset(rank, n_unets):
    import collections
    import mpgan
    torch.manual_seed(0)
    size = 64 if rank == 2 else 32
    gen = mpgan.CasNetGenerator((1,) + (size,) * rank, n_unet_blocks=n_unets, dims=rank, precision="bf16").cuda().eval()
    x = _rnd((2 if rank == 2 else 1, 1) + (size,) * rank, 3, F32).cuda()
    with torch.no_grad():
        gen.run_forward(x, save=False, need_wgrad=False)        # materialise and fold outside the recorded call
    return gen, x, collections.Counter


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [2, 3])
def test_eval_forward_routes(rank, routes):
    gen, x, Counter = _route_multiset(rank, 2 if rank == 2 else 1)
    n_unets = 2 if rank == 2 else 1
    routes.clear()
    with torch.no_grad():
        gen.run_forward(x, save=False, need_wgrad=False)
    torch.cuda.synchronize()
    got = Counter(routes)
    n_fused = len(_fused_convs(gen))
    if FALLBACK:
        assert not {"c1_conv_act", "tc_conv_act", "c1_tail_fwd"} & set(got), f"fusions ran with the switches set: {got}"
        assert got["bn_act_apply"] == n_fused, f"{got['bn_act_apply']} bn_act_apply for {n_fused} BatchNorm layers"
        return
    if rank == 2:
        per = {"c1_conv_fprop": 1, "c1_conv_act": 1, "tc_conv_fprop": 3, "tc_conv_act": 11, "tc_convt_to1": 1,
               "bn_finalize": 1, "c1_tail_fwd": 1}
    else:
        per = {"im2col_c1_vol": 2, "tc_conv_fprop(im2col vol)": 2, "bn_finalize": 2, "bn_act_apply": 2,
               "tc_conv_act": 11, "tc_conv_fprop": 3, "tc_conv_fprop(col2im vol)": 1, "col2im_c1_vol": 1,
               "stencil27": 1, "add_copy": 1}
    exp = Counter({k: v * n_unets for k, v in per.items()})
    exp["add_copy"] += 1          # the input cast to bf16
    exp["tanh_fwd"] += 1
    assert got == exp, f"rank-{rank} eval forward routes {dict(got)}, expected {dict(exp)}"
    if rank == 2:
        assert got["bn_act_apply"] == 0


# ------------------------------------------------------------------------------------------------ GPU: graph
def _graph_model():
    import mpgan
    torch.manual_seed(0)
    model = mpgan.GAN(1, 64, 64, precision="bf16").cuda()
    gen = model.generator
    with torch.no_grad():
        for m in gen.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                m.running_mean.uniform_(-0.1, 0.1)
                m.running_var.uniform_(0.5, 2.0)
    gen.eval()
    return model, gen


def _eager(gen, x):
    with torch.no_grad():
        y, _ = gen.run_forward(x, save=False, need_wgrad=False)
    return y.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("change", ["load_state_dict", "param_inplace", "running_var", "training_step"])
def test_graphed_generator_follows_weight_changes(change, routes):
    import mpgan
    from mpgan import inference
    from oracle.gan import synthetic_batch
    model, gen = _graph_model()
    x = _rnd((2, 1, 64, 64), 4, F32).cuda()
    gg = inference.GraphedGenerator(gen, (2, 1, 64, 64), torch.device("cuda"))
    y0 = gg(x)
    assert torch.equal(y0, _eager(gen, x))
    routes.clear()
    gg(x)
    assert routes == [], f"a replay with unchanged weights launched {routes}"
    if change == "load_state_dict":
        torch.manual_seed(5)
        other = mpgan.GAN(1, 64, 64, precision="bf16")
        gen.load_state_dict(other.generator.state_dict())
    elif change == "param_inplace":
        with torch.no_grad():
            next(m for m in gen.modules() if isinstance(m, torch.nn.Conv2d)).weight.mul_(1.5)
    elif change == "running_var":
        with torch.no_grad():
            next(m for m in gen.modules() if isinstance(m, torch.nn.BatchNorm2d)).running_var.mul_(3.0)
    else:
        batch = {k: v.cuda() for k, v in synthetic_batch(2, 2, 64, seed=3).items()}
        gen.train()
        model.discriminator.train()
        model.fused_step(batch)
        gen.eval()
    y1 = gg(x)                       # before any eager call could refresh the captured buffers
    ye = _eager(gen, x)
    assert not torch.equal(ye, y0), "the change did not change the generator's output"
    assert torch.equal(y1, ye), \
        f"after {change}: the replay differs from the eager forward (max |diff| {float((y1 - ye).abs().max()):.3g})"
    assert torch.equal(gg(x), ye)


@pytest.mark.gpu
def test_graphed_infer_volume_matches_eager_after_weight_change():
    import mpgan
    from mpgan import inference
    model, gen = _graph_model()
    vol = _rnd((5, 1, 64, 64), 6, F32).cuda()
    gg = inference.GraphedGenerator(gen, (2, 1, 64, 64), torch.device("cuda"))
    assert torch.equal(inference.infer_volume(gen, vol, batch=2, graphed=gg), inference.infer_volume(gen, vol, batch=2))
    torch.manual_seed(7)
    other = mpgan.GAN(1, 64, 64, precision="bf16")
    gen.load_state_dict(other.generator.state_dict())
    got = inference.infer_volume(gen, vol, batch=2, graphed=gg)      # 2 + 2 replayed, the ragged last slice eager
    ref = inference.infer_volume(gen, vol, batch=2)
    assert torch.equal(got, ref), f"slices {sorted(set(torch.nonzero(got != ref)[:, 0].tolist()))} differ"


@pytest.mark.gpu
def test_graphed_generator_refuses_moved_parameters():
    from mpgan import inference
    _, gen = _graph_model()
    x = _rnd((2, 1, 64, 64), 4, F32).cuda()
    gg = inference.GraphedGenerator(gen, (2, 1, 64, 64), torch.device("cuda"))
    gg(x)
    gen.runtime.materialize(torch.device("cuda"))
    with pytest.raises(RuntimeError, match="moved since the CUDA graph was captured"):
        gg(x)


# ------------------------------------------------------------------------------------------------ child run
@pytest.mark.gpu
def test_unfused_routes_in_child_process():
    """The GPU cases with MPGAN_NO_EVAL_FUSION, MPGAN_NO_TAIL_FUSION and MPGAN_NO_C1ACT set (read per call or once per
    process; a child keeps them out of this one): conv_act declines the one-channel layers, the generator's eval
    forward runs BatchNorm apply after every convolution, and the same references hold."""
    if FALLBACK:
        pytest.skip("this is the child run")
    env = dict(os.environ, **{s: "1" for s in SWITCHES}, **{CHILD: "1"})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
        ["-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-p", "no:cacheprovider", "-rA", "-s",
         "-k", "c1_conv_act or unfused_tail or routes or fold_bit"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    lines = [l[l.index("[inference-kernel]"):] for l in r.stdout.splitlines() if "[inference-kernel]" in l]
    print("\n".join(lines))
    assert r.returncode == 0, "unfused run failed:\n" + r.stdout[-6000:] + r.stderr[-3000:]
    assert lines and all(" unfused " in l or "fold r" in l for l in lines)
    assert any("c1_conv_act_unfused" in l for l in lines)
