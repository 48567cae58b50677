"""Every convolution engine, element-wise against fp64, at the edges of its own tiling.

Each case runs one ``ops.conv_*`` call on channel slices of wider buffers and compares every stored element with the
same operation computed in fp64 on the operands the kernel received (bf16- or fp32-rounded), under a bound derived
from the arithmetic, not fitted to the output:

    |got - ref| <= u_out * |ref| + K * 2^-23 * S  (+ u_out * |t| for every intermediate t the engine rounds)

* ``S`` is the same operation on |x|, |w| (and |bias|, |res|, |dw0|): it bounds every partial sum.
* ``K`` is the number of terms summed into one output (products, bias, residual, prior ``dw``).  fp32 accumulation of K
  terms in any order errs by at most (K - 1) * 2^-24 * S; 2^-23 per term leaves room for accumulators that truncate
  instead of rounding, and for the rounding of fp32 products when the operands themselves are fp32.
* ``u_out`` is the relative rounding of the stored value: 2^-8 for bf16 outputs, 2^-23 for fp32 (``dw``).
* Routes that store an intermediate and add to it later (``add_copy`` after the convolution, the bf16 per-tap partials
  of ``col2im_c1_vol``) round once more: their bound adds u_out times the magnitude of that intermediate.

Fused BatchNorm statistics are fp64 atomics of fp32 per-CTA partial sums of the STORED values (squares of bf16 values are
exact in fp32), so per channel |stats - sum(v)| <= L * 2^-23 * sum(|v|), L the longest fp32 chain: the pixels of the
tiles one CTA walks for the halo engines (``stats_chain``), every pixel of the call otherwise.

Where K is so large (2^20 pixels of a weight gradient) that K * 2^-23 * S would hide a whole tile, the case runs on
integer operands in {-1, 0, 1}: every partial sum is then an integer below 2^24, fp32 arithmetic is exact in any order,
and the bound is zero.

Every case also asserts the Python-level route, the sequence of C entry points ``ops`` called.  The choice made inside
one entry point (halo / stride-2 halo / weight-gradient halo engine, or the tap-GEMM / wgrad_kernel it falls back to) is
invisible here: the cases name the ``return 1`` predicates they satisfy, and ``test_fallback_engines_in_child_process``
re-runs the file with every ``MPGAN_NO_*`` switch set, so the fallback engines are checked at the same shapes.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BF, F32 = torch.bfloat16, torch.float32
U_ACC = 2.0 ** -23                     # per summed term (see the module docstring)
U_OUT = {BF: 2.0 ** -8, F32: 2.0 ** -23}
FILL = 1024.0                          # channels / images outside an input slice: any read of them is a large error
SENT = -320.0                          # output margins (exact in bf16): must be unchanged after the call
SWITCHES = ("MPGAN_NO_HALO", "MPGAN_NO_HALO_S2", "MPGAN_NO_WGRAD_HALO", "MPGAN_NO_C1RUN", "MPGAN_NO_C1MMA",
            "MPGAN_NO_CLS_MINOR", "MPGAN_NO_C1VOL", "MPGAN_NO_C1OUT", "MPGAN_NO_CONVT1", "MPGAN_NO_C1COL",
            "MPGAN_NO_C1ACT")
CHILD = "MPGAN_CONV_ENGINES_CHILD"     # set in the child run: every switch above is set, and it must not recurse
FALLBACK = os.environ.get(CHILD) == "1"
NOT_FUSED = {"conv_fprop", "conv_bprop", "stencil27", "col2im_c1_vol", "tc_conv_bprop_c1out"}   # return fused=False


# ------------------------------------------------------------------------------------------------ the checker
def _ncl(t):
    """N C *S -> N *S C."""
    return t.permute((0,) + tuple(range(2, t.dim())) + (1,))


def _nc(t):
    """N *S C -> N C *S."""
    return t.permute((0, t.dim() - 1) + tuple(range(1, t.dim() - 1)))


def check_elementwise(got, ref, bound, what, tile=None, names=None, tile_stride=1):
    """Assert |got - ref| <= bound element-wise; on failure name the worst element (and its tile: positions are divided
    by ``tile_stride`` first when the engine tiles a parity-class grid).  Returns the largest |got - ref| / bound."""
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
        if tile is not None and ratio.dim() >= 3:
            pos = idx[1:-1]
            pos = pos[-len(tile):]
            msg += f", tile {tuple(p // tile_stride // t for p, t in zip(pos, tile))} of {tile}"
            if tile_stride > 1:
                msg += f" of parity class {tuple(p % tile_stride for p in pos)}"
        msg += f" (got {float(got[idx]):.6g}, ref {float(ref[idx]):.6g}, bound {float(bound[idx]):.3g}); " \
               f"{int((ratio > 1).sum())} elements out of bounds"
        raise AssertionError(msg)
    return worst


def check_stats(stats, stored, what, chain=None):
    """stats: fp64 [2C] = per-channel sum and sum of squares of ``stored`` (N *S C).  ``chain``: the most values one fp32
    partial sum of the epilogue adds up (default: every pixel); the fp64 combination of the partials adds nothing
    visible at this scale."""
    v = stored.double().reshape(-1, stored.shape[-1])
    p = v.shape[0] if chain is None else min(chain, v.shape[0])
    r1 = check_elementwise(stats[: v.shape[1]].view(1, 1, -1), v.sum(0).view(1, 1, -1),
                           (p * U_ACC * v.abs().sum(0)).view(1, 1, -1), what + " (channel sums)")
    r2 = check_elementwise(stats[v.shape[1]:].view(1, 1, -1), (v * v).sum(0).view(1, 1, -1),
                           (p * U_ACC * (v * v).sum(0)).view(1, 1, -1), what + " (channel sums of squares)")
    return max(r1, r2)


# ------------------------------------------------------------------------------------------------ fp64 references
def _conv(rank):
    return F.conv2d if rank == 2 else F.conv3d


def _grad(rank):
    return (torch.nn.grad.conv2d_input, torch.nn.grad.conv2d_weight) if rank == 2 else \
        (torch.nn.grad.conv3d_input, torch.nn.grad.conv3d_weight)


def _w_nc(w, c):
    """[cy][taps][cx] -> (cy, cx, k, k[, k])."""
    return w.reshape(w.shape[0], *c.k, w.shape[2]).permute((0, c.rank + 1) + tuple(range(1, c.rank + 1)))


def reference(c, ops_in, absolute=False):
    """The case's operation in fp64 on the operands the kernel received (channels-last result).  ``absolute``: the same
    operation on |operands| (the bound's S).  Returns (total, conv part)."""
    f = (lambda t: None if t is None else (t.double().abs() if absolute else t.double()))
    x, w, b, res, dw0, slope = (f(ops_in.get(k)) for k in ("x", "w", "b", "res", "dw0", "slope"))
    gin, gw = _grad(c.rank)
    if c.op in ("fprop", "act"):
        part = _ncl(_conv(c.rank)(_nc(x), _w_nc(w, c), None, stride=c.s, padding=c.p))
        out = part + (b if b is not None else 0)
        if c.op == "act":
            out = out if absolute else torch.where(out >= 0, out, slope * out)
    elif c.op in ("bprop", "actT"):     # w: the forward layer's weight in both cases
        part = _ncl(gin((c.n, c.cx) + c.xs, _w_nc(w, c), _nc(x), stride=c.s, padding=c.p))
        out = part + (b if b is not None else 0)
        if c.op == "actT":
            out = out if absolute else torch.where(out >= 0, out, slope * out)
    else:
        y = f(ops_in["y"])
        part = gw(_nc(x), (c.cy, c.cx) + c.k, _nc(y), stride=c.s, padding=c.p)
        part = part.permute((0,) + tuple(range(2, c.rank + 2)) + (1,)).reshape(c.cy, c.taps, c.cx)
        out = part + dw0
    if res is not None:
        out = out + res
    return out, part


def bound_of(c, ops_in, route, ref, part, S, S_part, u_out):
    if c.exact:
        # integer operands: every product and partial sum is an integer of magnitude <= S < 2^24, so every fp32
        # addition (in any order, rounded or truncated) and the fp32 store are exact
        assert float(S.max()) < 2.0 ** 24
        return torch.zeros_like(ref)
    K = c.K + (1 if ops_in.get("b") is not None else 0) + (1 if ops_in.get("res") is not None else 0)
    bnd = u_out * ref.abs() + K * U_ACC * S
    if "add_copy" in route:           # the convolution is stored (rounded), then the residual is added and stored again
        bnd = bnd + u_out * (part + (ops_in["b"].double() if ops_in.get("b") is not None else 0)).abs()
    if "col2im_c1_vol" in route:      # bf16 per-tap partial products, summed by the gather: sum |partial_t| <= S
        bnd = bnd + U_OUT[BF] * S_part
    return bnd


# ------------------------------------------------------------------------------------------------ case tables
class Case:
    """One call of one entry point.  xs: X-grid spatial extents (the Y grid follows from k, s, p).  op: fprop (X -> Y),
    bprop (Y -> X), wgrad, act (conv_act, X -> Y) or actT (conv_act of the transposed layer, Y -> X).  route / route_fb:
    the C entry points ``ops`` calls by default / with every MPGAN_NO_* switch set (None: the same)."""

    def __init__(self, engine, op, rank, n, cx, cy, xs, k=3, s=1, p=1, *, route, route_fb=None, dtype=BF, bias=True,
                 stats=False, res=None, tile=None, kw=None, exact=False):
        self.engine, self.op, self.rank, self.n, self.cx, self.cy = engine, op, rank, n, cx, cy
        self.xs, self.k, self.s, self.p = tuple(xs), (k,) * rank, s, p
        self.taps = k ** rank
        self.ys = tuple((v + 2 * p - k) // s + 1 for v in self.xs)
        self.dtype, self.bias, self.stats, self.res, self.tile, self.kw = dtype, bias, stats, res, tile, kw or {}
        self.route, self.route_fb = tuple(route), tuple(route_fb) if route_fb is not None else tuple(route)
        self.exact = exact
        red = cx if op in ("fprop", "act") else cy
        self.K = self.n * prod(self.ys) + 1 if op == "wgrad" else red * self.taps
        self.id = (f"{engine}-{op}-r{rank}-n{n}-{cx}x{cy}-{'x'.join(map(str, self.xs))}-k{k}s{s}p{p}"
                   f"{'-f32' if dtype == F32 else ''}{'-stats' if stats else ''}{'-res_' + res if res else ''}"
                   f"{''.join('-' + a for a in self.kw)}")

    def expected(self):
        return self.route_fb if FALLBACK else self.route

    def out_grid(self):
        return (self.ys, self.cy) if self.op in ("fprop", "act") else (self.xs, self.cx)


def prod(t):
    r = 1
    for v in t:
        r *= v
    return r


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


TF, TB, TW = ("tc_conv_fprop",), ("tc_conv_bprop",), ("tc_conv_wgrad",)
TBR = ("tc_conv_bprop_res",)
HALO_TILE = (16, 8)

# tap-GEMM (conv_tc.cu run_tapgemm): layers no specialised engine takes.  KC = 64 / 32 / 16 for C % 64 / 32 / 16 == 0;
# BN = largest of 256..16 dividing N; 128-pixel tiles from choose_tile (several tiny images per tile for n = 37).
TAPGEMM = [
    # k4 s2 parity classes (fprop: 4 input-parity maps; bprop: 4 output-parity classes), odd extents
    Case("tapgemm", "fprop", 2, 2, 64, 128, (29, 31), 4, 2, 0, route=TF, stats=True),
    Case("tapgemm", "bprop", 2, 2, 64, 128, (29, 31), 4, 2, 0, route=TBR, stats=True, res="fused"),
    Case("tapgemm", "fprop", 2, 3, 128, 256, (17, 15), 4, 2, 1, route=TF),
    Case("tapgemm", "bprop", 2, 3, 128, 256, (17, 15), 4, 2, 1, route=TB + ("add_copy",), res="unaligned"),
    Case("tapgemm", "fprop", 3, 2, 32, 64, (9, 11, 13), 4, 2, 0, route=TF, stats=True),
    Case("tapgemm", "bprop", 3, 2, 32, 64, (9, 11, 13), 4, 2, 0, route=TBR, res="fused"),
    Case("tapgemm", "bprop", 3, 1, 16, 32, (7, 10, 9), 3, 2, 1, route=TB, stats=True),       # unequal tap classes
    Case("tapgemm", "fprop", 3, 2, 16, 32, (5, 6, 7), 3, 1, 1, route=TF, stats=True),
    # 1x1: a plain GEMM over pixels
    Case("tapgemm", "fprop", 2, 3, 64, 128, (17, 23), 1, 1, 0, route=TF, stats=True),
    Case("tapgemm", "bprop", 2, 3, 64, 128, (17, 23), 1, 1, 0, route=TB),
    # 3x3 s1 with 9 * C * N * 2 bytes of weights above the halo kernel's shared-memory budget (halo3x3_run: w_bytes)
    Case("tapgemm", "fprop", 2, 2, 128, 128, (17, 23), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "bprop", 2, 2, 128, 128, (19, 13), 3, 1, 0, route=TBR, res="fused"),
    # every BN, C giving KC = 16 / 32 / 64 (C = 48 / 96 / 192: no halo engine takes them)
    Case("tapgemm", "fprop", 2, 2, 48, 16, (9, 17), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "fprop", 2, 2, 96, 32, (9, 17), 3, 1, 0, route=TF, stats=True),
    Case("tapgemm", "fprop", 2, 2, 192, 64, (9, 17), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "fprop", 2, 2, 48, 128, (9, 17), 3, 1, 0, route=TF, stats=True),
    Case("tapgemm", "fprop", 2, 2, 96, 256, (9, 17), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "fprop", 2, 1, 192, 512, (9, 17), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "bprop", 2, 2, 16, 48, (9, 17), 3, 1, 1, route=TB, stats=True),
    Case("tapgemm", "bprop", 2, 2, 256, 96, (9, 17), 3, 1, 1, route=TB),
    Case("tapgemm", "bprop", 2, 1, 512, 192, (9, 17), 3, 1, 0, route=TB, bias=False),   # N = 512 > BN: two N tiles
    # choose_tile packing several tiny images into one 128-pixel tile
    Case("tapgemm", "fprop", 2, 37, 48, 32, (3, 5), 3, 1, 1, route=TF, stats=True),
    Case("tapgemm", "bprop", 2, 37, 32, 48, (3, 5), 3, 1, 1, route=TB, stats=True),
    # inference fusion on the tap-GEMM epilogue: PReLU + residual
    Case("tapgemm", "act", 2, 2, 64, 128, (29, 31), 4, 2, 0, route=("tc_conv_act",), res="fused"),
]

# wgrad_kernel (conv_tc.cu run_wgrad): nx = min(cx, 256) X channels per CTA, cx_blocks = cx / nx; "small" (<= 2^20 output
# pixels, cx <= 64) halves shared memory / TMEM.  k4 s2 and 1x1 layers: wgrad_halo_run needs a 3x3 kernel.
WGRAD = [
    Case("wgrad_kernel", "wgrad", 2, 2, 16, 32, (29, 31), 4, 2, 1, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 3, 32, 64, (17, 15), 4, 2, 0, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 2, 64, 128, (29, 31), 4, 2, 0, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 2, 128, 64, (19, 21), 3, 1, 1, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 2, 256, 32, (9, 17), 3, 1, 0, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 1, 512, 64, (9, 11), 3, 1, 1, route=TW),               # cx_blocks = 2
    Case("wgrad_kernel", "wgrad", 2, 37, 32, 16, (3, 5), 3, 2, 1, route=TW),               # tiny images; X != 2 Y
    Case("wgrad_kernel", "wgrad", 3, 2, 32, 64, (9, 11, 13), 4, 2, 0, route=TW),
    Case("wgrad_kernel", "wgrad", 3, 1, 64, 32, (5, 6, 7), 3, 1, 1, route=TW),
    Case("wgrad_kernel", "wgrad", 2, 2, 16, 128, (23, 17), 3, 1, 1, route=TW),             # cy = 128: no halo wgrad
    # both sides of the small split: 1 024 x 1 024 = 2^20 output pixels is small, one more image row is not.  With 2^20
    # summed terms the rounding bound would hide a whole tile, so these run on integer operands and must be exact.
    Case("wgrad_kernel", "wgrad", 2, 1, 16, 16, (1024, 1024), 1, 1, 0, route=TW, exact=True),
    Case("wgrad_kernel", "wgrad", 2, 1, 16, 16, (1025, 1024), 1, 1, 0, route=TW, exact=True),
    Case("wgrad_kernel", "wgrad", 2, 1, 64, 16, (1025, 1024), 1, 1, 0, route=TW, exact=True),
]

# halo3x3 (conv_halo.cuh): stride-1 3x3, pad 0 / 1, C and N in {16, 32, 64, 128} within the shared-memory budget,
# 16-byte aligned operands with pixel strides % 8 (the slices here keep that); 16 rows x 8 columns per output tile.
# Extents tile - 1, tile, tile + 1 and several tiles + a remainder; an image smaller than one tile.
HALO = [
    Case("halo", "fprop", 2, 3, 16, 16, (15, 7), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 16, 32, (18, 10), p=0, route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 32, 16, (17, 9), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 32, 64, (39, 29), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 64, 128, (35, 19), p=0, route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 128, 64, (20, 12), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 3, 128, 16, (5, 3), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 2, 64, 32, (40, 24), route=TF, stats=True, tile=HALO_TILE),
    # ring of input planes: N <= 64 and <= 32 * SMs tiles caps the ring (4 buffers for 32 -> 64) and ~10 tiles per CTA
    # wrap it; 5 120 tiles lift the cap (8 buffers); N = 128 is never capped
    Case("halo", "fprop", 2, 3, 32, 64, (256, 256), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 10, 32, 64, (256, 256), route=TF, stats=True, tile=HALO_TILE),
    Case("halo", "fprop", 2, 3, 16, 128, (256, 256), route=TF, stats=True, tile=HALO_TILE),
    # data gradient: w = transposed shadow, taps flipped, pad 2 - p; residual fused
    Case("halo", "bprop", 2, 2, 16, 32, (17, 9), route=TBR, stats=True, res="fused", tile=HALO_TILE),
    Case("halo", "bprop", 2, 3, 64, 16, (15, 7), p=0, route=TB, stats=True, tile=HALO_TILE),
    Case("halo", "bprop", 2, 2, 128, 64, (39, 29), route=TB + ("add_copy",), res="unaligned", tile=HALO_TILE),
    Case("halo", "bprop", 2, 2, 32, 128, (16, 8), route=TB, tile=HALO_TILE),
    Case("halo", "act", 2, 2, 32, 32, (39, 29), route=("tc_conv_act",), res="fused", tile=HALO_TILE),
    # one-input-channel data gradient: N padded to 16, only column 0 stored (bprop_c1out)
    Case("halo", "bprop", 2, 2, 1, 64, (17, 9), route=("tc_conv_bprop_c1out",), route_fb=("c1_conv_bprop",), bias=False,
         tile=HALO_TILE, kw={"force_c1out": True}),
    Case("halo", "bprop", 2, 3, 1, 16, (41, 30), p=0, route=("tc_conv_bprop_c1out",),
         route_fb=("c1_conv_bprop", "add_copy"), bias=False, res="fused", tile=HALO_TILE, kw={"force_c1out": True}),
    Case("halo", "bprop", 2, 1, 1, 128, (16, 8), route=("tc_conv_bprop_c1out",), route_fb=("c1_conv_bprop",), bias=False,
         tile=HALO_TILE, kw={"force_c1out": True}),
    # ConvTranspose(C -> 1, k3 s2 p1 op1) in pixel-shuffle mode: Y width % 8 == 0, statistics of the one channel
    Case("halo", "bprop", 2, 2, 1, 32, (34, 16), 3, 2, 1, route=("tc_convt_to1",), route_fb=("c1_conv_bprop",),
         stats=True, tile=(32, 16)),
    Case("halo", "bprop", 2, 3, 1, 16, (18, 48), 3, 2, 1, route=("tc_convt_to1", "add_copy"),
         route_fb=("c1_conv_bprop", "add_copy"), res="fused", tile=(32, 16)),
    Case("halo", "bprop", 2, 1, 1, 64, (2, 16), 3, 2, 1, route=("tc_convt_to1",), route_fb=("c1_conv_bprop",),
         stats=True, tile=(32, 16)),
]

# stride-2 halo (conv_s2.cuh halo_s2_run): k3 s2 p1 with X = 2 Y, 16 x 8 tiles on the Y grid.  Mode 0 (dir 0): C = cx in
# {16, 32}, N = cy in {32, 64, 128, 192}, statistics only for N <= 64 (with statistics a wider N goes to the tap-GEMM).
# Mode 1 (dir 1): N = cx in {16, 32}, C = cy in {32} or 64..512 in steps of 64.
S2 = [
    Case("halo_s2", "fprop", 2, 2, 16, 32, (30, 14), 3, 2, 1, route=TF, stats=True, tile=HALO_TILE),
    Case("halo_s2", "fprop", 2, 2, 32, 64, (32, 16), 3, 2, 1, route=TF, stats=True, tile=HALO_TILE),
    Case("halo_s2", "fprop", 2, 3, 16, 128, (34, 18), 3, 2, 1, route=TF, tile=HALO_TILE),
    Case("halo_s2", "fprop", 2, 2, 32, 192, (78, 58), 3, 2, 1, route=TF, tile=HALO_TILE),
    Case("halo_s2", "fprop", 2, 3, 16, 64, (8, 6), 3, 2, 1, route=TF, stats=True, tile=HALO_TILE),
    Case("halo_s2", "bprop", 2, 2, 16, 32, (30, 14), 3, 2, 1, route=TB, stats=True, tile=HALO_TILE),
    Case("halo_s2", "bprop", 2, 2, 32, 64, (32, 16), 3, 2, 1, route=TBR, stats=True, res="fused", tile=HALO_TILE),
    Case("halo_s2", "bprop", 2, 2, 16, 128, (34, 18), 3, 2, 1, route=TB, stats=True, tile=HALO_TILE),
    Case("halo_s2", "bprop", 2, 2, 32, 192, (78, 58), 3, 2, 1, route=TB, stats=True, tile=HALO_TILE),
    Case("halo_s2", "bprop", 2, 1, 16, 256, (36, 20), 3, 2, 1, route=TB, stats=True, tile=HALO_TILE),
    # the largest mode-1 layer within the budget (9 * C * N * 2 bytes of weights + a ring of C / 64 + 1 planes of
    # 17 x 9 x 64 x 2 bytes): N = 16, C = 320 (216 128 of 231 424 bytes)
    Case("halo_s2", "bprop", 2, 2, 16, 320, (30, 14), 3, 2, 1, route=TB, stats=True, tile=HALO_TILE),
    # above the budget (N = 32 from C = 256, N = 16 from C = 384): halo_s2_run returns 1, the tap-GEMM runs
    Case("tapgemm", "bprop", 2, 2, 32, 320, (8, 6), 3, 2, 1, route=TB),
    Case("tapgemm", "bprop", 2, 1, 16, 512, (34, 18), 3, 2, 1, route=TB + ("add_copy",), res="unaligned"),
    Case("halo_s2", "act", 2, 2, 32, 64, (34, 18), 3, 2, 1, route=("tc_conv_act",), res="fused", tile=HALO_TILE),
    Case("halo_s2", "actT", 2, 2, 16, 128, (30, 14), 3, 2, 1, route=("tc_conv_act",), res="fused", tile=HALO_TILE),
]

# weight-gradient halo (conv_wgrad_halo.cuh): cx in {16, 32}, cy in {16, 32, 64}, stride 1 (Y = X + 2p - 2) or stride 2
# pad 1 (X = 2 Y); wgrad_halo64 for cx = 64 stride 1, cy in {64, 128}.  16 x 8 tiles on the Y grid.
WGH = [
    Case("wgrad_halo", "wgrad", 2, 2, 16, 16, (15, 7), route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 3, 16, 32, (18, 10), p=0, route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 2, 16, 64, (39, 29), route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 2, 32, 16, (17, 9), p=0, route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 3, 32, 32, (5, 3), route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 2, 32, 64, (40, 24), route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 2, 16, 16, (30, 14), 3, 2, 1, route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 3, 16, 64, (34, 18), 3, 2, 1, route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 2, 32, 32, (32, 16), 3, 2, 1, route=TW, tile=HALO_TILE),
    Case("wgrad_halo", "wgrad", 2, 1, 32, 64, (78, 58), 3, 2, 1, route=TW, tile=HALO_TILE),
    Case("wgrad_halo64", "wgrad", 2, 2, 64, 64, (17, 9), route=TW, tile=HALO_TILE),        # Y 17 x 9: tile + 1
    Case("wgrad_halo64", "wgrad", 2, 3, 64, 128, (41, 30), p=0, route=TW, tile=HALO_TILE),
    Case("wgrad_halo64", "wgrad", 2, 1, 64, 64, (5, 3), route=TW, tile=HALO_TILE),
]

C1F, C1B, C1W = ("c1_conv_fprop",), ("c1_conv_bprop",), ("c1_conv_wgrad",)
C1COL = ("im2col_c1", "tc_conv_wgrad(im2col)", "fold_dw16")
# one-input-channel rank-2 3x3 layers.  conv_c1mma.cuh: bf16, stride 1, cy in {16, 32, 64}, width % 8 == 0 (128-pixel
# tiles run across image ends).  conv_c1_fast.cu: the run-based kernels (stride 1; stride 2 with width % 8 == 0 in bf16)
# and the pixel-at-a-time kernels otherwise, cy / 8 channel groups per pixel.  conv_c1.cu: the generic one-channel
# kernels (conv_to1, wgrad_x1).  conv_c1col.cu: im2col + tcgen05 weight gradient for cy % 16 == 0 <= 256.
C1 = [
    Case("c1mma", "fprop", 2, 3, 1, 16, (13, 16), route=C1F, stats=True),
    Case("c1mma", "fprop", 2, 2, 1, 32, (31, 40), p=0, route=C1F, stats=True),
    Case("c1mma", "fprop", 2, 5, 1, 64, (7, 8), route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 8, (13, 17), route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 16, (13, 18), 3, 2, 1, route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 32, (19, 19), p=0, route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 64, (9, 20), 3, 2, 0, route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 128, (11, 21), route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 256, (10, 22), 3, 2, 1, route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 1, 1, 512, (9, 23), route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 32, (14, 24), 3, 2, 1, route=C1F, stats=True),       # stride 2, 16-byte windows
    Case("c1_fast", "fprop", 2, 3, 1, 1, (21, 19), route=C1F, stats=True),
    Case("c1_fast", "fprop", 2, 2, 1, 32, (15, 21), route=C1F, stats=True, dtype=F32),
    Case("c1_fast", "fprop", 2, 2, 1, 16, (15, 21), 3, 2, 1, route=C1F, dtype=F32),
    Case("c1_fast", "bprop", 2, 2, 1, 8, (13, 17), route=C1B, stats=True),
    Case("c1_fast", "bprop", 2, 2, 1, 16, (14, 18), 3, 2, 1, route=C1B, stats=True),      # Y width 9: no convt_to1
    Case("c1_fast", "bprop", 2, 2, 1, 128, (22, 20), 3, 2, 1, route=C1B + ("add_copy",), res="fused"),
    Case("c1_fast", "bprop", 2, 2, 1, 256, (11, 21), route=C1B + ("add_copy",), res="fused"),
    Case("c1_fast", "bprop", 2, 3, 1, 1, (21, 19), p=0, route=C1B, stats=True),
    Case("c1_fast", "bprop", 2, 2, 1, 32, (15, 21), route=C1B, dtype=F32, stats=True),
    Case("c1_fast", "wgrad", 2, 2, 1, 8, (13, 17), route=C1W),
    Case("c1_fast", "wgrad", 2, 2, 1, 16, (14, 24), 3, 2, 1, route=C1W),
    Case("c1_fast", "wgrad", 2, 2, 1, 64, (19, 22), p=0, route=C1W),
    Case("c1_fast", "wgrad", 2, 3, 1, 1, (21, 24), route=C1W),                             # 1 -> 1: wgrad11 run kernel
    Case("c1_fast", "wgrad", 2, 2, 1, 32, (15, 21), 3, 2, 1, route=C1W, dtype=F32),
    Case("c1", "fprop", 2, 2, 32, 1, (13, 17), 3, 1, 1, route=C1F, stats=True),           # conv_to1, 32 input channels
    Case("c1", "fprop", 3, 2, 16, 1, (5, 6, 7), 3, 2, 1, route=C1F, stats=True, dtype=F32),
    Case("c1", "bprop", 3, 2, 1, 24, (5, 6, 7), 3, 2, 1, route=C1B, stats=True),
    Case("c1", "wgrad", 2, 2, 1, 96, (13, 17), route=C1W),                                 # wgrad_x1: cy / 8 > 8 groups
    Case("c1", "wgrad", 3, 2, 1, 24, (5, 6, 7), 3, 2, 1, route=C1W),
    Case("c1col", "wgrad", 2, 2, 1, 16, (31, 17), route=C1COL, route_fb=C1W, kw={"force_c1col": True}),
    Case("c1col", "wgrad", 2, 3, 1, 64, (20, 21), 3, 2, 1, route=C1COL, route_fb=C1W, kw={"force_c1col": True}),
    Case("c1col", "wgrad", 2, 1, 1, 256, (18, 9), p=0, route=C1COL, route_fb=("conv_wgrad",), kw={"force_c1col": True}),
]

# rank-3 one-input-channel 3x3x3 layers (conv_c1vol.cu): 27-point stencils for 1 -> 1 (stride 1, pad 1), otherwise
# im2col (27 taps -> 32 columns) + tcgen05 1x1x1 conv / weight gradient, and per-tap partials + col2im for the data
# gradient.  With MPGAN_NO_C1VOL they run on the one-channel and generic kernels.
VOL = [
    Case("c1vol", "fprop", 3, 3, 1, 1, (9, 8, 10), route=("stencil27",), route_fb=C1F),
    Case("c1vol", "fprop", 3, 3, 1, 1, (9, 8, 10), route=("stencil27",), route_fb=C1F, dtype=F32),
    Case("c1vol", "bprop", 3, 2, 1, 1, (7, 9, 6), route=("stencil27",), route_fb=C1B + ("add_copy",), res="fused"),
    Case("c1vol", "wgrad", 3, 2, 1, 1, (7, 9, 6), route=("stencil27_wgrad",), route_fb=C1W),
    Case("c1vol", "wgrad", 3, 2, 1, 1, (7, 9, 6), route=("stencil27_wgrad",), route_fb=C1W, dtype=F32),
    Case("c1vol", "fprop", 3, 2, 1, 64, (10, 9, 11), p=0, route=("im2col_c1_vol", "tc_conv_fprop(im2col vol)"),
         route_fb=("conv_fprop",), stats=True),
    Case("c1vol", "fprop", 3, 2, 1, 16, (12, 12, 13), 3, 2, 1, route=("im2col_c1_vol", "tc_conv_fprop(im2col vol)"),
         route_fb=("conv_fprop",), stats=True),
    Case("c1vol", "bprop", 3, 1, 1, 32, (8, 10, 6), 3, 2, 1, route=("tc_conv_fprop(col2im vol)", "col2im_c1_vol"),
         route_fb=C1B + ("add_copy",), res="fused"),
    Case("c1vol", "bprop", 3, 2, 1, 16, (7, 7, 9), route=("tc_conv_fprop(col2im vol)", "col2im_c1_vol"), route_fb=C1B),
    Case("c1vol", "wgrad", 3, 2, 1, 64, (10, 9, 11), p=0,
         route=("im2col_c1_vol", "tc_conv_wgrad(im2col vol)", "fold_dw32"), route_fb=("conv_wgrad",)),
    Case("c1vol", "wgrad", 3, 2, 1, 16, (12, 12, 13), 3, 2, 1,
         route=("im2col_c1_vol", "tc_conv_wgrad(im2col vol)", "fold_dw32"), route_fb=C1W),
]

# generic implicit-GEMM kernels (conv_generic.cu): whatever no other engine takes -- odd channel counts, fp32.
GF, GB, GW = ("conv_fprop",), ("conv_bprop",), ("conv_wgrad",)
GENERIC = [
    Case("generic", "fprop", 2, 2, 3, 5, (13, 11), route=GF, dtype=F32),
    Case("generic", "fprop", 2, 2, 3, 5, (13, 11), route=GF),
    Case("generic", "bprop", 2, 2, 3, 5, (13, 11), route=GB, dtype=F32, res="fused", route_fb=None),
    Case("generic", "bprop", 2, 2, 24, 40, (13, 15), 4, 2, 0, route=GB),
    Case("generic", "wgrad", 2, 2, 24, 40, (13, 15), 4, 2, 0, route=GW),
    Case("generic", "wgrad", 2, 2, 3, 5, (13, 11), route=GW, dtype=F32),
    Case("generic", "fprop", 3, 2, 7, 9, (7, 6, 5), 3, 2, 1, route=GF),
    Case("generic", "fprop", 3, 1, 6, 10, (8, 7, 9), 3, 1, 0, route=GF, dtype=F32),
    Case("generic", "bprop", 3, 2, 7, 9, (7, 6, 5), 3, 2, 1, route=GB, dtype=F32),
    Case("generic", "wgrad", 3, 2, 7, 9, (7, 6, 5), 3, 2, 1, route=GW),
    Case("generic", "fprop", 2, 2, 64, 128, (9, 10), 3, 1, 1, route=GF, dtype=F32),
    Case("generic", "wgrad", 2, 2, 32, 16, (9, 10), 3, 1, 1, route=GW, dtype=F32),
]
for _c in GENERIC:       # the add_copy that follows a generic data gradient with a residual
    if _c.op == "bprop" and _c.res:
        _c.route = _c.route_fb = _c.route + ("add_copy",)

ALL = TAPGEMM + WGRAD + HALO + S2 + WGH + C1 + VOL + GENERIC


# ------------------------------------------------------------------------------------------------ running one case
def _rnd(shape, seed, dtype, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return ((torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * scale).to(dtype)


def make_operands(c, seed=0):
    """Host tensors with the values the kernel receives (already rounded to the case's dtype)."""
    xs_in = c.xs if c.op in ("fprop", "act", "wgrad") else c.ys
    cin = c.cx if c.op in ("fprop", "act", "wgrad") else c.cy
    if c.exact:      # integers in {-1, 0, 1} (dw0 in -4..4): no rounding anywhere, a single missing pixel shows
        rnd = (lambda shape, seed, dtype, scale=1.0: _rnd(shape, seed, torch.float64, scale + 0.5).round().to(dtype))
    else:
        rnd = _rnd
    d = {"x": rnd((c.n,) + xs_in + (cin,), seed + 1, c.dtype),
         "w": rnd((c.cy, c.taps, c.cx), seed + 2, c.dtype)}
    if c.op == "wgrad":
        d["y"] = rnd((c.n,) + c.ys + (c.cy,), seed + 3, c.dtype)
        d["dw0"] = rnd((c.cy, c.taps, c.cx), seed + 4, F32, 4.0)
        return d
    (osp, cout) = c.out_grid()
    if c.bias:
        d["b"] = _rnd((cout,), seed + 5, F32)
    if c.res:
        d["res"] = _rnd((c.n,) + osp + (cout,), seed + 6, c.dtype)
    if c.op in ("act", "actT"):
        d["slope"] = torch.tensor([0.25])
    return d


def cpu_model(c, d):
    """A correct kernel, on the CPU: fp32 arithmetic on the rounded operands, one rounding of the stored result."""
    f = {k: v.float() for k, v in d.items()}
    if c.op == "wgrad":
        gin, gw = _grad(c.rank)
        part = gw(_nc(f["x"]), (c.cy, c.cx) + c.k, _nc(f["y"]), stride=c.s, padding=c.p)
        return f["dw0"] + part.permute((0,) + tuple(range(2, c.rank + 2)) + (1,)).reshape(c.cy, c.taps, c.cx)
    if c.op in ("fprop", "act"):
        out = _ncl(_conv(c.rank)(_nc(f["x"]), _w_nc(f["w"], c), f.get("b"), stride=c.s, padding=c.p))
    else:
        gin, _ = _grad(c.rank)
        out = _ncl(gin((c.n, c.cx) + c.xs, _w_nc(f["w"], c), _nc(f["x"]), stride=c.s, padding=c.p))
        if "b" in f:
            out = out + f["b"]
    if c.op in ("act", "actT"):
        out = torch.where(out >= 0, out, f["slope"] * out)
    if "res" in f:
        out = out + f["res"]
    return out.to(c.dtype)


def stats_chain(c, sms):
    """Longest fp32 chain of the fused statistics.  The halo engines walk tiles blockIdx.x, + gridDim.x, ... with
    gridDim.x = min(tiles, SMs) and add each tile's values into the CTA's shared-memory slots: at most
    ceil(tiles / grid) tiles of 128 pixels (512 X pixels in the pixel-shuffle and stride-2 data-gradient modes).  Other
    engines (and these cases with the halo engines switched off): every pixel."""
    if FALLBACK or c.engine not in ("halo", "halo_s2") or not c.stats:
        return None
    ysp = c.ys
    tiles = c.n * -(-ysp[0] // 16) * -(-ysp[1] // 8)
    if c.engine == "halo" and c.op == "bprop" and c.cx > 1:      # data gradient: tiles on the X grid
        tiles = c.n * -(-c.xs[0] // 16) * -(-c.xs[1] // 8)
    per = 512 if c.op == "bprop" and c.s == 2 else 128
    return per * -(-tiles // min(tiles, sms)) + 8


def check_case(c, d, got, route, stats=None, dev="cpu", sms=148):
    """Element-wise check of ``got`` against the fp64 reference of case ``c`` on operands ``d``; returns max err / bound."""
    dd = {k: v.to(dev) for k, v in d.items()}
    ref, part = reference(c, dd)
    S, S_part = reference(c, dd, absolute=True)
    u_out = U_OUT[F32] if c.op == "wgrad" else U_OUT[c.dtype]
    bnd = bound_of(c, dd, route, ref, part, S, S_part, u_out)
    tile, stride = c.tile, 1
    if tile is None and c.engine == "tapgemm" and c.op != "wgrad":
        # data gradients of stride-2 layers tile each output-parity class on its own grid of ceil(extent / 2)
        stride = c.s if c.op in ("bprop", "actT") else 1
        osp = tuple(-(-v // stride) for v in c.out_grid()[0])
        lw, lh, ld = tapgemm_tile(osp[-1], osp[-2], osp[0] if c.rank == 3 else 1, c.n, c.rank == 3)
        tile = ((1 << ld,) if c.rank == 3 else ()) + (1 << lh, 1 << lw)
    names = ["cy", "tap", "cx"] if c.op == "wgrad" else None
    worst = check_elementwise(got.to(dev), ref, bnd, c.id, tile=None if c.op == "wgrad" else tile, names=names,
                              tile_stride=stride)
    if stats is not None:
        worst = max(worst, check_stats(stats.to(dev), got.to(dev), c.id, stats_chain(c, sms)))
    return worst


# ------------------------------------------------------------------------------------------------ CPU self-tests
@pytest.mark.parametrize("c", ALL, ids=lambda c: c.id)
def test_checker_accepts_correct_model(c):
    """A kernel that computes in fp32 and rounds once passes the bound at every table shape."""
    d = make_operands(c)
    got = cpu_model(c, d)
    stats = None
    if c.stats:
        v = got.double().reshape(-1, got.shape[-1])
        stats = torch.cat([v.float().sum(0).double(), (v.float() * v.float()).sum(0).double()])
    assert check_case(c, d, got, c.route, stats) <= 1.0


SELF = Case("selftest", "fprop", 2, 2, 16, 32, (20, 28), route=TF, stats=True, tile=HALO_TILE)
SELF_W = Case("selftest", "wgrad", 2, 3, 16, 32, (20, 28), route=TW, tile=HALO_TILE)


def _fault(name):
    c = SELF
    d = make_operands(c)
    got = cpu_model(c, d).float()
    oh, ow = c.ys
    th, tw = HALO_TILE
    r0, c0 = (oh - 1) // th * th, (ow - 1) // tw * tw           # first row / column of the last (ragged) tile
    if name == "missing_tap":                 # tap (0, 0) dropped at the last pixel, in all channels
        i, r, q = c.n - 1, oh - 1, ow - 1
        got[i, r, q] -= d["x"].float()[i, r - 1, q - 1] @ d["w"].float()[:, 0, :].t()
    elif name == "bias_last_tile_row":
        got[:, r0:] -= d["b"]
    elif name == "last_tile_column_shifted":
        got[:, :, c0:] = got[:, :, c0 - 1:ow - 1].clone()
    elif name == "one_channel_one_tile":
        got[0, th:2 * th, tw:2 * tw, 5] *= 1.01
    return c, d, got.to(c.dtype)


@pytest.mark.parametrize("fault", ["missing_tap", "bias_last_tile_row", "last_tile_column_shifted",
                                   "one_channel_one_tile"])
def test_checker_rejects_output_fault(fault):
    c, d, got = _fault(fault)
    with pytest.raises(AssertionError, match="tile"):
        check_case(c, d, got, c.route)


def test_checker_rejects_statistics_without_last_tile():
    c = SELF
    d = make_operands(c)
    got = cpu_model(c, d)
    v = got.double()
    oh, ow = c.ys
    r0, c0 = (oh - 1) // 16 * 16, (ow - 1) // 8 * 8
    keep = torch.ones(v.shape[:-1], dtype=torch.bool)
    keep[c.n - 1, r0:, c0:] = False                            # the last tile of the last image
    vk = v[keep]
    stats = torch.cat([vk.sum(0), (vk * vk).sum(0)])
    with pytest.raises(AssertionError, match="channel sums"):
        check_case(c, d, got, c.route, stats)
    full = v.reshape(-1, v.shape[-1])
    assert check_case(c, d, got, c.route, torch.cat([full.sum(0), (full * full).sum(0)])) <= 1.0


@pytest.mark.parametrize("fault", ["last_partial_tile", "last_image"])
def test_checker_rejects_weight_gradient_fault(fault):
    c = SELF_W
    d = make_operands(c)
    y = d["y"].clone()
    oh, ow = c.ys
    if fault == "last_image":
        y[c.n - 1] = 0
    else:
        y[c.n - 1, (oh - 1) // 16 * 16:, (ow - 1) // 8 * 8:] = 0
    assert check_case(c, d, cpu_model(c, d), c.route) <= 1.0
    with pytest.raises(AssertionError, match="cy="):
        check_case(c, d, cpu_model(c, dict(d, y=y)), c.route)


@pytest.mark.parametrize("fault", ["missing_row", "missing_last_tile"])
def test_checker_rejects_weight_gradient_fault_at_two_to_the_20_pixels(fault):
    """The exact (integer) cases on both sides of wgrad_kernel's small split see one missing row or 64-pixel tile."""
    c = next(c for c in WGRAD if c.exact)
    d = make_operands(c)
    assert check_case(c, d, cpu_model(c, d), c.route) == 0.0
    y = d["y"].clone()
    if fault == "missing_row":
        y[0, c.ys[0] - 1] = 0
    else:
        lw, lh, _ = tapgemm_tile(c.ys[1], c.ys[0], 1, c.n, False, 64)
        y[0, -(1 << lh):, -(1 << lw):] = 0
    with pytest.raises(AssertionError, match="cy="):
        check_case(c, d, cpu_model(c, dict(d, y=y)), c.route)


def test_checker_rejects_statistics_without_last_tile_at_ring_shape():
    """At 3 x 256 x 256 (1 536 halo tiles on 148 SMs) the per-CTA chain bound still sees one missing tile."""
    c = next(c for c in HALO if c.stats and c.n == 3 and c.ys == (256, 256))
    got = cpu_model(c, make_operands(c))
    v = got.double()
    keep = torch.ones(v.shape[:-1], dtype=torch.bool)
    keep[c.n - 1, -16:, -8:] = False
    full, vk = v.reshape(-1, v.shape[-1]), v[keep]
    chain = stats_chain(c, 148)
    assert check_stats(torch.cat([full.sum(0), (full * full).sum(0)]), got, c.id, chain) <= 1.0
    with pytest.raises(AssertionError, match="channel sums"):
        check_stats(torch.cat([vk.sum(0), (vk * vk).sum(0)]), got, c.id, chain)


# ------------------------------------------------------------------------------------------------ GPU cases
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


def _slice(host, margin_lo=8, margin_hi=8, fill=FILL, extra_image=True):
    """host (N *S C) -> device view of the same values inside a buffer with channel margins and one trailing image of
    ``fill``.  Margins of 8 keep 16-byte alignment and pixel strides % 8 of the original channel count."""
    n, c = host.shape[0], host.shape[-1]
    big = torch.full((n + (1 if extra_image else 0),) + tuple(host.shape[1:-1]) + (margin_lo + c + margin_hi,), fill,
                     dtype=host.dtype, device="cuda")
    view = big[:n, ..., margin_lo:margin_lo + c]
    view.copy_(host.to("cuda"))
    return big, view


def _operand(host):
    """Channel slice of a wider buffer; a one-channel operand stays contiguous (the one-channel engines read it as a
    plain image) with only the trailing image of FILL after it."""
    return _slice(host, 0, 0)[1] if host.shape[-1] == 1 else _slice(host)[1]


def run_gpu(c, d, routes, o_off=16):
    """o_off: byte offset of the output view in its buffer -- 32 lets the engines take their 32-byte store path
    (``wide``: 32-byte aligned, pixel stride % 16 == 0), 16 the narrow one."""
    from mpgan import ops
    spec = ops.ConvSpec(c.rank, c.cx, c.cy, c.k[0], c.s, c.p)
    x = _operand(d["x"])
    w = d["w"].cuda()
    b = d["b"].cuda() if "b" in d else None
    osp, cout = c.out_grid()
    keep = []
    if c.op == "wgrad":
        y = _slice(d["y"], 0, 0)[1] if c.cx == 1 and c.cy == 1 else _slice(d["y"])[1]
        # dw is dense [cy][taps][cx] (no stride argument): sentinels before it and one weight row of them after it
        m = c.cy * c.taps * c.cx
        big = torch.full((64 + m + c.taps * c.cx,), SENT, dtype=F32, device="cuda")
        dw = big[64:64 + m].view(c.cy, c.taps, c.cx)
        dw.copy_(d["dw0"].cuda())
        keep.append((big, (slice(64, 64 + m),)))
        routes.clear()
        ops.conv_wgrad(spec, x, y, dw, **c.kw)
        torch.cuda.synchronize()
        return dw.cpu(), None, keep
    # the output: a view with channel margins (where the engine takes a pixel stride) and one trailing image of sentinels
    m = o_off * 8 // torch.finfo(c.dtype).bits if cout > 1 else 0
    bigo = torch.full((c.n + 1,) + osp + (cout + 2 * m,), SENT, dtype=c.dtype, device="cuda")
    out = bigo[:c.n, ..., m:m + cout]
    keep.append((bigo, (slice(0, c.n),) + (slice(None),) * len(osp) + (slice(m, m + cout),)))
    stats = None
    if c.stats:
        bigs = torch.full((2 * cout + 16,), SENT, dtype=torch.float64, device="cuda")
        stats = bigs[8:8 + 2 * cout]
        stats.zero_()
        keep.append((bigs, (slice(8, 8 + 2 * cout),)))
    res = None
    if c.res == "fused":
        res = _operand(d["res"])
    elif c.res == "unaligned":      # pixel stride not a multiple of 8, 2-byte offset: no engine can fuse it
        res = _slice(d["res"], margin_lo=1, margin_hi=2, fill=FILL)[1]
    routes.clear()
    if c.op == "fprop":
        _, fused = ops.conv_fprop(spec, x, w, b, out=out, stats=stats, **c.kw)
    elif c.op == "bprop":
        wt = None
        if c.cx > 1 and c.dtype == BF:
            wt = torch.empty(w.numel(), dtype=BF, device="cuda")
            ops.weight_transpose(w, wt, c.cy, c.taps, c.cx)
        routes.clear()
        _, fused = ops.conv_bprop(spec, x, w, wt, b, xs=c.xs, out=out, stats=stats, res=res, **c.kw)
    else:
        slope = d["slope"].cuda()
        if c.op == "act":
            r = ops.conv_act(spec, x, w, b, slope, res=res, out=out)
        else:
            wt = torch.empty(w.numel(), dtype=BF, device="cuda")
            ops.weight_transpose(w, wt, c.cy, c.taps, c.cx)
            spec_t = ops.ConvSpec(c.rank, c.cx, c.cy, c.k[0], c.s, c.p, transposed=True,
                                  output_padding=c.xs[0] - ((c.ys[0] - 1) * c.s - 2 * c.p + c.k[0]))
            routes.clear()
            r = ops.conv_act(spec_t, x, wt, b, slope, res=res, out=out)
        assert r is not None, f"{c.id}: conv_act reports the layer as not covered"
        fused = False
    torch.cuda.synchronize()
    last = [r for r in routes if r != "add_copy"]
    expect_fused = bool(c.stats) and bool(last) and last[-1] not in NOT_FUSED
    assert fused == expect_fused, f"{c.id}: fused statistics {fused}, expected {expect_fused} on route {routes}"
    if c.stats and not fused:
        assert torch.all(stats == 0), f"{c.id}: statistics written although the call reports them unfused"
        stats = None
    return out.cpu(), (stats.cpu() if stats is not None else None), keep


def _sentinels_intact(c, keep):
    for big, inner in keep:
        mask = torch.ones(big.shape, dtype=torch.bool, device=big.device)
        mask[inner] = False
        outside = big[mask]
        assert torch.all(outside == SENT), \
            f"{c.id}: {int((outside != SENT).sum())} elements outside the output view were written"


# bf16 outputs with 16 | channels run twice: 32-byte aligned (the 256-bit store path every contiguous production
# output takes) and 16 bytes off (the 128-bit path); the rest once, 16 bytes off
GPU_CASES = [(c, o) for c in ALL
             for o in ((32, 16) if c.op != "wgrad" and c.dtype == BF and c.out_grid()[1] % 16 == 0 else (16,))]


@pytest.mark.gpu
@pytest.mark.parametrize("c,o_off", GPU_CASES, ids=[f"{c.id}-o{o}" for c, o in GPU_CASES])
def test_engine_elementwise(c, o_off, routes):
    d = make_operands(c)
    got, stats, keep = run_gpu(c, d, routes, o_off)
    assert tuple(routes) == c.expected(), f"{c.id}: route {routes}, expected {list(c.expected())}"
    _sentinels_intact(c, keep)
    worst = check_case(c, d, got, routes, stats, dev="cuda", sms=torch.cuda.get_device_properties(0).multi_processor_count)
    print(f"[conv-engine] {'fallback' if FALLBACK else 'default'} {c.engine} {c.id}-o{o_off} max|err|/bound {worst:.4f}")


@pytest.mark.gpu
def test_fallback_engines_in_child_process():
    """The same cases with every MPGAN_NO_* switch set (read once per process, hence a child): tap-GEMM, wgrad_kernel,
    the pixel-at-a-time one-channel kernels and the generic paths at the specialised engines' shapes."""
    if FALLBACK:
        pytest.skip("this is the child run")
    env = dict(os.environ, **{s: "1" for s in SWITCHES}, **{CHILD: "1"})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
        ["-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-p", "no:cacheprovider", "-rA"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("[conv-engine]")]
    print("\n".join(lines))
    assert r.returncode == 0, "fallback run failed:\n" + r.stdout[-6000:] + r.stderr[-3000:]
