"""Tensor-level wrappers over the C ABI (include/mpgan.h).  torch is used for device memory and streams only.

Activation tensors are channels-last ``(N, *spatial, C)`` with unit channel stride and pixel-linear leading
strides (a channel slice of a wider concat buffer is fine).
"""
import bisect
import ctypes
import os

import torch

from . import _lib
from ._lib import ACT_LEAKY, ACT_NONE, ACT_PRELU, ACT_TANH, BF16, F32, ConvGeom, check

_NULL = None


def _stream():
    return torch.cuda.current_stream().cuda_stream


def dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {t.dtype}")


def ptr(t):
    return None if t is None else t.data_ptr()


def ld(t):
    return t.stride(-2) if t.dim() >= 2 else t.shape[-1]


def pixels(t):
    return t.numel() // t.shape[-1]


def check_act(t, what="activation"):
    if not t.is_cuda:
        raise RuntimeError(f"{what} must be a CUDA tensor: the mpgan kernels have no CPU path")
    if t.stride(-1) != 1 and t.shape[-1] != 1:
        raise RuntimeError(f"{what}: channel stride must be 1, got strides {t.stride()}")
    l = ld(t)
    exp = l
    for i in range(t.dim() - 2, -1, -1):
        if t.shape[i] != 1 and t.stride(i) != exp:
            raise RuntimeError(f"{what}: not pixel-linear, shape {tuple(t.shape)} strides {t.stride()}")
        exp *= t.shape[i]
    return t


class ConvSpec:
    """Geometry of one Conv / ConvTranspose layer in terms of its underlying convolution X -> Y."""

    def __init__(self, rank, cx, cy, k, stride, pad, transposed=False, output_padding=0):
        self.rank, self.cx, self.cy = rank, cx, cy
        self.k, self.stride, self.pad = (k,) * rank, (stride,) * rank, (pad,) * rank
        self.transposed, self.output_padding = transposed, output_padding
        self.taps = k ** rank

    @classmethod
    def from_module(cls, m):
        import torch.nn as nn
        transposed = isinstance(m, (nn.ConvTranspose2d, nn.ConvTranspose3d))
        rank = len(m.kernel_size)
        k, s, p = m.kernel_size[0], m.stride[0], m.padding[0]
        assert all(v == k for v in m.kernel_size) and all(v == s for v in m.stride) and all(v == p for v in m.padding)
        if transposed:  # ConvT(in, out): in lives on the Y grid, out on the X grid
            return cls(rank, m.out_channels, m.in_channels, k, s, p, True, m.output_padding[0])
        return cls(rank, m.in_channels, m.out_channels, k, s, p, False)

    def y_of_x(self, xs):
        return tuple((v + 2 * p - k) // s + 1 for v, k, s, p in zip(xs, self.k, self.stride, self.pad))

    def x_of_y(self, ys):
        return tuple((v - 1) * s - 2 * p + k + self.output_padding
                     for v, k, s, p in zip(ys, self.k, self.stride, self.pad))

    def geom(self, n, xs, ys):
        g = ConvGeom()
        g.rank, g.n, g.cx, g.cy = self.rank, n, self.cx, self.cy
        pad3 = 3 - self.rank
        for i in range(3):
            j = i - pad3
            g.xs[i] = xs[j] if j >= 0 else 1
            g.ys[i] = ys[j] if j >= 0 else 1
            g.k[i] = self.k[j] if j >= 0 else 1
            g.stride[i] = self.stride[j] if j >= 0 else 1
            g.pad[i] = self.pad[j] if j >= 0 else 0
        return g


_C1VOL = os.environ.get("MPGAN_NO_C1VOL", "0") != "1"
_SPEC_1X1X1 = {}


def _spec_1x1x1(cx, cy):
    if (cx, cy) not in _SPEC_1X1X1:
        _SPEC_1X1X1[(cx, cy)] = ConvSpec(3, cx, cy, 1, 1, 0)
    return _SPEC_1X1X1[(cx, cy)]


def _vol_c1(spec):
    """Rank-3 3x3x3 layer with ONE X-grid channel (csrc/conv_c1vol.cu)."""
    return (_C1VOL and spec.rank == 3 and spec.cx == 1 and spec.k == (3, 3, 3) and spec.stride[0] in (1, 2)
            and spec.pad[0] in (0, 1))


def _i3(v):
    return (ctypes.c_int32 * 3)(*v)


def tc_supported(geom, direction):
    return bool(_lib.load().mpgan_tc_supported(ctypes.byref(geom), direction))


# ---------------------------------------------------------------------------------------------------------
# convolution.  w: OTI [cy][taps][cx] in the activation dtype; wt: transposed bf16 shadow (tcgen05 bprop)
# ---------------------------------------------------------------------------------------------------------
def conv_fprop(spec, x, w, bias, out=None, stats=None, use_tc=True, use_c1=True):
    """X-grid tensor -> Y-grid tensor (Conv forward; ConvTranspose data gradient)."""
    lib = _lib.require_device()
    check_act(x, "conv input")
    n, xs = x.shape[0], tuple(x.shape[1:-1])
    ys = spec.y_of_x(xs)
    if out is None:
        out = torch.empty((n,) + ys + (spec.cy,), dtype=x.dtype, device=x.device)
    check_act(out, "conv output")
    g = spec.geom(n, xs, ys)
    if use_c1 and _vol_c1(spec) and x.is_contiguous():
        if spec.cy == 1 and spec.stride[0] == 1 and spec.pad[0] == 1 and out.is_contiguous():
            check(lib.mpgan_stencil27(dt(x), 0, ptr(x), n, xs[0], xs[1], xs[2], ptr(w), ptr(bias), None, ptr(out), _stream()),
                  "stencil27")
            return out, False
        if use_tc and x.dtype == torch.bfloat16 and spec.cy % 16 == 0 and spec.cy <= 512:
            # one input channel: im2col (27 taps -> 32 "channels") + the tcgen05 1x1x1 convolution (fused statistics)
            xcol = torch.empty((n,) + ys + (32,), dtype=torch.bfloat16, device=x.device)
            check(lib.mpgan_im2col_c1_vol(ptr(x), n, _i3(xs), _i3(ys), spec.stride[0], spec.pad[0], ptr(xcol), _stream()),
                  "im2col_c1_vol")
            w32 = torch.zeros((spec.cy, 32), dtype=torch.bfloat16, device=x.device)
            w32[:, :27].copy_(w.reshape(spec.cy, 27))
            g1 = _spec_1x1x1(32, spec.cy).geom(n, ys, ys)
            check(lib.mpgan_tc_conv_fprop(ctypes.byref(g1), ptr(xcol), 32, ptr(w32), ptr(bias), ptr(out), ld(out), ptr(stats),
                                          _stream()), "tc_conv_fprop(im2col vol)")
            return out, stats is not None
    if use_tc and x.dtype == torch.bfloat16 and tc_supported(g, 0):
        check(lib.mpgan_tc_conv_fprop(ctypes.byref(g), ptr(x), ld(x), ptr(w), ptr(bias), ptr(out), ld(out), ptr(stats),
                                      _stream()), "tc_conv_fprop")
        return out, stats is not None
    if use_c1 and lib.mpgan_c1_supported(ctypes.byref(g), 0):
        check(lib.mpgan_c1_conv_fprop(ctypes.byref(g), dt(x), ptr(x), ld(x), ptr(w), ptr(bias), ptr(out), ld(out),
                                      ptr(stats), _stream()), "c1_conv_fprop")
        return out, stats is not None
    check(lib.mpgan_conv_fprop(ctypes.byref(g), dt(x), ptr(x), ld(x), ptr(w), ptr(bias), ptr(out), ld(out), _stream()),
          "conv_fprop")
    return out, False


def conv_act(spec, x, w, bias, slope, res=None, out=None):
    """Inference-mode fused layer on the tcgen05 path: out = prelu(conv(x, w) + bias) + res with BatchNorm already
    folded into (w, bias).  Transposed layers take the transposed weights.  Returns None when the layer is not covered
    (the caller then runs the unfused kernels)."""
    lib = _lib.require_device()
    if x.dtype != torch.bfloat16:
        return None
    n, ins = x.shape[0], tuple(x.shape[1:-1])
    if spec.transposed:
        xs, ys, direction, cout = spec.x_of_y(ins), ins, 1, spec.cx
    else:
        xs, ys, direction, cout = ins, spec.y_of_x(ins), 0, spec.cy
    g = spec.geom(n, xs, ys)
    if (not spec.transposed and spec.cx == 1 and spec.rank == 2 and res is None and spec.cy % 8 == 0 and x.is_contiguous()
            and os.environ.get("MPGAN_NO_C1ACT", "0") != "1"):
        # one input channel (the UNet's first layer): the run-based CUDA-core kernel with the PReLU in its store path
        o = out if out is not None else torch.empty((n,) + tuple(ys) + (cout,), dtype=x.dtype, device=x.device)
        rc = lib.mpgan_c1_conv_act(ctypes.byref(g), dt(x), ptr(x), ld(x), ptr(w), ptr(bias), ptr(slope), ptr(o), ld(o), _stream())
        if rc == 0:
            return o
        if rc != -2:
            check(rc, "c1_conv_act")
    if not tc_supported(g, direction):
        return None
    if out is None:
        out = torch.empty((n,) + tuple(xs if spec.transposed else ys) + (cout,), dtype=x.dtype, device=x.device)
    if res is not None and (res.dtype != torch.bfloat16 or ld(res) % 8 or res.data_ptr() % 16):
        return None
    check(lib.mpgan_tc_conv_act(ctypes.byref(g), direction, ptr(x), ld(x), ptr(w), ptr(bias), ptr(slope), ptr(res),
                                ld(res) if res is not None else 0, ptr(out), ld(out), _stream()), "tc_conv_act")
    return out


_C1OUT = os.environ.get("MPGAN_NO_C1OUT", "0") != "1"
_CONVT1 = os.environ.get("MPGAN_NO_CONVT1", "0") != "1"


def conv_bprop(spec, y, w, wt, bias, xs=None, out=None, stats=None, use_tc=True, use_c1=True, res=None,
               force_c1out=False):
    """Y-grid tensor -> X-grid tensor (ConvTranspose forward; Conv data gradient).  ``res``: an X-grid tensor added
    to the result (gradient accumulation of a residual / skip branch) -- fused into the tcgen05 epilogue, otherwise
    one add kernel after the convolution."""
    lib = _lib.require_device()
    check_act(y, "conv input")
    n, ys = y.shape[0], tuple(y.shape[1:-1])
    if xs is None:
        xs = spec.x_of_y(ys)
    if out is None:
        out = torch.empty((n,) + tuple(xs) + (spec.cx,), dtype=y.dtype, device=y.device)
    check_act(out, "conv output")
    g = spec.geom(n, xs, ys)
    if use_c1 and _vol_c1(spec) and out.is_contiguous() and w is not None and (res is None or (res.is_contiguous() and res.dtype == out.dtype)):
        if (spec.cy == 1 and spec.stride[0] == 1 and spec.pad[0] == 1 and y.is_contiguous() and tuple(xs) == ys
                and w.dtype == y.dtype):
            check(lib.mpgan_stencil27(dt(y), 1, ptr(y), n, ys[0], ys[1], ys[2], ptr(w), ptr(bias), ptr(res), ptr(out), _stream()),
                  "stencil27")
            return out, False
        if (use_tc and y.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and spec.cy % 16 == 0 and ld(y) % 8 == 0
                and y.data_ptr() % 16 == 0):
            # one output channel: per-tap partial products through the tcgen05 1x1x1 convolution, then a 27-point gather
            wt32 = torch.zeros((32, spec.cy), dtype=torch.bfloat16, device=y.device)
            wt32[:27].copy_(w.reshape(spec.cy, 27).t())
            part = torch.empty((n,) + ys + (32,), dtype=torch.bfloat16, device=y.device)
            g1 = _spec_1x1x1(spec.cy, 32).geom(n, ys, ys)
            check(lib.mpgan_tc_conv_fprop(ctypes.byref(g1), ptr(y), ld(y), ptr(wt32), None, ptr(part), 32, None, _stream()),
                  "tc_conv_fprop(col2im vol)")
            check(lib.mpgan_col2im_c1_vol(ptr(part), n, _i3(xs), _i3(ys), spec.stride[0], spec.pad[0], ptr(bias), ptr(res),
                                          ptr(out), _stream()), "col2im_c1_vol")
            return out, False
    if (use_tc and use_c1 and w is not None and w.dtype == torch.bfloat16 and y.dtype == torch.bfloat16 and spec.rank == 2 and spec.cx == 1
            and spec.k == (3, 3) and spec.stride == (1, 1) and spec.cy in (16, 32, 64, 128) and stats is None
            and bias is None and ld(y) % 8 == 0 and (res is None or res.dtype == torch.bfloat16) and _C1OUT
            and (force_c1out or n * xs[0] * xs[1] > (1 << 20))):
        # one input channel, large layer (D layer 1): the halo tcgen05 kernel with the weights zero-padded to 16 columns
        wt16 = torch.zeros((16, 9, spec.cy), dtype=torch.bfloat16, device=y.device)
        wt16[0].copy_(w.reshape(spec.cy, 9).t())   # [cy][9][1] -> transposed [9][cy]
        check(lib.mpgan_tc_conv_bprop_c1out(ctypes.byref(g), ptr(y), ld(y), ptr(wt16), ptr(out), ld(out), ptr(res),
                                            ld(res) if res is not None else 0, _stream()), "tc_conv_bprop_c1out")
        return out, False
    if (use_tc and use_c1 and w is not None and w.dtype == torch.bfloat16 and y.dtype == torch.bfloat16 and spec.rank == 2
            and spec.cx == 1 and spec.k == (3, 3) and spec.stride == (2, 2) and spec.pad == (1, 1) and spec.cy in (16, 32, 64)
            and tuple(xs) == (2 * ys[0], 2 * ys[1]) and ld(y) % 8 == 0 and out.is_contiguous() and _CONVT1
            and ys[1] % 8 == 0):
        # stride-2 ConvTranspose / data gradient into one channel: halo tcgen05 kernel in pixel-shuffle mode
        check(lib.mpgan_tc_convt_to1(ctypes.byref(g), ptr(y), ld(y), ptr(w), ptr(bias), ptr(out), ptr(stats), _stream()),
              "tc_convt_to1")
        if res is not None:
            add_copy(out, res, out)
        return out, stats is not None
    if use_tc and wt is not None and y.dtype == torch.bfloat16 and tc_supported(g, 1):
        if res is not None and res.dtype == torch.bfloat16 and ld(res) % 8 == 0 and res.data_ptr() % 16 == 0:
            check(lib.mpgan_tc_conv_bprop_res(ctypes.byref(g), ptr(y), ld(y), ptr(wt), ptr(bias), ptr(out), ld(out),
                                              ptr(res), ld(res), ptr(stats), _stream()), "tc_conv_bprop_res")
            return out, stats is not None
        check(lib.mpgan_tc_conv_bprop(ctypes.byref(g), ptr(y), ld(y), ptr(wt), ptr(bias), ptr(out), ld(out), ptr(stats),
                                      _stream()), "tc_conv_bprop")
        if res is not None:
            add_copy(out, res, out)
        return out, stats is not None
    if use_c1 and lib.mpgan_c1_supported(ctypes.byref(g), 1):
        check(lib.mpgan_c1_conv_bprop(ctypes.byref(g), dt(y), ptr(y), ld(y), ptr(w), ptr(bias), ptr(out), ld(out),
                                      ptr(stats), _stream()), "c1_conv_bprop")
        if res is not None:
            add_copy(out, res, out)
        return out, stats is not None
    check(lib.mpgan_conv_bprop(ctypes.byref(g), dt(y), ptr(y), ld(y), ptr(w), ptr(bias), ptr(out), ld(out), _stream()),
          "conv_bprop")
    if res is not None:
        add_copy(out, res, out)
    return out, False


_C1COL = os.environ.get("MPGAN_NO_C1COL", "0") != "1"
_SPEC_1X1 = {}


def _spec_1x1(cx, cy):
    if (cx, cy) not in _SPEC_1X1:
        _SPEC_1X1[(cx, cy)] = ConvSpec(2, cx, cy, 1, 1, 0)
    return _SPEC_1X1[(cx, cy)]


def conv_wgrad(spec, x, y, dw, use_tc=True, use_c1=True, force_c1col=False):
    """dw[cy][taps][cx] (fp32, accumulates) from the X-grid tensor and the Y-grid tensor."""
    lib = _lib.require_device()
    check_act(x), check_act(y)
    n, xs, ys = x.shape[0], tuple(x.shape[1:-1]), tuple(y.shape[1:-1])
    g = spec.geom(n, xs, ys)
    assert dw.dtype == torch.float32
    if use_c1 and _vol_c1(spec) and x.is_contiguous():
        if spec.cy == 1 and spec.stride[0] == 1 and spec.pad[0] == 1 and y.is_contiguous() and x.dtype == y.dtype:
            check(lib.mpgan_stencil27_wgrad(dt(x), ptr(x), ptr(y), n, xs[0], xs[1], xs[2], ptr(dw), None, _stream()),
                  "stencil27_wgrad")
            return
        if (use_tc and x.dtype == torch.bfloat16 and y.dtype == torch.bfloat16 and spec.cy % 16 == 0 and ld(y) % 8 == 0
                and y.data_ptr() % 16 == 0):
            xcol = torch.empty((n,) + ys + (32,), dtype=torch.bfloat16, device=x.device)
            check(lib.mpgan_im2col_c1_vol(ptr(x), n, _i3(xs), _i3(ys), spec.stride[0], spec.pad[0], ptr(xcol), _stream()),
                  "im2col_c1_vol")
            dw32 = torch.zeros((spec.cy, 32), dtype=torch.float32, device=x.device)
            g1 = _spec_1x1x1(32, spec.cy).geom(n, ys, ys)
            check(lib.mpgan_tc_conv_wgrad(ctypes.byref(g1), ptr(xcol), 32, ptr(y), ld(y), ptr(dw32), None, 0, _stream()),
                  "tc_conv_wgrad(im2col vol)")
            check(lib.mpgan_fold_dw32(ptr(dw32), spec.cy, ptr(dw), _stream()), "fold_dw32")
            return
    if (use_tc and use_c1 and x.dtype == torch.bfloat16 and spec.rank == 2 and spec.cx == 1 and spec.k == (3, 3)
            and spec.cy % 16 == 0 and spec.cy <= 256 and ld(x) == 1 and x.is_contiguous() and _C1COL
            and (force_c1col or n * ys[0] * ys[1] > (1 << 20))):   # measured: a win for D layer 1, not for G's 0.5M-pixel layers
        # one input channel: im2col (9 taps -> 16 "channels") + the tcgen05 weight gradient of the equivalent 1x1 layer
        xcol = torch.empty((n,) + ys + (16,), dtype=torch.bfloat16, device=x.device)
        check(lib.mpgan_im2col_c1(ptr(x), n, xs[0], xs[1], ys[0], ys[1], spec.stride[0], spec.pad[0], ptr(xcol),
                                  _stream()), "im2col_c1")
        dw16 = torch.zeros((spec.cy, 16), dtype=torch.float32, device=x.device)
        g1 = _spec_1x1(16, spec.cy).geom(n, ys, ys)
        check(lib.mpgan_tc_conv_wgrad(ctypes.byref(g1), ptr(xcol), 16, ptr(y), ld(y), ptr(dw16), None, 0, _stream()),
              "tc_conv_wgrad(im2col)")
        check(lib.mpgan_fold_dw16(ptr(dw16), spec.cy, ptr(dw), _stream()), "fold_dw16")
    elif use_tc and x.dtype == torch.bfloat16 and tc_supported(g, 2):
        check(lib.mpgan_tc_conv_wgrad(ctypes.byref(g), ptr(x), ld(x), ptr(y), ld(y), ptr(dw), None, 0, _stream()),
              "tc_conv_wgrad")
    elif use_c1 and lib.mpgan_c1_supported(ctypes.byref(g), 2):
        check(lib.mpgan_c1_conv_wgrad(ctypes.byref(g), dt(x), ptr(x), ld(x), ptr(y), ld(y), ptr(dw), _stream()),
              "c1_conv_wgrad")
    else:
        check(lib.mpgan_conv_wgrad(ctypes.byref(g), dt(x), ptr(x), ld(x), ptr(y), ld(y), ptr(dw), _stream()),
              "conv_wgrad")


def colsum(x, out):
    lib = _lib.require_device()
    check(lib.mpgan_colsum(dt(x), ptr(x), ld(x), pixels(x), x.shape[-1], ptr(out), _stream()), "colsum")


# ---------------------------------------------------------------------------------------------------------
# batch norm + activation
# ---------------------------------------------------------------------------------------------------------
def bn_stats(x, stats):
    lib = _lib.require_device()
    check(lib.mpgan_bn_stats(dt(x), ptr(x), ld(x), pixels(x), x.shape[-1], ptr(stats), _stream()), "bn_stats")


def bn_finalize(stats, npix, bn, training, mean, invstd, scale, shift):
    lib = _lib.require_device()
    mom = 0.1 if bn.momentum is None else bn.momentum
    check(lib.mpgan_bn_finalize(ptr(stats), npix, bn.num_features, ptr(bn.weight), ptr(bn.bias), bn.eps, mom,
                                1 if training else 0, ptr(bn.running_mean), ptr(bn.running_var),
                                ptr(bn.num_batches_tracked), ptr(mean), ptr(invstd), ptr(scale), ptr(shift),
                                _stream()), "bn_finalize")


def bn_act_apply(x, scale, shift, act, alpha, leaky, res, out):
    lib = _lib.require_device()
    check_act(x), check_act(out)
    check(lib.mpgan_bn_act_apply(dt(x), ptr(x), ld(x), pixels(x), x.shape[-1], ptr(scale), ptr(shift), act,
                                 ptr(alpha), leaky, ptr(res), ld(res) if res is not None else 0, ptr(out), ld(out),
                                 _stream()), "bn_act_apply")
    return out


def bn_train_apply(x, stats, bn, saved, act, alpha, leaky, res, out):
    """Training-mode BatchNorm finalize + normalise + activation (+ residual) in one launch.
    saved: (4, C) fp32 buffer receiving mean, invstd, scale, shift."""
    lib = _lib.require_device()
    check_act(x), check_act(out)
    mom = 0.1 if bn.momentum is None else bn.momentum
    check(lib.mpgan_bn_train_apply(dt(x), ptr(x), ld(x), pixels(x), x.shape[-1], ptr(stats), ptr(bn.weight),
                                   ptr(bn.bias), bn.eps, mom, ptr(bn.running_mean), ptr(bn.running_var),
                                   ptr(bn.num_batches_tracked), ptr(saved[0]), ptr(saved[1]), ptr(saved[2]),
                                   ptr(saved[3]), act, ptr(alpha), leaky, ptr(res), ld(res) if res is not None else 0,
                                   ptr(out), ld(out), _stream()), "bn_train_apply")
    return out


def c1_tail_fwd(c, stats, bn, saved, alpha, w9, bias, want_h):
    """Fused UNet tail on a one-channel bf16 image (n, h, w, 1): returns (hmap or None, y).  ``stats=None``:
    evaluation mode -- ``saved[2]`` / ``saved[3]`` hold the scale / shift of the running statistics (``bn_finalize``)."""
    lib = _lib.require_device()
    assert c.dtype == torch.bfloat16 and c.is_contiguous() and c.shape[-1] == 1 and c.dim() == 4
    n, h, w = c.shape[0], c.shape[1], c.shape[2]
    hmap = torch.empty_like(c) if want_h else None
    y = torch.empty_like(c)
    mom = 0.1 if bn.momentum is None else bn.momentum
    check(lib.mpgan_c1_tail_fwd(ptr(c), n, h, w, ptr(stats), ptr(bn.weight), ptr(bn.bias), bn.eps, mom,
                                ptr(bn.running_mean), ptr(bn.running_var), ptr(bn.num_batches_tracked), ptr(saved[0]),
                                ptr(saved[1]), ptr(saved[2]), ptr(saved[3]), ptr(alpha), ptr(w9), ptr(bias), ptr(hmap),
                                ptr(y), _stream()), "c1_tail_fwd")
    return hmap, y


def c1_tail_bwd(dy, c, saved, bn, alpha, w9, sums, dgamma, dbeta, dalpha, dbias):
    """Backward of the fused UNet tail down to the ConvTranspose output: dc (gradient of the raw ConvTranspose
    output c) from dy (gradient of the tail's output).  Two launches: fused data-gradient + BatchNorm reduction, then
    the BatchNorm / PReLU backward apply."""
    lib = _lib.require_device()
    assert dy.dtype == torch.bfloat16 and dy.is_contiguous() and c.is_contiguous() and c.shape == dy.shape
    n, h, w = c.shape[0], c.shape[1], c.shape[2]
    mean, invstd, scale, shift = saved
    dh = torch.empty_like(c)
    check(lib.mpgan_c1_tail_bwd_reduce(ptr(dy), ptr(c), n, h, w, ptr(mean), ptr(invstd), ptr(scale), ptr(shift), ptr(alpha),
                                       ptr(w9), ptr(dh), ptr(sums), _stream()), "c1_tail_bwd_reduce")
    dc = torch.empty_like(c)
    check(lib.mpgan_bn_act_bwd_apply(dt(c), ptr(dh), ld(dh), ptr(c), ld(c), pixels(c), 1, ptr(mean), ptr(invstd),
                                     ptr(scale), ptr(shift), ACT_PRELU, ptr(alpha), 0.0, ptr(sums), ptr(dgamma),
                                     ptr(dbeta), ptr(dalpha), ptr(dbias), ptr(dc), ld(dc), _stream()), "bn_act_bwd_apply")
    return dc


def bn_act_bwd(dy, x, mean, invstd, scale, shift, act, alpha, leaky, sums, dgamma, dbeta, dalpha, dx, dbias=None):
    lib = _lib.require_device()
    check_act(dy), check_act(x), check_act(dx)
    c = x.shape[-1]
    check(lib.mpgan_bn_act_bwd_reduce(dt(x), ptr(dy), ld(dy), ptr(x), ld(x), pixels(x), c, ptr(mean), ptr(invstd),
                                      ptr(scale), ptr(shift), act, ptr(alpha), leaky, ptr(sums), _stream()),
          "bn_act_bwd_reduce")
    check(lib.mpgan_bn_act_bwd_apply(dt(x), ptr(dy), ld(dy), ptr(x), ld(x), pixels(x), c, ptr(mean), ptr(invstd),
                                     ptr(scale), ptr(shift), act, ptr(alpha), leaky, ptr(sums), ptr(dgamma),
                                     ptr(dbeta), ptr(dalpha), ptr(dbias), ptr(dx), ld(dx), _stream()), "bn_act_bwd_apply")
    return dx


def act_bwd(dy, z, act, leaky, dx):
    """dx = dy * act'(z) for a parameter-free activation (LeakyReLU backward on a saved pre-activation)."""
    lib = _lib.require_device()
    check_act(dy), check_act(z), check_act(dx)
    dummy = torch.zeros(1, dtype=torch.float64, device=z.device)
    check(lib.mpgan_bn_act_bwd_apply(dt(z), ptr(dy), ld(dy), ptr(z), ld(z), pixels(z), z.shape[-1], None, None, None,
                                     None, act, None, leaky, ptr(dummy), None, None, None, None, ptr(dx), ld(dx),
                                     _stream()), "act_bwd")
    return dx


# ---------------------------------------------------------------------------------------------------------
# elementwise
# ---------------------------------------------------------------------------------------------------------
def add_copy(a, b, out):
    """out = a (+ b) over channels-last tensors with independent pixel strides / dtypes (a, b same dtype)."""
    lib = _lib.require_device()
    check_act(a), check_act(out)
    if b is not None:
        check_act(b)
        assert b.dtype == a.dtype
    check(lib.mpgan_add_copy(dt(a), ptr(a), ld(a), ptr(b), ld(b) if b is not None else 0, dt(out), ptr(out), ld(out),
                             pixels(a), a.shape[-1], _stream()), "add_copy")
    return out


def tanh_fwd(x, out):
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous()
    check(lib.mpgan_tanh_fwd(dt(x), ptr(x), dt(out), ptr(out), x.numel(), _stream()), "tanh_fwd")
    return out


def tanh_bwd(dy, y, dx):
    lib = _lib.require_device()
    assert dy.is_contiguous() and y.is_contiguous() and dx.is_contiguous() and dy.dtype == y.dtype == dx.dtype
    check(lib.mpgan_tanh_bwd(dt(dy), ptr(dy), ptr(y), ptr(dx), dy.numel(), _stream()), "tanh_bwd")
    return dx


def cast(src, dst):
    lib = _lib.require_device()
    assert src.is_contiguous() and dst.is_contiguous() and src.numel() == dst.numel()
    check(lib.mpgan_cast(dt(src), ptr(src), dt(dst), ptr(dst), src.numel(), _stream()), "cast")
    return dst


def weight_transpose(src, dst, cy, taps, cx):
    lib = _lib.require_device()
    check(lib.mpgan_weight_transpose(dt(src), ptr(src), dt(dst), ptr(dst), cy, taps, cx, _stream()), "weight_transpose")
    return dst


def weight_transpose_batch(table, n, max_elems):
    """table: (n, 5) int64 device tensor {src ptr, dst ptr, cy, taps, cx} of bf16 tensors."""
    lib = _lib.require_device()
    check(lib.mpgan_weight_transpose_batch(ptr(table), n, max_elems, _stream()), "weight_transpose_batch")


def permute_flatten(src, dst, rows, c, spatial, to_cl, accumulate=False):
    lib = _lib.require_device()
    check(lib.mpgan_permute_flatten(dt(src), ptr(src), dt(dst), ptr(dst), rows, c, spatial, 1 if to_cl else 0,
                                    1 if accumulate else 0, _stream()), "permute_flatten")
    return dst


# ---------------------------------------------------------------------------------------------------------
# linear, losses, optimiser, patches
# ---------------------------------------------------------------------------------------------------------
def linear_fwd(x, w, bias, y):
    """x (B,K) and w (J,K) share dtype and flatten order; y (B,J) fp32 must be zeroed by the caller."""
    lib = _lib.require_device()
    b, k = x.shape
    check(lib.mpgan_linear_fwd(dt(x), ptr(x), ptr(w), ptr(bias), ptr(y), b, k, w.shape[0], _stream()), "linear_fwd")
    return y


def linear_bwd(x, w, dy, dx, dw, db):
    lib = _lib.require_device()
    b, k = x.shape
    check(lib.mpgan_linear_bwd(dt(x), ptr(x), ptr(w), ptr(dy), ptr(dx), ptr(dw), ptr(db), b, k, w.shape[0],
                               _stream()), "linear_bwd")


_LINEAR_TC = os.environ.get("MPGAN_NO_LINEAR_TC", "0") != "1"


def linear_tc_ok(x, j, k):
    """A Linear layer that is a real GEMM (the patch discriminator's Linear(512 * 8^d, 64) over 4 096 patches,
    test_runs/GAN.py:176-181) runs on the tcgen05 kernels as a 1x1 convolution over a (1, B / 16, 16, K) "image"."""
    b = x.shape[0]
    return (_LINEAR_TC and x.dtype == torch.bfloat16 and x.is_contiguous() and b % 16 == 0 and b >= 256 and j % 16 == 0
            and 16 <= j <= 512 and k % 256 == 0)


def _gemm_geom(cin, cout, b):
    return ConvSpec(2, cin, cout, 1, 1, 0).geom(1, (b // 16, 16), (b // 16, 16))


def linear_tc_fwd(x, w, bias):
    """z (B, J) fp32 = x (B, K) bf16 . w (J, K)^T bf16 + bias, fp32 accumulation in TMEM."""
    lib = _lib.require_device()
    b, k = x.shape
    j = w.shape[0]
    z16 = torch.empty((b, j), dtype=torch.bfloat16, device=x.device)
    g = _gemm_geom(k, j, b)
    check(lib.mpgan_tc_conv_fprop(ctypes.byref(g), ptr(x), k, ptr(w), ptr(bias), ptr(z16), j, None, _stream()), "linear_tc_fwd")
    return cast(z16, torch.empty((b, j), dtype=torch.float32, device=x.device))


def linear_tc_bwd(x, w, dz, dx, dw, db):
    """dx (B, K) bf16 = dz . w;  dw (J, K) fp32 += dz^T . x;  db (J) += column sums of dz.  dz (B, J) fp32."""
    lib = _lib.require_device()
    b, k = x.shape
    j = w.shape[0]
    dz16 = cast(dz.contiguous(), torch.empty((b, j), dtype=torch.bfloat16, device=x.device))
    wt = weight_transpose(w, torch.empty(j * k, dtype=torch.bfloat16, device=x.device), j, 1, k)      # [K][J]
    g = _gemm_geom(j, k, b)
    check(lib.mpgan_tc_conv_fprop(ctypes.byref(g), ptr(dz16), j, ptr(wt), None, ptr(dx), k, None, _stream()), "linear_tc_dx")
    if dw is not None:
        g2 = _gemm_geom(k, j, b)
        check(lib.mpgan_tc_conv_wgrad(ctypes.byref(g2), ptr(x), k, ptr(dz16), j, ptr(dw), None, 0, _stream()), "linear_tc_dw")
    if db is not None:
        colsum(dz16, db)


def sigmoid_fwd(z, p):
    lib = _lib.require_device()
    check(lib.mpgan_sigmoid_fwd(ptr(z), ptr(p), z.numel(), _stream()), "sigmoid_fwd")
    return p


def sigmoid_bwd(dp, p, dz):
    lib = _lib.require_device()
    check(lib.mpgan_sigmoid_bwd(ptr(dp), ptr(p), ptr(dz), p.numel(), _stream()), "sigmoid_bwd")
    return dz


def bce_fwd(prob, target, weight, loss):
    lib = _lib.require_device()
    check(lib.mpgan_bce_fwd(ptr(prob), ptr(target), weight, ptr(loss), prob.numel(), _stream()), "bce_fwd")


def bce_bwd(prob, target, weight, gscale, dprob):
    lib = _lib.require_device()
    check(lib.mpgan_bce_bwd(ptr(prob), ptr(target), weight, ptr(gscale), ptr(dprob), prob.numel(), _stream()),
          "bce_bwd")
    return dprob


def l1_fwd(a, b, weight, loss):
    lib = _lib.require_device()
    assert a.is_contiguous() and b.is_contiguous() and a.dtype == b.dtype
    check(lib.mpgan_l1_fwd(dt(a), ptr(a), ptr(b), a.numel(), weight, ptr(loss), _stream()), "l1_fwd")


def l1_bwd(a, b, weight, gscale, da, accumulate):
    lib = _lib.require_device()
    assert a.is_contiguous() and b.is_contiguous() and da.is_contiguous() and a.dtype == b.dtype == da.dtype
    check(lib.mpgan_l1_bwd(dt(a), ptr(a), ptr(b), a.numel(), weight, ptr(gscale), ptr(da), 1 if accumulate else 0,
                           _stream()), "l1_bwd")
    return da


def l1_fwd_bwd(a, b, weight, loss, da, accumulate, gscale=None):
    """One pass over (a, b): loss += weight * mean|a - b| (loss: fp32 or fp64 one-element device tensor, or None) and
    da (+)= weight / n * sign(a - b)."""
    lib = _lib.require_device()
    assert a.is_contiguous() and b.is_contiguous() and a.dtype == b.dtype and a.numel() == b.numel()
    assert da is None or (da.is_contiguous() and da.dtype == a.dtype and da.numel() == a.numel())
    l32 = loss if (loss is not None and loss.dtype == torch.float32) else None
    l64 = loss if (loss is not None and loss.dtype == torch.float64) else None
    assert loss is None or l32 is not None or l64 is not None
    check(lib.mpgan_l1_fwd_bwd(dt(a), ptr(a), ptr(b), a.numel(), weight, ptr(gscale), ptr(l32), ptr(l64), ptr(da),
                               1 if accumulate else 0, _stream()), "l1_fwd_bwd")
    return da


class LazyL1:
    """Gradient of ``weight * l1_loss(mine, other)`` w.r.t. ``mine`` that has not been materialised: the consumer
    accumulates it into its own gradient tensor (and the loss into ``loss``) with ONE pass over the pair."""

    def __init__(self, mine, other, weight, loss):
        self.mine, self.other, self.weight, self.loss = mine, other, weight, loss

    def add_to(self, target):
        """target += d loss / d mine; the loss term is accumulated by the same kernel."""
        return l1_fwd_bwd(self.mine, self.other, self.weight, self.loss, target, True)

    def materialize(self):
        return l1_fwd_bwd(self.mine, self.other, self.weight, self.loss, torch.empty_like(self.mine), False)


def adam_step(param, grad, m, v, lr, b1, b2, eps, state, shadow=None):
    lib = _lib.require_device()
    check(lib.mpgan_adam_step(ptr(param), ptr(grad), ptr(m), ptr(v), param.numel(), lr, b1, b2, eps, ptr(state),
                              ptr(shadow), _stream()), "adam_step")


def patch_gather(vol, origins, num_samples, roi, out=None):
    """vol (B,*S,C) channels-last contiguous; origins int32 device (B*num_samples, rank)."""
    lib = _lib.require_device()
    assert vol.is_contiguous() and origins.dtype == torch.int32 and origins.is_contiguous()
    b, sp, c = vol.shape[0], tuple(vol.shape[1:-1]), vol.shape[-1]
    rank = len(sp)
    if out is None:
        out = torch.empty((b * num_samples,) + (roi,) * rank + (c,), dtype=vol.dtype, device=vol.device)
    spatial = (ctypes.c_int32 * rank)(*sp)
    check(lib.mpgan_patch_gather(dt(vol), ptr(vol), b, rank, spatial, c, ptr(origins), num_samples, roi, ptr(out),
                                 _stream()), "patch_gather")
    return out


def patch_scatter_add(dpatch, origins, num_samples, roi, dvol):
    lib = _lib.require_device()
    assert dvol.is_contiguous() and dpatch.is_contiguous() and origins.dtype == torch.int32
    b, sp, c = dvol.shape[0], tuple(dvol.shape[1:-1]), dvol.shape[-1]
    rank = len(sp)
    spatial = (ctypes.c_int32 * rank)(*sp)
    check(lib.mpgan_patch_scatter_add(dt(dvol), ptr(dpatch), b, rank, spatial, c, ptr(origins), num_samples, roi,
                                      ptr(dvol), _stream()), "patch_scatter_add")
    return dvol


class WindowTable:
    """Geometry table of ``window_gather`` / ``window_blend`` (layout: include/mpgan.h), as a host tensor and its device
    copy.  ``size``, ``roi``: per spatial dim (2 or 3 of them); ``starts``: per dim, increasing window starts in padded
    coordinates; ``taps``: per dim, ``roi[d]`` importance taps in (0, 1]."""

    def __init__(self, size, roi, starts, taps, device):
        lead = 3 - len(size)        # rank 2: a trivial leading dim
        size3, roi3 = (1,) * lead + tuple(size), (1,) * lead + tuple(roi)
        starts3, taps3 = [[0]] * lead + [list(s) for s in starts], [[1.0]] * lead + [list(t) for t in taps]
        lo3 = [max(r - s, 0) // 2 for s, r in zip(size3, roi3)]
        self.nwin = 1
        for s in starts3:
            self.nwin *= len(s)
        words = [len(size), *size3, *roi3, *lo3, *(len(s) for s in starts3), 0, 0, 0]
        for s in starts3:
            words += s
        for s, r, st in zip(size3, roi3, starts3):
            for p in range(max(s, r)):                 # windows j_first .. j_last cover p: p - roi < s_j <= p
                words += [bisect.bisect_right(st, p - r), bisect.bisect_right(st, p) - 1]
        words += [0] * (len(words) & 1)
        host = torch.tensor(words, dtype=torch.int32)
        tap = torch.tensor([t for ts in taps3 for t in ts], dtype=torch.float64)
        self.host = torch.cat([host, tap.view(torch.int32)])
        self.dev = self.host.to(device)


def window_gather(x, table, first, count, cval, out):
    """out (count, C, *roi) = windows [first, first + count) of x (B, C, *S) with ``cval`` outside S."""
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous() and x.dtype == out.dtype == torch.float32
    check(lib.mpgan_window_gather(ptr(x), x.shape[0], x.shape[1], ptr(table.host), ptr(table.dev), table.host.numel(),
                                  first, count, cval, ptr(out), _stream()), "window_gather")
    return out


def window_blend(pred, batch, table, out):
    """pred (batch * nwin, C, *roi) -> out (batch, C, *S), the importance-weighted mean of the covering windows."""
    lib = _lib.require_device()
    assert pred.is_contiguous() and out.is_contiguous() and pred.dtype == out.dtype == torch.float32
    check(lib.mpgan_window_blend(ptr(pred), batch, pred.shape[1], ptr(table.host), ptr(table.dev), table.host.numel(),
                                 ptr(out), _stream()), "window_blend")
    return out


def resample_linear(x, items, rank, in_size, out_size, geom_map, default_value, out):
    """out (items, *out grid) = ITK-linear resampling of x (items, *in grid); sizes in ITK order (x, y, z), ``geom_map``
    the 24 fp64 words of include/mpgan.h."""
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous() and x.dtype == out.dtype == torch.float32
    check(lib.mpgan_resample_linear(ptr(x), items, rank, _i3(in_size), _i3(out_size), (ctypes.c_double * 24)(*geom_map),
                                    default_value, ptr(out), _stream()), "resample_linear")
    return out


def resample_nearest(x, items, rank, in_size, out_size, geom_map, default_bits, out):
    """out (items, *out grid) = nearest-neighbour resampling of x (items, *in grid), a bit copy of 1- or 4-byte
    elements; outside voxels get the low bytes of ``default_bits``."""
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous() and x.dtype == out.dtype and x.element_size() in (1, 4)
    check(lib.mpgan_resample_nearest(ptr(x), x.element_size(), items, rank, _i3(in_size), _i3(out_size),
                                     (ctypes.c_double * 24)(*geom_map), default_bits, ptr(out), _stream()),
          "resample_nearest")
    return out


def bspline_coefficients(x, items, rank, size, coef):
    """coef (items, *grid) fp64 = cubic B-spline coefficients of x (items, *grid) fp32, mirror boundaries."""
    lib = _lib.require_device()
    assert x.is_contiguous() and coef.is_contiguous() and x.dtype == torch.float32 and coef.dtype == torch.float64
    assert coef.numel() == x.numel()
    check(lib.mpgan_bspline_coefficients(ptr(x), items, rank, _i3(size), ptr(coef), _stream()), "bspline_coefficients")
    return coef


def resample_bspline(coef, items, rank, in_size, out_size, geom_map, default_value, out):
    """out (items, *out grid) fp32 = cubic B-spline interpolation of the coefficients coef (items, *in grid) fp64."""
    lib = _lib.require_device()
    assert coef.is_contiguous() and out.is_contiguous() and coef.dtype == torch.float64 and out.dtype == torch.float32
    check(lib.mpgan_resample_bspline(ptr(coef), items, rank, _i3(in_size), _i3(out_size),
                                     (ctypes.c_double * 24)(*geom_map), default_value, ptr(out), _stream()),
          "resample_bspline")
    return out


def mutual_info(a, b, items, n, bins, counts, edges, out5, mask=None):
    """Joint histogram and entropies of ``items`` image pairs of ``n`` voxels: counts (items, bins, bins) int64, edges
    (items, 2, bins + 1) fp32 or None, out5 (items, 5) fp64 = H1, H2, H12, MI, NMI (include/mpgan.h).  ``mask``: None,
    or a contiguous uint8 tensor laid out like the images; then only the voxels where it is non-zero count."""
    lib = _lib.require_device()
    assert a.is_contiguous() and b.is_contiguous() and a.dtype == b.dtype == torch.float32
    assert counts.dtype == torch.int64 and out5.dtype == torch.float64
    nbytes = int(lib.mpgan_mutual_info_workspace(items))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=a.device)
    if mask is None:
        check(lib.mpgan_mutual_info(ptr(a), ptr(b), items, n, bins, ptr(counts), ptr(edges), ptr(out5), ptr(ws), nbytes,
                                    _stream()), "mutual_info")
    else:
        assert mask.is_contiguous() and mask.dtype == torch.uint8 and mask.numel() == a.numel()
        check(lib.mpgan_mutual_info_masked(ptr(a), ptr(b), ptr(mask), items, n, bins, ptr(counts), ptr(edges),
                                           ptr(out5), ptr(ws), nbytes, _stream()), "mutual_info_masked")
    return counts, edges, out5


def otsu_threshold(x, items, n, bins, thr):
    """thr (items,) fp32 = Otsu's threshold of each of the ``items`` images of ``n`` voxels in x (include/mpgan.h)."""
    lib = _lib.require_device()
    assert x.is_contiguous() and x.dtype == thr.dtype == torch.float32 and thr.numel() == items
    nbytes = int(lib.mpgan_otsu_threshold_workspace(items, bins))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    check(lib.mpgan_otsu_threshold(ptr(x), items, n, bins, ptr(thr), ptr(ws), nbytes, _stream()), "otsu_threshold")
    return thr


def threshold_mask(x, thr, items, n, mask):
    """mask (uint8, laid out like x) = x > thr[item], for ``items`` images of ``n`` voxels."""
    lib = _lib.require_device()
    assert x.is_contiguous() and mask.is_contiguous() and x.dtype == thr.dtype == torch.float32
    assert mask.dtype == torch.uint8 and mask.numel() == x.numel() and thr.numel() == items
    check(lib.mpgan_threshold_mask(ptr(x), ptr(thr), items, n, ptr(mask), _stream()), "threshold_mask")
    return mask


def _morph_workspace(lib, items, dhw, device):
    nbytes = int(lib.mpgan_morphology_workspace(items, *dhw))
    return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes


def label(mask, rank, items, dhw, connectivity, labels, count):
    """labels (int32, laid out like mask) and count (int32 [items]) of ``items`` uint8 masks of extent ``dhw`` = (d, h,
    w) (include/mpgan.h)."""
    lib = _lib.require_device()
    assert mask.is_contiguous() and mask.dtype == torch.uint8 and labels.dtype == count.dtype == torch.int32
    assert labels.is_contiguous() and labels.numel() == mask.numel() and count.numel() == items
    ws, nbytes = _morph_workspace(lib, items, dhw, mask.device)
    check(lib.mpgan_label(ptr(mask), rank, items, *dhw, connectivity, ptr(labels), ptr(count), ptr(ws), nbytes, _stream()),
          "label")
    return labels, count


def mask_op(name, mask, rank, items, dhw, connectivity, out, *extra):
    """out (uint8, laid out like mask) = ``name`` ("largest_component", "fill_holes" or "binary_morphology" with extra
    = (op, iterations)) of ``items`` uint8 masks of extent ``dhw`` (include/mpgan.h)."""
    lib = _lib.require_device()
    assert mask.is_contiguous() and out.is_contiguous() and mask.dtype == out.dtype == torch.uint8
    assert out.numel() == mask.numel()
    ws, nbytes = _morph_workspace(lib, items, dhw, mask.device)
    check(getattr(lib, "mpgan_" + name)(ptr(mask), rank, items, *dhw, connectivity, *extra, ptr(out), ptr(ws), nbytes,
                                        _stream()), name)
    return out


def distance_transform(mask, rank, items, dhw, sampling, out):
    """out (fp64, laid out like mask) = the Euclidean distance transform of ``items`` uint8 masks of extent ``dhw`` =
    (d, h, w) with voxel spacing ``sampling`` = (sd, sh, sw) (include/mpgan.h)."""
    lib = _lib.require_device()
    assert mask.is_contiguous() and out.is_contiguous() and mask.dtype == torch.uint8 and out.dtype == torch.float64
    assert out.numel() == mask.numel()
    nbytes = int(lib.mpgan_distance_transform_workspace(items, *dhw))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=mask.device)
    check(lib.mpgan_distance_transform(ptr(mask), rank, items, *dhw, *sampling, ptr(out), ptr(ws), nbytes, _stream()),
          "distance_transform")
    return out


def mask_agreement(pred, truth, rank, items, dhw, sampling, connectivity, percentile, out6):
    """out6 (items, 6) fp64 = dice, jaccard, hausdorff, hausdorff_percentile, average_surface_distance,
    symmetric_surface_distance of ``items`` pairs of uint8 masks (include/mpgan.h)."""
    lib = _lib.require_device()
    assert pred.is_contiguous() and truth.is_contiguous() and pred.dtype == truth.dtype == torch.uint8
    assert pred.numel() == truth.numel() and out6.is_contiguous() and out6.dtype == torch.float64
    assert out6.numel() == 6 * items
    nbytes = int(lib.mpgan_mask_agreement_workspace(items, *dhw))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=pred.device)
    check(lib.mpgan_mask_agreement(ptr(pred), ptr(truth), rank, items, *dhw, *sampling, connectivity, percentile,
                                   ptr(out6), ptr(ws), nbytes, _stream()), "mask_agreement")
    return out6


def _dv(v):
    return (ctypes.c_double * len(v))(*[float(a) for a in v])


_MAPS_ENTRIES = {"linear": "mpgan_resample_linear_maps", "nearest": "mpgan_resample_nearest_maps",
                 "bspline": "mpgan_resample_bspline_maps"}


def resample_maps(mode, x, items, rank, in_size, out_size, maps, default, out):
    """out (items, *out grid) = resampling of x (items, *in grid; fp64 coefficients for "bspline") with item i read
    through maps[i] (device fp64 (items, 24)); ``default`` is the fp32 default value, or the bits for "nearest"."""
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous() and maps.is_contiguous() and maps.dtype == torch.float64
    assert maps.numel() == 24 * items
    fn = getattr(lib, _MAPS_ENTRIES[mode])
    if mode == "nearest":
        rc = fn(ptr(x), x.element_size(), items, rank, _i3(in_size), _i3(out_size), ptr(maps), default, ptr(out),
                _stream())
    else:
        rc = fn(ptr(x), items, rank, _i3(in_size), _i3(out_size), ptr(maps), default, ptr(out), _stream())
    check(rc, _MAPS_ENTRIES[mode])
    return out


def gaussian_filter(x, items, rank, size, taps_xyz, out):
    """out = the separable fp64 Gaussian of ``items`` fp32 images of ITK size ``size`` with taps per axis (x, y, z)."""
    lib = _lib.require_device()
    assert x.is_contiguous() and out.is_contiguous() and x.dtype == out.dtype == torch.float32
    radius = [len(t) // 2 for t in taps_xyz]
    nbytes = int(lib.mpgan_gaussian_filter_workspace(items, _i3(size)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    check(lib.mpgan_gaussian_filter(ptr(x), items, rank, _i3(size), _i3(radius), _dv([w for t in taps_xyz for w in t]),
                                    ptr(out), ptr(ws), nbytes, _stream()), "gaussian_filter")
    return out


def rigid_maps(params, items, rank, base, center, maps):
    """maps (items, 24) fp64 = the rigid transforms ``params`` (items, P) composed with the 24-word ``base``."""
    lib = _lib.require_device()
    assert params.is_contiguous() and maps.is_contiguous() and params.dtype == maps.dtype == torch.float64
    check(lib.mpgan_rigid_maps(ptr(params), items, rank, _dv(base), _dv(center), ptr(maps), _stream()), "rigid_maps")
    return maps


def rigid_level(state, status, items, rank, base, center, initial, t0, first, step):
    lib = _lib.require_device()
    check(lib.mpgan_rigid_level(ptr(state), ptr(status), items, rank, _dv(base), _dv(center), ptr(initial), _dv(t0),
                                int(first), float(step), _stream()), "rigid_level")


def rigid_step(state, status, items, rank, base, center, min_step, last):
    lib = _lib.require_device()
    check(lib.mpgan_rigid_step(ptr(state), ptr(status), items, rank, _dv(base), _dv(center), float(min_step), int(last),
                               _stream()), "rigid_step")


def mattes_workspace(items, fixed_size, moving_size, bins, device):
    lib = _lib.require_device()
    nbytes = int(lib.mpgan_mattes_workspace(items, _i3(fixed_size), _i3(moving_size), bins))
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def mattes_prepare(fixed, moving, mask, items, rank, fixed_size, moving_size, shrink, bins, fixed_matrix, min_scale,
                   state, status, ws):
    lib = _lib.require_device()
    check(lib.mpgan_mattes_prepare(ptr(fixed), ptr(moving), ptr(mask), items, rank, _i3(fixed_size), _i3(moving_size),
                                   shrink, bins, _dv(fixed_matrix), float(min_scale), ptr(state), ptr(status), ptr(ws),
                                   ws.numel(), _stream()), "mattes_prepare")


def mattes_evaluate(fixed, moving, mask, items, rank, fixed_size, moving_size, shrink, bins, gradient, only_running,
                    state, status, hist, metric, ws):
    lib = _lib.require_device()
    check(lib.mpgan_mattes_evaluate(ptr(fixed), ptr(moving), ptr(mask), items, rank, _i3(fixed_size),
                                    _i3(moving_size), shrink, bins, int(gradient), int(only_running), ptr(state),
                                    ptr(status), ptr(hist), ptr(metric), ptr(ws), ws.numel(), _stream()),
          "mattes_evaluate")
