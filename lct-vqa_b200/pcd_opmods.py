"""The candidate operations of operations.py as stand-alone native ops (what `OPS[name](C, stride, affine)` modules run when
they are called on their own, and what a network derived from a genotype is built from — SURVEY.md §8f-4).

    unit_apply      ReLU -> depthwise KxK -> 1x1 -> BatchNorm    one autograd Function over pcd_dwconv_* / pcd_pwconv_* /
                                                                  pcd_bn_apply / pcd_bn_backward_stats
                    DilConv (operations.py:35-47) is one unit, SepConv (operations.py:50-66) two
    pool_apply      AvgPool2d(3, s, 1, count_include_pad=False) / MaxPool2d(3, s, 1)        (operations.py:6-7)
    affine_apply    gamma * yhat + beta behind the preprocess kernels' normalised output (ReLUConvBN / FactorizedReduce with
                    affine=True, operations.py:22-33,90-104)

BatchNorm in training mode (batch statistics; running statistics updated like nn.BatchNorm2d) or, in eval mode under
torch.no_grad(), from the running statistics (forward only, nothing written).
"""
import ctypes as C

import torch

import pcd_native as N
from pcd_ops import BN_EPS, BN_MOMENTUM, _empty, _empty_like, _f32c, autograd_records


def _bn_running(bn):
    """(running_mean | running_var) as ONE 2C buffer, which is what the kernels update; nn.BatchNorm2d keeps two tensors, so
    they are re-bound once to two halves of one allocation (a parent arena may already have done that)."""
    rm, rv = bn.running_mean, bn.running_var
    c = rm.numel()
    if rv.data_ptr() != rm.data_ptr() + 4 * c:
        both = torch.cat([rm.detach().reshape(-1), rv.detach().reshape(-1)])
        rm.data, rv.data = both[:c], both[c:]
    return rm.data_ptr(), bn.num_batches_tracked.data_ptr()


class UnitFunction(torch.autograd.Function):
    """y = BN(pw(dw(relu(x)))), BatchNorm in training mode, gamma / beta optional."""

    @staticmethod
    def forward(ctx, x, w_dw, w_pw, gamma, beta, meta):
        ks, stride, pad, dil, run_ptr, nbt_ptr = meta
        lib = N.lib_for(x)
        xc, wd, wp = _f32c(x), _f32c(w_dw), _f32c(w_pw)
        B, cin, H, W = xc.shape
        cout = wp.shape[0]
        ho = (H + 2 * pad - dil * (ks - 1) - 1) // stride + 1
        wo = (W + 2 * pad - dil * (ks - 1) - 1) // stride + 1
        dev, st = xc.device, N.stream_for(xc)
        t = _empty((B, cin, ho, wo), torch.float32, dev)
        a = N.DwConvArgs(B, cin, H, W, ks, stride, pad, dil, 1, N.ptr(xc), N.ptr(wd), N.ptr(t), None, None, None)
        N.check(lib, lib.pcd_dwconv_forward(C.byref(a), st), "pcd_dwconv_forward")
        z = _empty((B, cout, ho, wo), torch.float32, dev)
        stats = _empty(2 * cout, torch.float64, dev)
        p = N.PwConvArgs(B, cin, cout, ho * wo, BN_EPS, N.ptr(t), N.ptr(wp), N.ptr(z), N.ptr(stats), None, None, None, None, None)
        N.check(lib, lib.pcd_pwconv_forward(C.byref(p), st), "pcd_pwconv_forward")
        y = _empty_like(z)
        g = _f32c(gamma) if gamma is not None else None
        b = _f32c(beta) if beta is not None else None
        n = N.BnArgs(B, cout, ho * wo, BN_EPS, BN_MOMENTUM, N.ptr(z), N.ptr(stats), N.ptr(g), N.ptr(b), run_ptr, nbt_ptr, N.ptr(y),
                     None, None)
        N.check(lib, lib.pcd_bn_apply(C.byref(n), st), "pcd_bn_apply")
        ctx.meta = (ks, stride, pad, dil, B, cin, cout, H, W, ho, wo)
        ctx.shapes = (w_dw.shape, w_pw.shape)
        ctx.save_for_backward(xc, wd, wp, g, t, z, stats)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, wd, wp, g, t, z, stats = ctx.saved_tensors
        ks, stride, pad, dil, B, cin, cout, H, W, ho, wo = ctx.meta
        lib = N.lib_for(x)
        dev, st = x.device, N.stream_for(x)
        gy = _f32c(gy)
        bstats = _empty(2 * cout, torch.float64, dev)
        n = N.BnArgs(B, cout, ho * wo, BN_EPS, BN_MOMENTUM, N.ptr(z), N.ptr(stats), None, None, None, None, None, N.ptr(gy), N.ptr(bstats))
        N.check(lib, lib.pcd_bn_backward_stats(C.byref(n), st), "pcd_bn_backward_stats")
        need_x, need_wd, need_wp = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        gx = gwd = gwp = None
        if need_x or need_wd or need_wp:
            dt = _empty_like(t) if (need_x or need_wd) else None
            gwp = _empty(wp.numel(), torch.float32, dev) if need_wp else None
            p = N.PwConvArgs(B, cin, cout, ho * wo, BN_EPS, N.ptr(t), N.ptr(wp), N.ptr(z), N.ptr(stats), N.ptr(gy), N.ptr(g),
                             N.ptr(bstats), N.ptr(dt), N.ptr(gwp))
            N.check(lib, lib.pcd_pwconv_backward(C.byref(p), st), "pcd_pwconv_backward")
            if need_x or need_wd:
                gx = _empty_like(x) if need_x else None
                gwd = _empty(wd.numel(), torch.float32, dev) if need_wd else None
                a = N.DwConvArgs(B, cin, H, W, ks, stride, pad, dil, 1, N.ptr(x), N.ptr(wd), None, N.ptr(dt), N.ptr(gx), N.ptr(gwd))
                N.check(lib, lib.pcd_dwconv_backward(C.byref(a), st), "pcd_dwconv_backward")
        # d beta = sum dy, d gamma = sum dy * yhat: the two sums BatchNorm's backward needs anyway
        ggamma = bstats[cout:].to(torch.float32) if ctx.needs_input_grad[3] else None
        gbeta = bstats[:cout].to(torch.float32) if ctx.needs_input_grad[4] else None
        return (gx, gwd.view(ctx.shapes[0]) if gwd is not None else None, gwp.view(ctx.shapes[1]) if gwp is not None else None,
                ggamma, gbeta, None)


def _check(x, bn, what):
    if not bn.track_running_stats or bn.momentum is None or abs(bn.momentum - BN_MOMENTUM) > 1e-12 or abs(bn.eps - BN_EPS) > 1e-12:
        raise NotImplementedError(f"{what}: BatchNorm2d(eps={BN_EPS}, momentum={BN_MOMENTUM}, track_running_stats=True) expected")
    if x.dim() != 4 or x.dtype != torch.float32:
        raise NotImplementedError(f"{what}: float32 NCHW input expected")


def _eval_guard(tensors, bn, what):
    """True in eval mode (BatchNorm from running statistics: forward only); raises if autograd would record that forward."""
    if bn.training:
        return False
    if autograd_records(tensors):
        raise NotImplementedError(f"{what} in eval mode (BatchNorm from running statistics) is forward-only: wrap the call in "
                                  "torch.no_grad() or torch.inference_mode(), or call .train() to differentiate")
    return True


def _unit_eval(x, dw, pw, bn):
    """Eval-mode unit: dwconv -> pwconv (its batch sums go to a scratch buffer, unused) -> per-channel running-stat affine."""
    lib = N.lib_for(x)
    xc = _f32c(x)
    ks, stride, pad, dil = dw.kernel_size[0], dw.stride[0], dw.padding[0], dw.dilation[0]
    B, cin, H, W = xc.shape
    cout = pw.out_channels
    ho = (H + 2 * pad - dil * (ks - 1) - 1) // stride + 1
    wo = (W + 2 * pad - dil * (ks - 1) - 1) // stride + 1
    dev, st = xc.device, N.stream_for(xc)
    t = _empty((B, cin, ho, wo), torch.float32, dev)
    a = N.DwConvArgs(B, cin, H, W, ks, stride, pad, dil, 1, N.ptr(xc), N.ptr(_f32c(dw.weight)), N.ptr(t), None, None, None)
    N.check(lib, lib.pcd_dwconv_forward(C.byref(a), st), "pcd_dwconv_forward")
    z = _empty((B, cout, ho, wo), torch.float32, dev)
    scratch = _empty(2 * cout, torch.float64, dev)
    p = N.PwConvArgs(B, cin, cout, ho * wo, BN_EPS, N.ptr(t), N.ptr(_f32c(pw.weight)), N.ptr(z), N.ptr(scratch), None, None, None,
                     None, None)
    N.check(lib, lib.pcd_pwconv_forward(C.byref(p), st), "pcd_pwconv_forward")
    # ATen's inference BatchNorm: scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale
    scale = 1.0 / torch.sqrt(bn.running_var + bn.eps)
    if bn.affine:
        scale = scale * bn.weight
    shift = -bn.running_mean * scale
    if bn.affine:
        shift = shift + bn.bias
    y = _empty_like(z)
    N.check(lib, lib.pcd_channel_affine(N.ptr(z), N.ptr(_f32c(scale)), N.ptr(_f32c(shift)), N.ptr(y), B, cout, ho * wo, st),
            "pcd_channel_affine")
    return y


def unit_apply(x, dw, pw, bn, what="unit"):
    """ReLU -> `dw` (depthwise nn.Conv2d) -> `pw` (1x1 nn.Conv2d) -> `bn` on the native kernels."""
    is_eval = _eval_guard([x, dw.weight, pw.weight, bn.weight, bn.bias], bn, what)
    _check(x, bn, what)
    ks, stride, pad, dil = dw.kernel_size[0], dw.stride[0], dw.padding[0], dw.dilation[0]
    if dw.groups != dw.in_channels or dw.kernel_size[0] != dw.kernel_size[1] or ks not in (3, 5, 7) or stride not in (1, 2) or \
            dw.bias is not None or pw.bias is not None or pw.kernel_size != (1, 1) or pw.in_channels % 4 or pw.out_channels % 4 or \
            max(pw.in_channels, pw.out_channels) > 128 or max(x.shape[2], x.shape[3]) > 64:
        raise RuntimeError(f"{what}: shape not supported by the compiled kernels (PCD_ERR_UNSUPPORTED)")
    if is_eval:
        return _unit_eval(x, dw, pw, bn)
    run_ptr, nbt_ptr = _bn_running(bn)
    return UnitFunction.apply(x, dw.weight, pw.weight, bn.weight if bn.affine else None, bn.bias if bn.affine else None,
                              (ks, stride, pad, dil, run_ptr, nbt_ptr))


class PoolFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, is_max, stride):
        lib = N.lib_for(x)
        xc = _f32c(x)
        B, c, H, W = xc.shape
        y = _empty((B, c, (H - 1) // stride + 1, (W - 1) // stride + 1), torch.float32, xc.device)
        a = N.PoolArgs(B, c, H, W, stride, int(is_max), N.ptr(xc), N.ptr(y), None, None)
        N.check(lib, lib.pcd_pool3x3_forward(C.byref(a), N.stream_for(xc)), "pcd_pool3x3_forward")
        ctx.meta = (is_max, stride)
        ctx.save_for_backward(xc)
        return y

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        is_max, stride = ctx.meta
        lib = N.lib_for(x)
        B, c, H, W = x.shape
        gy = _f32c(gy)
        gx = _empty_like(x)
        a = N.PoolArgs(B, c, H, W, stride, int(is_max), N.ptr(x), None, N.ptr(gy), N.ptr(gx))
        N.check(lib, lib.pcd_pool3x3_backward(C.byref(a), N.stream_for(x)), "pcd_pool3x3_backward")
        return gx, None, None


def pool_apply(x, kind, stride):
    if x.dim() != 4 or x.dtype != torch.float32 or stride not in (1, 2) or max(x.shape[2], x.shape[3]) > 64:
        raise RuntimeError("3x3 pool: shape not supported by the compiled kernels (PCD_ERR_UNSUPPORTED)")
    return PoolFunction.apply(x, kind == "max", stride)


class ChannelAffineFunction(torch.autograd.Function):
    """y = gamma[c] * yhat + beta[c]."""

    @staticmethod
    def forward(ctx, yhat, gamma, beta):
        lib = N.lib_for(yhat)
        yh, g, b = _f32c(yhat), _f32c(gamma), _f32c(beta)
        B, c, H, W = yh.shape
        y = _empty_like(yh)
        N.check(lib, lib.pcd_channel_affine(N.ptr(yh), N.ptr(g), N.ptr(b), N.ptr(y), B, c, H * W, N.stream_for(yh)), "pcd_channel_affine")
        ctx.save_for_backward(yh, g)
        return y

    @staticmethod
    def backward(ctx, gy):
        yh, g = ctx.saved_tensors
        lib = N.lib_for(yh)
        B, c, H, W = yh.shape
        gy = _f32c(gy)
        st = N.stream_for(yh)
        gx = None
        if ctx.needs_input_grad[0]:
            gx = _empty_like(yh)
            N.check(lib, lib.pcd_channel_affine(N.ptr(gy), N.ptr(g), None, N.ptr(gx), B, c, H * W, st), "pcd_channel_affine")
        ggamma = gbeta = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            # sum dy and sum dy * yhat per channel: the BatchNorm-backward statistics kernel on an identity normalisation
            ident = torch.zeros(2 * c, dtype=torch.float64, device=yh.device)
            ident[c:] = float(B * H * W) * (1.0 - BN_EPS)        # mean 0, biased variance 1 - eps  =>  rstd = 1
            bstats = _empty(2 * c, torch.float64, yh.device)
            n = N.BnArgs(B, c, H * W, BN_EPS, BN_MOMENTUM, N.ptr(yh), N.ptr(ident), None, None, None, None, None, N.ptr(gy), N.ptr(bstats))
            N.check(lib, lib.pcd_bn_backward_stats(C.byref(n), st), "pcd_bn_backward_stats")
            ggamma, gbeta = bstats[c:].to(torch.float32), bstats[:c].to(torch.float32)
        return gx, ggamma, gbeta


def affine_apply(yhat, bn):
    return ChannelAffineFunction.apply(yhat, bn.weight, bn.bias)
