"""torch.autograd.Function wrappers over the C ABI, and the flat parameter arenas they rely on.

Boundary (SURVEY.md §8b): one Function per fused unit — stem, Cell (14 MixedOps + node sums +
preprocess), stand-alone MixedOp, adaptive pool.  All device memory (outputs, saved activations,
scratch) is allocated here with torch and handed to the library as raw pointers; the library
enqueues on torch's current stream.
"""
import ctypes as C
import math
import numbers

import torch

import pcd_native as N

import os

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
# debugging aid: PCD_DEBUG_POISON=1 fills every scratch / output buffer with NaN before the kernels run, so a
# read of memory the kernels never wrote cannot hide behind stale-but-plausible values
_POISON = os.environ.get("PCD_DEBUG_POISON", "0") == "1"


_DEBUG_KEEP = None      # set to a list to retain the buffers of every CellFunction.backward (debugging)


def _empty(shape, dtype, device):
    if _POISON and dtype in (torch.float32, torch.float64):
        return torch.full(shape if isinstance(shape, tuple) else (shape,), float("nan"), dtype=dtype, device=device)
    return torch.empty(shape, dtype=dtype, device=device)


def _empty_like(t):
    return _empty(tuple(t.shape), t.dtype, t.device)


# --------------------------------------------------------------------------------------------
# flat arenas: the kernels address a module's weights / BN buffers as ONE contiguous block in
# registration order; the nn.Parameter / buffer tensors stay ordinary leaves whose .data are views.
# --------------------------------------------------------------------------------------------
_LAYOUT_EPOCH = [0]


def bump_layout_epoch():
    """Called from Module._apply overrides: .to()/.cuda()/.float() replace storages (and buffer objects)."""
    _LAYOUT_EPOCH[0] += 1


def _is_run(tensors):
    """True when the tensors sit back to back in memory in the given order."""
    nxt = None
    for t in tensors:
        if not t.is_contiguous():
            return False
        p = t.data_ptr()
        if nxt is not None and p != nxt:
            return False
        nxt = p + t.numel() * t.element_size()
    return True


def _flatten_(tensors):
    """Rebind every tensor's .data to a view of one new flat tensor (values preserved)."""
    t0 = tensors[0]
    total = sum(t.numel() for t in tensors)
    flat = torch.empty(total, dtype=t0.dtype, device=t0.device)   # allocator blocks are >= 64-byte aligned
    off = 0
    with torch.no_grad():
        for t in tensors:
            n = t.numel()
            view = flat[off:off + n].view(t.shape)
            view.copy_(t.detach())
            t.data = view
            off += n
    return flat


class Arena:
    """Contiguity manager for a root module (Network, or a Cell / MixedOp used on its own)."""

    def __init__(self, module):
        self.module = module
        self.valid = False
        self.epoch = -1

    def _collect(self):
        m = self.module
        self.params = list(m.parameters())
        bufs = list(m.named_buffers())
        self.running = [b for k, b in bufs if not k.endswith("num_batches_tracked")]
        self.nbt = [b for k, b in bufs if k.endswith("num_batches_tracked")]

    def ensure(self):
        """Cheap when nothing moved: two pointer compares per group; full check after .to()/load."""
        if self.valid and self.epoch == _LAYOUT_EPOCH[0]:
            ok = True
            for group, first, last in self._ends:
                if group[0].data_ptr() != first or group[-1].data_ptr() != last:
                    ok = False
                    break
            if ok:
                return self
        self._collect()
        self._keep = []
        for group in (self.params, self.running, self.nbt):
            if group and (not _is_run(group) or group[0].data_ptr() % 16):
                self._keep.append(_flatten_(group))
        self._ends = [(g, g[0].data_ptr(), g[-1].data_ptr()) for g in (self.params, self.running, self.nbt) if g]
        self.param_ptr = self.params[0].data_ptr()
        self.running_ptr = self.running[0].data_ptr()
        self.nbt_ptr = self.nbt[0].data_ptr()
        self.param_floats = sum(p.numel() for p in self.params)
        self.valid = True
        self.epoch = _LAYOUT_EPOCH[0]
        return self

    def invalidate(self):
        self.valid = False

    def verify(self):
        """Every parameter / buffer still sits at its place in the arena (the kernels read them by raw pointer: a tensor
        re-bound by `p.data = ...`, load_state_dict(assign=True) or a parametrization would silently go stale).  ensure() only
        compares the ends of each group; this full check runs once per optimizer step (SearchStep / Architect)."""
        self.ensure()
        for group in (self.params, self.running, self.nbt):
            if group and not _is_run(group):
                self.valid = False
                raise RuntimeError("a parameter or buffer of the search network left its flat arena (re-bound .data?); "
                                   "call arena.invalidate() + forward, or do not re-bind storages")
        return self

    def flat(self, which):
        """One flat tensor aliasing a whole group ('params' | 'running' | 'nbt') of this arena."""
        group = getattr(self, which)
        t0 = group[0]
        n = sum(t.numel() for t in group)
        return torch.empty(0, dtype=t0.dtype, device=t0.device).set_(t0.untyped_storage(), t0.storage_offset(), (n,))


def _views(flat, params):
    """Split a flat grad arena into per-parameter views (a single C++ call)."""
    return torch._C._nn.unflatten_dense_tensors(flat, params)


# Activation-only backward (SURVEY.md §8b): the two finite-difference passes of the Hessian-vector
# product only need d loss / d alpha,beta (architect_vqa.py:110,115).  autograd's needs_input_grad cannot
# express that (it mirrors requires_grad, not the targets of autograd.grad), so the architect says so
# explicitly; the cell kernels then skip every weight-gradient phase and no per-parameter autograd edges
# are created.
_WEIGHT_GRADS = [True]


class weight_grads:
    def __init__(self, enabled):
        self.enabled = enabled

    def __enter__(self):
        self.prev = _WEIGHT_GRADS[0]
        _WEIGHT_GRADS[0] = self.enabled

    def __exit__(self, *exc):
        _WEIGHT_GRADS[0] = self.prev
        return False


def weight_grads_enabled():
    return _WEIGHT_GRADS[0]


def _param_grads(ctx, *idx):
    """Which PARAMETER gradients a dense Function's backward has to produce: needs_input_grad mirrors requires_grad, so inside
    `weight_grads(False)` (the architect's passes that only differentiate w.r.t. alpha / beta) every weight / bias product —
    two of the three GEMMs of a Linear, the LSTM's dW_ih / dW_hh — would be computed and thrown away."""
    on = _WEIGHT_GRADS[0]
    return tuple(bool(on and i is not None and ctx.needs_input_grad[i]) for i in idx)


# ---- weight-grad overlap (pcd_set_overlap): buffers of a Cell backward stay alive until the join ----------------
_OVERLAP = {"on": False, "keep": []}


def set_wgrad_overlap(on):
    """Run the cells' deferred weight-grad jobs on the library's low-priority stream, overlapping the rest of the backward
    pass.  They are joined at the start of the stem's backward (the last native op of every pass that computes weight
    grads) or by overlap_join().  Opt-in: used by SearchStep-driven runs."""
    lib = N.load_cuda()
    N.check(lib, lib.pcd_set_overlap(1 if on else 0), "pcd_set_overlap")
    _OVERLAP["on"] = bool(on)


def overlap_join(ref):
    """Make `ref`'s current stream wait for the outstanding weight-grad jobs; release their buffers."""
    if _OVERLAP["on"] or _OVERLAP["keep"]:
        lib = N.lib_for(ref)
        N.check(lib, lib.pcd_overlap_join(N.stream_for(ref)), "pcd_overlap_join")
        _OVERLAP["keep"].clear()


def _f32c(t):
    t = t.detach()
    if t.dtype != torch.float32:
        raise TypeError("pcdarts_sm100 kernels are fp32 only")
    return t if t.is_contiguous() else t.contiguous()


# --------------------------------------------------------------------------------------------
# Cell
# --------------------------------------------------------------------------------------------
class CellHandle:
    """Static description of one cell + where its arenas start (byte pointers)."""

    def __init__(self, c_prev_prev, c_prev, channels, reduction, reduction_prev):
        self.cfg = (c_prev_prev, c_prev, channels, int(bool(reduction)), int(bool(reduction_prev)))
        self._sizes = {}
        self.param_ptr = self.running_ptr = self.nbt_ptr = None

    def shape(self, batch, height, width):
        cpp, cp, ch, red, redp = self.cfg
        return N.CellShape(batch, cpp, cp, ch, height, width, red, redp, 4, BN_EPS, BN_MOMENTUM)

    def sizes(self, lib, batch, height, width):
        key = (batch, height, width)
        if key not in self._sizes:
            sz = N.CellSizes()
            sh = self.shape(batch, height, width)
            N.check(lib, lib.pcd_cell_sizes_of(C.byref(sh), C.byref(sz)), "pcd_cell_sizes_of")
            self._sizes[key] = sz
        return self._sizes[key]


class CellFunction(torch.autograd.Function):
    """Cell.forward (model_search.py:83-94) as one autograd node."""

    @staticmethod
    def forward(ctx, s0, s1, weights, weights2, handle, *params):
        lib = N.lib_for(s1)
        s0c, s1c, w, w2 = _f32c(s0), _f32c(s1), _f32c(weights), _f32c(weights2)
        B, _, H, W = s1c.shape
        sz = handle.sizes(lib, B, H, W)
        dev = s1c.device
        out = _empty((B, 4 * handle.cfg[2], sz.out_height, sz.out_width), torch.float32, dev)
        saved = _empty(sz.saved_floats, torch.float32, dev)
        stats = _empty(sz.stats_doubles, torch.float64, dev)
        # activation-only passes (no parameter takes part in autograd) never run the weight-grad jobs: skip what only they read
        skip_t = int(not any(ctx.needs_input_grad[5:]))
        a = N.CellFwdArgs(handle.shape(B, H, W), N.ptr(s0c), N.ptr(s1c), N.ptr(w), N.ptr(w2), handle.param_ptr,
                          handle.running_ptr, handle.nbt_ptr, N.ptr(out), N.ptr(saved), N.ptr(stats), skip_t)
        N.check(lib, lib.pcd_cell_forward(C.byref(a), N.stream_for(s1c)), "pcd_cell_forward")
        ctx.handle, ctx.params, ctx.geom = handle, params, (B, H, W)
        ctx.save_for_backward(s0c, s1c, w, w2, out, saved, stats)
        return out

    @staticmethod
    def backward(ctx, gout):
        s0, s1, w, w2, out, saved, stats = ctx.saved_tensors
        handle, params = ctx.handle, ctx.params
        lib = N.lib_for(s1)
        B, H, W = ctx.geom
        sz = handle.sizes(lib, B, H, W)
        dev = s1.device
        gout = _f32c(gout)
        need_in = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        need_par = len(params) > 0 and any(ctx.needs_input_grad[5:])
        gs0 = _empty_like(s0) if need_in else None
        gs1 = _empty_like(s1) if need_in else None
        gw = _empty_like(w)
        gw2 = _empty_like(w2)
        gpar = _empty(sz.param_floats, torch.float32, dev) if need_par else None
        work = _empty(sz.bwd_work_floats, torch.float32, dev)
        bstats = _empty(sz.bwd_stats_doubles, torch.float64, dev)
        a = N.CellBwdArgs(handle.shape(B, H, W), N.ptr(s0), N.ptr(s1), N.ptr(w), N.ptr(w2), handle.param_ptr,
                          N.ptr(out), N.ptr(saved), N.ptr(stats), N.ptr(gout), N.ptr(gs0), N.ptr(gs1), N.ptr(gw),
                          N.ptr(gw2), N.ptr(gpar), N.ptr(work), N.ptr(bstats), int(need_par), int(need_in))
        N.check(lib, lib.pcd_cell_backward(C.byref(a), N.stream_for(s1)), "pcd_cell_backward")
        if _OVERLAP["on"] and need_par:        # the aux-stream jobs read all of these until overlap_join()
            _OVERLAP["keep"].append((s0, s1, w, w2, out, saved, stats, gout, gpar, work, bstats))
        if _DEBUG_KEEP is not None:
            _DEBUG_KEEP.append(dict(cfg=handle.cfg, gout=gout, gs0=gs0, gs1=gs1, work=work, bstats=bstats, gpar=gpar,
                                    s0=s0, s1=s1, saved=saved, stats=stats, w=w, w2=w2, sizes=sz))
        pg = _views(gpar, params) if need_par else [None] * len(params)
        return (gs0, gs1, gw, gw2, None, *pg)


# --------------------------------------------------------------------------------------------
# MixedOp on its own
# --------------------------------------------------------------------------------------------
class MixedHandle:
    def __init__(self, channels, stride):
        self.channels, self.stride = channels, stride
        self._sizes = {}
        self.param_ptr = self.running_ptr = self.nbt_ptr = None

    def shape(self, B, H, W):
        return N.MixedShape(B, self.channels, H, W, self.stride, BN_EPS, BN_MOMENTUM)

    def sizes(self, lib, B, H, W):
        key = (B, H, W)
        if key not in self._sizes:
            sz = N.MixedSizes()
            sh = self.shape(B, H, W)
            N.check(lib, lib.pcd_mixedop_sizes_of(C.byref(sh), C.byref(sz)), "pcd_mixedop_sizes_of")
            self._sizes[key] = sz
        return self._sizes[key]


class MixedOpFunction(torch.autograd.Function):
    """MixedOp.forward (model_search.py:44-58) as one autograd node."""

    @staticmethod
    def forward(ctx, x, weights, handle, *params):
        lib = N.lib_for(x)
        xc, w = _f32c(x), _f32c(weights)
        B, Cc, H, W = xc.shape
        sz = handle.sizes(lib, B, H, W)
        dev = xc.device
        out = _empty((B, Cc, sz.out_height, sz.out_width), torch.float32, dev)
        saved = _empty(sz.saved_floats, torch.float32, dev)
        stats = _empty(sz.stats_doubles, torch.float64, dev)
        a = N.MixedFwdArgs(handle.shape(B, H, W), N.ptr(xc), N.ptr(w), handle.param_ptr, handle.running_ptr,
                           handle.nbt_ptr, N.ptr(out), N.ptr(saved), N.ptr(stats))
        N.check(lib, lib.pcd_mixedop_forward(C.byref(a), N.stream_for(xc)), "pcd_mixedop_forward")
        ctx.handle, ctx.params, ctx.geom = handle, params, (B, H, W)
        ctx.save_for_backward(xc, w, saved, stats)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, w, saved, stats = ctx.saved_tensors
        handle, params = ctx.handle, ctx.params
        lib = N.lib_for(x)
        B, H, W = ctx.geom
        sz = handle.sizes(lib, B, H, W)
        dev = x.device
        gout = _f32c(gout)
        need_par = len(params) > 0 and any(ctx.needs_input_grad[3:])
        gx = _empty_like(x)
        gw = _empty_like(w)
        gpar = _empty(sz.param_floats, torch.float32, dev) if need_par else None
        work = _empty(sz.bwd_work_floats, torch.float32, dev)
        bstats = _empty(sz.bwd_stats_doubles, torch.float64, dev)
        a = N.MixedBwdArgs(handle.shape(B, H, W), N.ptr(x), N.ptr(w), handle.param_ptr, N.ptr(saved), N.ptr(stats),
                           N.ptr(gout), N.ptr(gx), N.ptr(gw), N.ptr(gpar), N.ptr(work), N.ptr(bstats), int(need_par))
        N.check(lib, lib.pcd_mixedop_backward(C.byref(a), N.stream_for(x)), "pcd_mixedop_backward")
        pg = _views(gpar, params) if need_par else [None] * len(params)
        return (gx, gw, None, *pg)


# --------------------------------------------------------------------------------------------
# stem, adaptive pool, shuffle
# --------------------------------------------------------------------------------------------
class StemFunction(torch.autograd.Function):
    """Network.stem (model_search.py:110-113): Conv2d(3, 3C, 3, pad 1) + affine BatchNorm2d."""

    @staticmethod
    def forward(ctx, x, ptrs, conv_w, bn_w, bn_b):
        lib = N.lib_for(x)
        xc = _f32c(x)
        B, cin, H, W = xc.shape
        if cin != 3:
            raise ValueError("stem expects 3 input channels")
        cout = conv_w.shape[0]
        dev = xc.device
        out = _empty((B, cout, H, W), torch.float32, dev)
        z = _empty_like(out)
        stats = _empty(2 * cout, torch.float64, dev)
        a = N.StemArgs(B, cout, H, W, BN_EPS, BN_MOMENTUM, N.ptr(xc), ptrs[0], ptrs[1], ptrs[2], N.ptr(out), N.ptr(z),
                       N.ptr(stats), None, None, None, None)
        N.check(lib, lib.pcd_stem_forward(C.byref(a), N.stream_for(xc)), "pcd_stem_forward")
        ctx.ptrs, ctx.meta = ptrs, (B, cout, H, W)
        ctx.shapes = (conv_w.shape, bn_w.shape, bn_b.shape)
        ctx.save_for_backward(xc, z, stats)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, z, stats = ctx.saved_tensors
        if ctx.needs_input_grad[0]:
            raise NotImplementedError("gradient w.r.t. the image is not part of the search path")
        lib = N.lib_for(x)
        overlap_join(x)
        B, cout, H, W = ctx.meta
        gout = _f32c(gout)
        need_par = any(ctx.needs_input_grad[2:])
        if not need_par:
            return (None, None, None, None, None)
        gpar = _empty(cout * 29, torch.float32, x.device)
        bstats = _empty(2 * cout, torch.float64, x.device)
        a = N.StemArgs(B, cout, H, W, BN_EPS, BN_MOMENTUM, N.ptr(x), ctx.ptrs[0], None, None, None, N.ptr(z),
                       N.ptr(stats), N.ptr(gout), None, N.ptr(gpar), N.ptr(bstats))
        N.check(lib, lib.pcd_stem_backward(C.byref(a), N.stream_for(x)), "pcd_stem_backward")
        gw, gg, gb = gpar.split_with_sizes([cout * 27, cout, cout])
        return (None, None, gw.view(ctx.shapes[0]), gg, gb)


class AdaptiveAvgPoolFunction(torch.autograd.Function):
    """Network.global_pooling (model_search.py:129,176)."""

    @staticmethod
    def forward(ctx, x, size):
        lib = N.lib_for(x)
        xc = _f32c(x)
        B, Cc, H, W = xc.shape
        y = _empty((B, Cc, size, size), torch.float32, xc.device)
        N.check(lib, lib.pcd_adaptive_avgpool_forward(N.ptr(xc), N.ptr(y), B, Cc, H, W, size, size, N.stream_for(xc)),
                "pcd_adaptive_avgpool_forward")
        ctx.meta = (B, Cc, H, W, size)
        return y

    @staticmethod
    def backward(ctx, gy):
        B, Cc, H, W, size = ctx.meta
        lib = N.lib_for(gy)
        gy = _f32c(gy)
        gx = _empty((B, Cc, H, W), torch.float32, gy.device)
        N.check(lib, lib.pcd_adaptive_avgpool_backward(N.ptr(gy), N.ptr(gx), B, Cc, H, W, size, size, N.stream_for(gy)),
                "pcd_adaptive_avgpool_backward")
        return gx, None


def _droppath_args(x, meta, **tensors):
    drop1, drop2, keep, seed, cell, node, offset = meta
    B = x.shape[0]
    a = N.DropPathArgs(B, x.numel() // B if B else 0, int(drop1), int(drop2), cell, node, offset, N.ptr(seed), N.ptr(keep))
    for k, t in tensors.items():
        setattr(a, k, N.ptr(t))
    return a


class DropPathSumFunction(torch.autograd.Function):
    """One node of a derived cell, d1 * h1 + d2 * h2 with DARTS's drop-path on the flagged inputs (pcd_droppath_sum_*)."""

    @staticmethod
    def forward(ctx, h1, h2, meta):
        lib = N.lib_for(h1)
        a1, a2 = _f32c(h1), _f32c(h2)
        if a1.shape != a2.shape:
            raise ValueError(f"droppath_sum: inputs of one node differ in shape: {tuple(a1.shape)} vs {tuple(a2.shape)}")
        out = _empty(a1.shape, torch.float32, a1.device)
        N.check(lib, lib.pcd_droppath_sum_forward(C.byref(_droppath_args(a1, meta, h1=a1, h2=a2, out=out)),
                                                  N.stream_for(a1)), "pcd_droppath_sum_forward")
        ctx.meta = meta
        return out

    @staticmethod
    def backward(ctx, g):
        drop1, drop2 = ctx.meta[:2]
        if not (drop1 or drop2):
            return g, g, None
        lib = N.lib_for(g)
        g = _f32c(g)
        g1 = _empty(g.shape, torch.float32, g.device) if drop1 and ctx.needs_input_grad[0] else None
        g2 = _empty(g.shape, torch.float32, g.device) if drop2 and ctx.needs_input_grad[1] else None
        N.check(lib, lib.pcd_droppath_sum_backward(C.byref(_droppath_args(g, ctx.meta, grad_out=g, grad_h1=g1, grad_h2=g2)),
                                                   N.stream_for(g)), "pcd_droppath_sum_backward")
        return (g1 if drop1 else g), (g2 if drop2 else g), None


def droppath_sum(h1, h2, drop1, drop2, keep, seed, cell, node, sample_offset=0):
    """node = d1 * h1 + d2 * h2 of a derived cell (pcdarts/model.py), in one kernel pass.  d_i x = (x / keep) * m_i(b) for a
    flagged input (DARTS's drop_path: x.div_(keep_prob).mul_(mask), one Bernoulli(keep) mask per sample), else x; with no flag
    set, or keep = 1, the result is bit-equal to h1 + h2.  The mask of sample b is a pure function of (seed, sample_offset + b,
    cell, 2 * node + input) (include/pcdarts_sm100.h), recomputed in the backward.

    keep: 1-element float32 tensor on the inputs' device, seed: 1-element int64 tensor there; both are read when the kernel
    runs (a CUDA graph follows what they hold at replay time) and may be None when neither flag is set."""
    if drop1 or drop2:
        for t, dt, what in ((keep, torch.float32, "keep"), (seed, torch.int64, "seed")):
            if not torch.is_tensor(t) or t.dtype != dt or t.numel() != 1 or t.device != h1.device:
                raise ValueError(f"droppath_sum: {what} must be a 1-element {dt} tensor on {h1.device}")
    if sample_offset < 0:
        raise ValueError(f"droppath_sum: sample_offset must be >= 0, got {sample_offset}")
    return DropPathSumFunction.apply(h1, h2, (bool(drop1), bool(drop2), keep, seed, int(cell), int(node), int(sample_offset)))


class ChannelShuffleFunction(torch.autograd.Function):
    """channel_shuffle (model_search.py:14-28); backward is the inverse permutation."""

    @staticmethod
    def forward(ctx, x, groups):
        lib = N.lib_for(x)
        xc = _f32c(x)
        B, Cc, H, W = xc.shape
        y = _empty_like(xc)
        N.check(lib, lib.pcd_channel_shuffle(N.ptr(xc), N.ptr(y), B, Cc, H * W, groups, N.stream_for(xc)),
                "pcd_channel_shuffle")
        ctx.groups = groups
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = N.lib_for(gy)
        gy = _f32c(gy)
        B, Cc, H, W = gy.shape
        gx = _empty_like(gy)
        # inverse of a (groups, C/groups) transpose is the (C/groups, groups) transpose
        N.check(lib, lib.pcd_channel_shuffle(N.ptr(gy), N.ptr(gx), B, Cc, H * W, Cc // ctx.groups, N.stream_for(gy)),
                "pcd_channel_shuffle")
        return gx, None


# --------------------------------------------------------------------------------------------
# stand-alone preprocess ops (ReLUConvBN 1x1 / FactorizedReduce, affine=False)
# --------------------------------------------------------------------------------------------
class PreprocessFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, meta, *weights):
        fr, c_in, c_out, ptrs = meta
        lib = N.lib_for(x)
        xc = _f32c(x)
        B, _, H, W = xc.shape
        ho, wo = (H // 2, W // 2) if fr else (H, W)
        y = _empty((B, c_out, ho, wo), torch.float32, xc.device)
        stats = _empty(2 * c_out, torch.float64, xc.device)
        a = N.PreArgs(B, c_in, c_out, H, W, int(fr), BN_EPS, BN_MOMENTUM, N.ptr(xc), ptrs[0], ptrs[1], ptrs[2],
                      N.ptr(y), N.ptr(stats), None, None, None, None)
        N.check(lib, lib.pcd_preprocess_forward(C.byref(a), N.stream_for(xc)), "pcd_preprocess_forward")
        ctx.meta, ctx.wshapes = (fr, c_in, c_out, ptrs, B, H, W), [w.shape for w in weights]
        ctx.save_for_backward(xc, y, stats)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, y, stats = ctx.saved_tensors
        fr, c_in, c_out, ptrs, B, H, W = ctx.meta
        lib = N.lib_for(x)
        gy = _f32c(gy)
        gx = _empty_like(x) if ctx.needs_input_grad[0] else None
        need_w = any(ctx.needs_input_grad[2:])
        gw = _empty(c_out * c_in, torch.float32, x.device) if need_w else None
        bstats = _empty(2 * c_out, torch.float64, x.device)
        a = N.PreArgs(B, c_in, c_out, H, W, int(fr), BN_EPS, BN_MOMENTUM, N.ptr(x), ptrs[0], None, None, N.ptr(y),
                      N.ptr(stats), N.ptr(gy), N.ptr(gx), N.ptr(gw), N.ptr(bstats))
        N.check(lib, lib.pcd_preprocess_backward(C.byref(a), N.stream_for(x)), "pcd_preprocess_backward")
        if need_w:
            parts = gw.split_with_sizes([s.numel() for s in ctx.wshapes])
            gws = [p.view(s) for p, s in zip(parts, ctx.wshapes)]
        else:
            gws = [None] * len(ctx.wshapes)
        return (gx, None, *gws)


def preprocess_apply(module, x, fr):
    """Stand-alone forward of ReLUConvBN(k=1) / FactorizedReduce through the Cell's preprocess kernels."""
    if fr:
        c_in, c_out, affine = module._spec
        bn = module.bn
    else:
        c_in, c_out, k, stride, pad, affine = module._spec
        if (k, stride, pad) != (1, 1, 0):
            raise NotImplementedError("only the 1x1/stride 1/pad 0 ReLUConvBN of the search network is accelerated")
        bn = module.op[2]
    is_eval = eval_forward(module, x)
    if not hasattr(module, "_pcd_arena"):
        module._pcd_arena = Arena(module)
    ar = module._pcd_arena.ensure()
    if is_eval:
        return preprocess_forward_eval(x, fr, c_in, c_out, ar.param_ptr, ar.running_ptr,
                                       bn.weight if affine else None, bn.bias if affine else None)
    meta = (fr, c_in, c_out, (ar.param_ptr, ar.running_ptr, ar.nbt_ptr))
    convs = [module.conv_1.weight, module.conv_2.weight] if fr else [module.op[1].weight]     # first in the arena, back to back
    yhat = PreprocessFunction.apply(x, meta, *convs)
    if affine:          # BatchNorm2d(affine=True): gamma * yhat + beta on the affine kernel (pcd_opmods.ChannelAffineFunction)
        from pcd_opmods import affine_apply
        return affine_apply(yhat, bn)
    return yhat


# --------------------------------------------------------------------------------------------
# eval mode: BatchNorm from running statistics, forward only (plain calls, no autograd Functions)
# --------------------------------------------------------------------------------------------
def autograd_records(tensors):
    """True when a forward over `tensors` would be recorded by autograd."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def eval_forward(module, *inputs):
    """True when `module` is in eval mode, i.e. its forward runs the eval kernels.  There is no eval-mode backward, so eval
    mode while autograd records (grad enabled and any parameter or input requiring grad) raises NotImplementedError."""
    if module.training:
        return False
    if autograd_records(inputs) or autograd_records(module.parameters()):
        raise NotImplementedError(
            f"{type(module).__name__} in eval mode (BatchNorm from running statistics) is forward-only: wrap the call in "
            "torch.no_grad() or torch.inference_mode(), or call .train() to differentiate")
    return True


def cell_forward_eval(s0, s1, weights, weights2, handle):
    """Cell.forward in eval mode: two preprocess launches + one launch per node."""
    lib = N.lib_for(s1)
    s0c, s1c, w, w2 = _f32c(s0), _f32c(s1), _f32c(weights), _f32c(weights2)
    B, _, H, W = s1c.shape
    sz = handle.sizes(lib, B, H, W)
    out = _empty((B, 4 * handle.cfg[2], sz.out_height, sz.out_width), torch.float32, s1c.device)
    sh = handle.shape(B, H, W)
    nwork = C.c_int64()
    N.check(lib, lib.pcd_cell_eval_work_floats(C.byref(sh), C.byref(nwork)), "pcd_cell_eval_work_floats")
    work = _empty(nwork.value, torch.float32, s1c.device)
    a = N.CellEvalArgs(sh, N.ptr(s0c), N.ptr(s1c), N.ptr(w), N.ptr(w2), handle.param_ptr, handle.running_ptr, N.ptr(out),
                       N.ptr(work))
    N.check(lib, lib.pcd_cell_forward_eval(C.byref(a), N.stream_for(s1c)), "pcd_cell_forward_eval")
    return out


def mixedop_forward_eval(x, weights, handle):
    lib = N.lib_for(x)
    xc, w = _f32c(x), _f32c(weights)
    B, Cc, H, W = xc.shape
    sz = handle.sizes(lib, B, H, W)
    out = _empty((B, Cc, sz.out_height, sz.out_width), torch.float32, xc.device)
    a = N.MixedEvalArgs(handle.shape(B, H, W), N.ptr(xc), N.ptr(w), handle.param_ptr, handle.running_ptr, N.ptr(out))
    N.check(lib, lib.pcd_mixedop_forward_eval(C.byref(a), N.stream_for(xc)), "pcd_mixedop_forward_eval")
    return out


def stem_forward_eval(x, param_ptr, running_ptr, c_out):
    lib = N.lib_for(x)
    xc = _f32c(x)
    B, cin, H, W = xc.shape
    if cin != 3:
        raise ValueError("stem expects 3 input channels")
    out = _empty((B, c_out, H, W), torch.float32, xc.device)
    a = N.StemEvalArgs(B, c_out, H, W, BN_EPS, N.ptr(xc), param_ptr, running_ptr, N.ptr(out))
    N.check(lib, lib.pcd_stem_forward_eval(C.byref(a), N.stream_for(xc)), "pcd_stem_forward_eval")
    return out


def preprocess_forward_eval(x, fr, c_in, c_out, weight_ptr, running_ptr, gamma=None, beta=None):
    lib = N.lib_for(x)
    xc = _f32c(x)
    B, _, H, W = xc.shape
    ho, wo = (H // 2, W // 2) if fr else (H, W)
    y = _empty((B, c_out, ho, wo), torch.float32, xc.device)
    g = _f32c(gamma) if gamma is not None else None
    b = _f32c(beta) if beta is not None else None
    a = N.PreEvalArgs(B, c_in, c_out, H, W, int(fr), BN_EPS, N.ptr(xc), weight_ptr, running_ptr, N.ptr(g), N.ptr(b), N.ptr(y))
    N.check(lib, lib.pcd_preprocess_forward_eval(C.byref(a), N.stream_for(xc)), "pcd_preprocess_forward_eval")
    return y


# --------------------------------------------------------------------------------------------
# dense projection on the tcgen05 tensor cores (3xTF32, fp32 accumulation): nn.Linear drop-in
# --------------------------------------------------------------------------------------------
def _pad4(n):
    return (n + 3) // 4 * 4


def _gemm_tn(lib, a, lda, b, ldb, c, ldc, m, n, k, bias, split_k, ref):
    N.check(lib, lib.pcd_gemm_tn_3xtf32(N.ptr(a), lda, N.ptr(b), ldb, N.ptr(c), ldc, m, n, k, N.ptr(bias), split_k,
                                        N.stream_for(ref)), "pcd_gemm_tn_3xtf32")


# nn.Linear products of at least 0.5 GFLOP (vocabulary projection, LSTM projections, image fc) run on the tcgen05 GEMM;
# the small ones (answer head fc1 / fc2, question fc2 at batch 64: 0.07 - 0.13 GFLOP, bound by launch latency and one read of
# W) run on the library's own exact-fp32 FMA kernel pcd_gemm_small_f32 — no cuBLAS either way.  They are kept off 3xTF32
# on purpose: the search network's gradients amplify the head's rounding noise ~100x (measured on the full-size step: median
# weight-gradient error against float64 9e-5 with the fp32 head, 5e-4 with the 3xTF32 head; fp32 oracle itself 2e-4).
_TC_MIN_FLOP = float(os.environ.get("PCD_TC_MIN_FLOP", "5e8"))

# Shapes outside the kernels' envelope (a Linear whose depth is not a multiple of 4, an LSTM whose hidden size is not a power
# of two, ...) raise instead of quietly running stock torch ops.  Tests that pin the reference's toy dimensions (hidden 16,
# word embedding 10) opt in explicitly with allow_stock_ops(True).
_ALLOW_STOCK = [False]


def allow_stock_ops(on=True):
    """Opt in to stock torch ops for shapes the native kernels do not take (default: raise).  Returns the previous setting."""
    prev = _ALLOW_STOCK[0]
    _ALLOW_STOCK[0] = bool(on)
    return prev


def _stock(what):
    if not _ALLOW_STOCK[0]:
        raise RuntimeError(f"{what}: shape not supported by the compiled kernels (PCD_ERR_UNSUPPORTED); "
                           "pcd_ops.allow_stock_ops(True) opts in to the stock torch op")


_SMS = 148          # B200


def _auto_split(m, n, k):
    """K split of pcd_gemm_tn_3xtf32 when the output has fewer tiles than SMs.  The persistent kernel deals its work items
    (tile x split) round-robin to one CTA per SM, so the time is rounds x (k-blocks per item + pipeline fill): 30 tiles x 5 splits
    = 150 items is TWO rounds on 148 SMs (the previous rule, ceil(148 / tiles)), 30 x 4 = 120 items one.  Fewest splits within
    2 % of the best (each split adds one atomic pass over the output); >= 8 k-blocks per split; tiles as the kernel picks them
    (128 x 256 x 16 for N >= 256, else 128 x 128 x 32)."""
    bn, bk = (256, 16) if n >= 256 else (128, 32)
    tiles = ((m + 127) // 128) * ((n + bn - 1) // bn)
    kb = (k + bk - 1) // bk
    smax = max(1, min(32, kb // 8))
    if tiles >= _SMS or smax == 1:
        return 1
    cost = {s: -(-tiles * s // _SMS) * (kb / s + 8.0) for s in range(1, smax + 1)}
    best = min(cost.values())
    return min(s for s, c in cost.items() if c <= 1.02 * best)


class Linear3xTF32Function(torch.autograd.Function):
    """y = x @ W^T + b through pcd_gemm_tn_3xtf32 (nn.Linear drop-in; the vocabulary projection vqa_model.py:192-194, the
    image `fc` vqa_model.py:56,61, the question `fc2` and the answer head vqa_model.py:308-316).

    The TMA descriptors need 16-byte row pitches: y, its gradient and the transposed operands of the backward products
    live in buffers whose row pitch is rounded up to a multiple of 4 (pad columns are zero); y is returned as a view.
    """

    @staticmethod
    def forward(ctx, x, weight, bias):
        lib = N.lib_for(x)
        x2 = _f32c(x.reshape(-1, x.shape[-1]))
        w = _f32c(weight)
        m, k = x2.shape
        n = w.shape[0]
        npad = _pad4(n)
        out = _empty((m, npad), torch.float32, x2.device)
        _gemm_tn(lib, x2, k, w, k, out, npad, m, n, k, _f32c(bias) if bias is not None else None, _auto_split(m, n, k), x2)
        ctx.save_for_backward(x2, w)
        ctx.meta = (x.shape, n, npad, bias is not None)
        return out[:, :n].view(*x.shape[:-1], n)

    @staticmethod
    def backward(ctx, gy):
        x2, w = ctx.saved_tensors
        xshape, n, npad, has_bias = ctx.meta
        lib = N.lib_for(x2)
        m, k = x2.shape
        g2 = _f32c(gy.reshape(m, n))
        gx = gw = gb = None
        need_w, need_b = _param_grads(ctx, 1, 2 if has_bias else None)
        if ctx.needs_input_grad[0]:
            if npad == n:
                gp = g2
            else:
                gp = _empty((m, npad), torch.float32, x2.device)    # dL/dy with a 16-byte row pitch
                gp[:, :n].copy_(g2)
                gp[:, n:].zero_()
            wt = _transpose_pad(lib, w, k, n, k, npad, x2)          # W^T (k, npad)
            gx2 = _empty((m, k), torch.float32, x2.device)
            _gemm_tn(lib, gp, npad, wt, npad, gx2, k, m, k, npad, None, _auto_split(m, k, npad), x2)
            gx = gx2.view(xshape)
        if need_w or need_b:
            mp = _pad4(m)
            gt = _transpose_pad(lib, g2, n, m, n, mp, x2)           # (n, mp)
            if need_b:
                gb = gt.sum(1)
            if need_w:
                xt = _transpose_pad(lib, x2, k, m, k, mp, x2)       # (k, mp)
                gw = _empty((n, k), torch.float32, x2.device)
                _gemm_tn(lib, gt, mp, xt, mp, gw, k, n, k, mp, None, _auto_split(n, k, mp), x2)
        return gx, gw, gb


class SmallLinearFunction(torch.autograd.Function):
    """y = x @ W^T + b for the small heads through pcd_gemm_small_f32 (exact fp32 FMA; strides instead of transposes)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        lib = N.lib_for(x)
        x2 = _f32c(x.reshape(-1, x.shape[-1]))
        w = _f32c(weight)
        m, k = x2.shape
        n = w.shape[0]
        y = _empty((m, n), torch.float32, x2.device)
        N.check(lib, lib.pcd_gemm_small_f32(N.ptr(x2), k, 1, N.ptr(w), k, 1, N.ptr(y), n, m, n, k,
                                            N.ptr(_f32c(bias)) if bias is not None else None, N.stream_for(x2)), "pcd_gemm_small_f32")
        ctx.save_for_backward(x2, w)
        ctx.meta = (x.shape, bias is not None)
        return y.view(*x.shape[:-1], n)

    @staticmethod
    def backward(ctx, gy):
        x2, w = ctx.saved_tensors
        xshape, has_bias = ctx.meta
        lib = N.lib_for(x2)
        m, k = x2.shape
        n = w.shape[0]
        g2 = _f32c(gy.reshape(m, n))
        st = N.stream_for(x2)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:         # dx[m][k] = sum_n dy[m][n] W[n][k]
            gx2 = _empty((m, k), torch.float32, x2.device)
            N.check(lib, lib.pcd_gemm_small_f32(N.ptr(g2), n, 1, N.ptr(w), 1, k, N.ptr(gx2), k, m, k, n, None, st), "pcd_gemm_small_f32")
            gx = gx2.view(xshape)
        need_w, need_b = _param_grads(ctx, 1, 2 if has_bias else None)
        if need_w:                          # dW[n][k] = sum_m dy[m][n] x[m][k]
            gw = _empty((n, k), torch.float32, x2.device)
            N.check(lib, lib.pcd_gemm_small_f32(N.ptr(g2), 1, n, N.ptr(x2), 1, k, N.ptr(gw), k, n, k, m, None, st), "pcd_gemm_small_f32")
        if need_b:
            gb = g2.sum(0)
        return gx, gw, gb


def linear_3xtf32(x, weight, bias):
    """nn.Linear forward: tcgen05 GEMM for the large products, the exact-fp32 FMA kernel for the small ones and for depths
    TMA cannot take (not a multiple of 4).  Never a library GEMM."""
    if not (x.is_cuda or N._emu_lib is not None):
        raise RuntimeError("pcdarts_sm100 kernels need CUDA tensors (no CPU fallback)")
    m = x.numel() // x.shape[-1]
    if x.shape[-1] % 4 or 2.0 * m * weight.shape[0] * weight.shape[1] < _TC_MIN_FLOP:
        return SmallLinearFunction.apply(x, weight, bias)      # no alignment requirement: also takes what TMA cannot
    return Linear3xTF32Function.apply(x, weight, bias)


def _transpose_pad(lib, src, ld_s, rows, cols, ld_d, ref):
    """(cols, ld_d) buffer with dst[c][r] = src[r][c]; columns >= rows are zero."""
    dst = _empty((cols, ld_d), torch.float32, ref.device)
    N.check(lib, lib.pcd_transpose_pad(N.ptr(src), ld_s, rows, cols, N.ptr(dst), ld_d, N.stream_for(ref)), "pcd_transpose_pad")
    return dst


class VocabCrossEntropyFunction(torch.autograd.Function):
    """mean_r CE(x_r @ W^T + b, target_r) over the rows with 0 <= target < V  — the question-decoder loss
    (vqa_model.py:192-194 + 356-358) without ever slicing or re-laying-out the (B*T, V) logits: projection on the
    tensor cores into a 16-byte-pitch buffer, row statistics and the loss from it, gradient written in the same layout,
    transposed once for the K-major operand of dW."""

    @staticmethod
    def forward(ctx, x, weight, bias, targets):
        lib = N.lib_for(x)
        x2 = _f32c(x.reshape(-1, x.shape[-1]))
        w = _f32c(weight)
        m, k = x2.shape
        v = w.shape[0]
        vp = _pad4(v)
        tg = targets.reshape(-1).contiguous()
        logits = _empty((m, vp), torch.float32, x2.device)
        _gemm_tn(lib, x2, k, w, k, logits, vp, m, v, k, _f32c(bias) if bias is not None else None, 1, x2)
        lse = _empty(m, torch.float32, x2.device)
        rows = _empty(m, torch.float32, x2.device)
        N.check(lib, lib.pcd_ce_forward(N.ptr(logits), vp, m, v, N.ptr(tg), N.ptr(lse), N.ptr(rows), N.stream_for(x2)), "pcd_ce_forward")
        # a row is ignored when its target is negative or >= V (the kernels score both 0); checked on the device, so the
        # step stays capturable: a host-side range check would synchronise
        nvalid = ((tg >= 0) & (tg < v)).sum().clamp_min(1).to(torch.float32)
        ctx.save_for_backward(x2, w, logits, lse, tg, nvalid)
        ctx.meta = (x.shape, v, vp, bias is not None)
        return rows.sum() / nvalid

    @staticmethod
    def backward(ctx, g):
        x2, w, logits, lse, tg, nvalid = ctx.saved_tensors
        xshape, v, vp, has_bias = ctx.meta
        lib = N.lib_for(x2)
        m, k = x2.shape
        scale = (g / nvalid).to(torch.float32).reshape(1).contiguous()
        dl = _empty((m, vp), torch.float32, x2.device)
        N.check(lib, lib.pcd_ce_backward(N.ptr(logits), vp, m, v, N.ptr(tg), N.ptr(lse), N.ptr(scale), N.ptr(dl),
                                         N.stream_for(x2)), "pcd_ce_backward")
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            wt = _transpose_pad(lib, w, k, v, k, vp, x2)                     # W^T (k, vp)
            gx2 = _empty((m, k), torch.float32, x2.device)
            _gemm_tn(lib, dl, vp, wt, vp, gx2, k, m, k, vp, None, _auto_split(m, k, vp), x2)
            gx = gx2.view(xshape)
        need_w, need_b = _param_grads(ctx, 1, 2 if has_bias else None)
        if need_w or need_b:
            mp = _pad4(m)
            dlt = _transpose_pad(lib, dl, vp, m, v, mp, x2)                  # dlogits^T (v, mp)
            if need_b:
                gb = dlt.sum(1)
            if need_w:
                xt = _transpose_pad(lib, x2, k, m, k, mp, x2)                # h^T (k, mp)
                gw = _empty((v, k), torch.float32, x2.device)
                _gemm_tn(lib, dlt, mp, xt, mp, gw, k, v, k, mp, None, 1, x2)
        return gx, gw, gb, None


def vocab_cross_entropy(x, weight, bias, targets):
    """Fused projection + cross-entropy (ignore a target < 0 or >= V, mean over the rest); a depth that is not a multiple of 4 raises
    unless allow_stock_ops."""
    if not (x.is_cuda or N._emu_lib is not None):
        raise RuntimeError("pcdarts_sm100 kernels need CUDA tensors (no CPU fallback)")
    if x.shape[-1] % 4:
        _stock(f"vocabulary projection with depth {x.shape[-1]}")
        logits = torch.nn.functional.linear(x, weight, bias)
        return torch.nn.functional.cross_entropy(logits.reshape(-1, logits.shape[-1]), targets.reshape(-1), ignore_index=-100)
    return VocabCrossEntropyFunction.apply(x, weight, bias, targets)


# --------------------------------------------------------------------------------------------
# single-layer LSTM: dense projections on tcgen05, recurrence in persistent cooperative kernels
# --------------------------------------------------------------------------------------------
class LstmFunction(torch.autograd.Function):
    """nn.LSTM(E, H, 1) forward/backward (time-major input (T, B, E), h0 = c0 given) — vqa_model.py:165,176-184.

    gx = x W_ih^T + (b_ih + b_hh) and the four backward products (dx, dW_ih, dW_hh over all T*B rows) go through
    pcd_gemm_tn_3xtf32; the two recurrences through pcd_lstm_forward / pcd_lstm_backward."""

    @staticmethod
    def forward(ctx, x, h0, c0, w_ih, w_hh, b_ih, b_hh):
        lib = N.lib_for(x)
        xc, h0c, c0c, wi, wh = _f32c(x), _f32c(h0), _f32c(c0), _f32c(w_ih), _f32c(w_hh)
        T, B, E = xc.shape
        H = wh.shape[1]
        dev = xc.device
        x2 = xc.view(T * B, E)
        gx = _empty((T * B, 4 * H), torch.float32, dev)
        _gemm_tn(lib, x2, E, wi, E, gx, 4 * H, T * B, 4 * H, E, (b_ih + b_hh).detach().contiguous(), _auto_split(T * B, 4 * H, E), xc)
        act = _empty((T, B, 4 * H), torch.float32, dev)
        cs = _empty((T, B, H), torch.float32, dev)
        hs = _empty((T, B, H), torch.float32, dev)
        N.check(lib, lib.pcd_lstm_forward(T, B, H, N.ptr(gx), N.ptr(wh), N.ptr(h0c), N.ptr(c0c), N.ptr(act), N.ptr(cs), N.ptr(hs),
                                          N.stream_for(xc)), "pcd_lstm_forward")
        ctx.save_for_backward(xc, h0c, c0c, wi, wh, act, cs, hs)
        return hs, hs[T - 1].clone(), cs[T - 1].clone()

    @staticmethod
    def backward(ctx, dhs, dhT, dcT):
        xc, h0c, c0c, wi, wh, act, cs, hs = ctx.saved_tensors
        lib = N.lib_for(xc)
        T, B, E = xc.shape
        H = wh.shape[1]
        dev = xc.device
        dhs = _f32c(dhs) if dhs is not None else None
        dhT = _f32c(dhT) if dhT is not None else None
        dcT = _f32c(dcT) if dcT is not None else None
        dg = _empty((T * B, 4 * H), torch.float32, dev)
        dh0 = _empty((B, H), torch.float32, dev)
        dc0 = _empty((B, H), torch.float32, dev)
        pbuf = _empty(lib.pcd_lstm_pbuf_floats(B, H), torch.float32, dev)
        N.check(lib, lib.pcd_lstm_backward(T, B, H, N.ptr(dhs), N.ptr(dhT), N.ptr(dcT), N.ptr(act), N.ptr(cs), N.ptr(c0c), N.ptr(wh),
                                           N.ptr(dg), N.ptr(dh0), N.ptr(dc0), N.ptr(pbuf), N.stream_for(xc)), "pcd_lstm_backward")
        m = T * B
        gx_in = gwi = gwh = gb = None
        if ctx.needs_input_grad[0]:
            wit = _transpose_pad(lib, wi, E, 4 * H, E, 4 * H, xc)              # W_ih^T (E, 4H)
            gx_in = _empty((m, E), torch.float32, dev)
            _gemm_tn(lib, dg, 4 * H, wit, 4 * H, gx_in, E, m, E, 4 * H, None, _auto_split(m, E, 4 * H), xc)
            gx_in = gx_in.view(T, B, E)
        need_wi, need_wh, need_bi, need_bh = _param_grads(ctx, 3, 4, 5, 6)
        if need_wi or need_wh or need_bi or need_bh:
            mp = _pad4(m)
            dgt = _transpose_pad(lib, dg, 4 * H, m, 4 * H, mp, xc)             # dgates^T (4H, mp)
            gb = dgt.sum(1) if (need_bi or need_bh) else None
            if need_wi:
                xt = _transpose_pad(lib, xc.view(m, E), E, m, E, mp, xc)       # x^T (E, mp)
                gwi = _empty((4 * H, E), torch.float32, dev)
                _gemm_tn(lib, dgt, mp, xt, mp, gwi, E, 4 * H, E, mp, None, _auto_split(4 * H, E, mp), xc)
            if need_wh:
                hprev = torch.cat((h0c.unsqueeze(0), hs[:-1]), 0).view(m, H)   # h_{t-1} for every step
                ht = _transpose_pad(lib, hprev, H, m, H, mp, xc)               # (H, mp)
                gwh = _empty((4 * H, H), torch.float32, dev)
                _gemm_tn(lib, dgt, mp, ht, mp, gwh, H, 4 * H, H, mp, None, _auto_split(4 * H, H, mp), xc)
        return (gx_in, dh0 if ctx.needs_input_grad[1] else None, dc0 if ctx.needs_input_grad[2] else None, gwi, gwh,
                gb if need_bi else None,
                # b_ih and b_hh get the same values but must not share one buffer: in-place consumers (the data-parallel
                # all-reduce, the flat clip scaling) would otherwise touch it twice — concurrently, in the clip kernel
                (gb.clone() if need_bi else gb) if need_bh else None)


_LSTM_BATCH = 64        # rows one launch of the cooperative recurrence / decode kernels takes; larger batches are tiled


def lstm_supported(x, hidden):
    """Shapes the cooperative recurrence kernels take: hidden a power of two in [16, 512], E % 4 == 0 (any batch: tiled by 64)."""
    return (x.is_cuda or N._emu_lib is not None) and x.dim() == 3 and x.shape[2] % 4 == 0 and \
        16 <= hidden <= 512 and (hidden & (hidden - 1)) == 0


def lstm_forward(lstm, x, h0, c0):
    """nn.LSTM(x, (h0, c0)) for a single-layer unidirectional module on the native kernels.  The recurrence is independent per
    sample, so a batch above 64 runs as ceil(B / 64) launches over contiguous slices (no stock fallback)."""
    if lstm.num_layers != 1 or lstm.bidirectional or lstm.batch_first or not lstm_supported(x, lstm.hidden_size):
        _stock(f"LSTM(E={x.shape[-1]}, H={lstm.hidden_size}, layers={lstm.num_layers})")
        out, (h, c) = lstm(x, (h0, c0))
        return out, (h, c)
    B = x.shape[1]
    w = (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0)
    if B <= _LSTM_BATCH:
        out, hT, cT = LstmFunction.apply(x, h0[0], c0[0], *w)
        return out, (hT.unsqueeze(0), cT.unsqueeze(0))
    outs, hs, cs = [], [], []
    for b0 in range(0, B, _LSTM_BATCH):
        sl = slice(b0, min(B, b0 + _LSTM_BATCH))
        o, h, c = LstmFunction.apply(x[:, sl].contiguous(), h0[0, sl].contiguous(), c0[0, sl].contiguous(), *w)
        outs.append(o); hs.append(h); cs.append(c)
    return torch.cat(outs, 1), (torch.cat(hs, 0).unsqueeze(0), torch.cat(cs, 0).unsqueeze(0))


# --------------------------------------------------------------------------------------------
# Question decode (QstEncoder.generate): one persistent cooperative kernel, greedy, sampled or beam search
# --------------------------------------------------------------------------------------------
def decode_supported(h0, lstm, word2vec, proj):
    """Shapes pcd_decode takes in greedy and sampled mode (single-layer LSTM, hidden a multiple of 32 up to 512, E % 4 == 0;
    any batch: tiled by 64)."""
    H = lstm.hidden_size
    return (h0.is_cuda or N._emu_lib is not None) and lstm.num_layers == 1 and not lstm.bidirectional and lstm.bias and \
        32 <= H <= 512 and H % 32 == 0 and word2vec.embedding_dim % 4 == 0 and \
        proj.in_features == H and proj.bias is not None and h0.dtype == torch.float32


def _decode_stop(V, end_token, pad_token, length_penalty=0.0):
    """(end_token, pad_token, length_penalty as fp32) of an end-of-sequence decode (None for end_token=None: no stop).
    ValueError for an end or pad word outside [0, V) or a length penalty that is not finite."""
    if end_token is None:                               # every hypothesis has max_length words: length_penalty is not used
        return None
    a32 = C.c_float(float(length_penalty)).value        # what the kernel divides by
    if not math.isfinite(a32):
        raise ValueError(f"decode: length_penalty must be finite, got {length_penalty}")
    for name, w in (("end_token", end_token), ("pad_token", pad_token)):
        if isinstance(w, bool) or int(w) != w or not 0 <= w < V:
            raise ValueError(f"decode: {name} must be an integer in [0, vocabulary size {V}), got {w}")
    return int(end_token), int(pad_token), a32


def _check_envelope(what, h0, lstm, word2vec, proj):
    """Modes that exist on the decode kernel only (beams, end-of-sequence decoding): no stock loop outside its envelope."""
    if not decode_supported(h0, lstm, word2vec, proj):
        raise RuntimeError(f"{what}: LSTM(layers={lstm.num_layers}, H={lstm.hidden_size}) with E = "
                           f"{word2vec.embedding_dim} is outside the decode kernel's envelope (PCD_ERR_UNSUPPORTED)")


def _decode_truncation(V, top_k, top_p):
    """(top_k, top_p as fp32) of a truncated sampled decode, None for the defaults (top_k = 0, top_p = 1: no truncation).
    ValueError for a top_k that is not a non-negative integer or a top_p outside (0, 1]."""
    if isinstance(top_k, bool) or not isinstance(top_k, numbers.Integral) or top_k < 0:
        raise ValueError(f"decode_sample: top_k must be a non-negative integer (0: no limit), got {top_k!r}")
    p32 = C.c_float(float(top_p)).value                 # what the kernel compares against
    if not math.isfinite(p32) or not 0.0 < p32 <= 1.0:
        raise ValueError(f"decode_sample: top_p must lie in (0, 1], got {top_p!r}")
    if top_k == 0 and p32 == 1.0:
        return None
    return min(int(top_k), V), p32                      # any top_k >= V keeps every word


def _decode(mode, h0, lstm, word2vec, proj, max_length, start_token, K=1, temperature=1.0, seed=None, stop=None,
            truncation=None):
    """One pcd_decode per slice of floor(64 / K) items (the kernel takes 64 rows; row_offset = the slice's first item), each
    with its own outputs and workspace.  Returns (tokens, scores): tokens (B, max_length) and scores None, or for beams
    tokens (B, K, max_length) and scores (B, K).  The arguments are validated by the caller; stop: _decode_stop's tuple,
    truncation: _decode_truncation's."""
    lib = N.lib_for(h0)
    V, E = word2vec.weight.shape
    beam = mode == N.DECODE_BEAM
    ops = [_f32c(t) for t in (word2vec.weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0)]
    wout, bout = _f32c(proj.weight), _f32c(proj.bias)
    end_token, pad_token, length_penalty = stop or (0, 0, 0.0)
    top_k, top_p = truncation or (0, 1.0)
    per = _LSTM_BATCH // K
    tokens, scores = [], []
    for b0 in range(0, max(h0.shape[0], 1), per):       # an empty batch reaches the kernel, which rejects it
        h0c = _f32c(h0[b0:b0 + per])
        B, H = h0c.shape
        tok = torch.empty((B, K, max_length) if beam else (B, max_length), dtype=torch.long, device=h0.device)
        sc = torch.empty((B, K), dtype=torch.float32, device=h0.device) if beam else None
        a = N.DecodeArgs(mode=mode, T=max_length, B=B, K=K, H=H, E=E, V=V, start_token=start_token, stop=stop is not None,
                         end_token=end_token, pad_token=pad_token, length_penalty=length_penalty, temperature=temperature,
                         row_offset=b0, truncate=truncation is not None, top_k=top_k, top_p=top_p, seed=N.ptr(seed),
                         emb=N.ptr(ops[0]), w_ih=N.ptr(ops[1]), w_hh=N.ptr(ops[2]),
                         b_ih=N.ptr(ops[3]), b_hh=N.ptr(ops[4]), h0=N.ptr(h0c), c0=N.ptr(h0c), w_out=N.ptr(wout),
                         b_out=N.ptr(bout), tokens=N.ptr(tok), scores=N.ptr(sc))
        work = torch.empty(int(lib.pcd_decode_work_floats(C.byref(a))), dtype=torch.float32, device=h0.device)
        a.work = N.ptr(work)
        N.check(lib, lib.pcd_decode(C.byref(a), N.stream_for(h0)), "pcd_decode")
        tokens.append(tok)
        scores.append(sc)
    if len(tokens) == 1:
        return tokens[0], scores[0]
    return torch.cat(tokens, 0), (torch.cat(scores, 0) if beam else None)


def decode_greedy(h0, lstm, word2vec, proj, max_length, start_token=2, end_token=None, pad_token=0):
    """tokens (B, max_length) int64 of the greedy decode that starts from `start_token` with h0 = c0 = `h0` (B, H).
    end_token: once a row has emitted it, its later positions are `pad_token`: the unstopped decode truncated after the
    first end_token, and the kernel stops when every row of a launch has finished.
    Not differentiable (neither is the reference's argmax): parameters are read detached."""
    stop = _decode_stop(proj.out_features, end_token, pad_token)
    if stop is not None:
        _check_envelope("decode_greedy", h0, lstm, word2vec, proj)
    return _decode(N.DECODE_GREEDY, h0, lstm, word2vec, proj, max_length, start_token, stop=stop)[0]


def decode_sample(h0, lstm, word2vec, proj, max_length, temperature, start_token=2, seed=None, end_token=None, pad_token=0,
                  top_k=0, top_p=1.0):
    """tokens (B, max_length) int64 of the sampled decode (QstEncoder.sample with deterministic=False): every word is drawn from
    softmax(logits / temperature), by the Gumbel-max trick on counter-based Philox noise (pcd_decode in sampled mode).

    top_k > 0 draws only among the top_k most likely words, top_p < 1 only among the smallest set of most likely words whose
    probability reaches top_p (the nucleus, taken within the top-k words when both are set): the distribution is
    softmax(logits / temperature) restricted to that set and renormalised, with the same noise (pcd_decode with truncate = 1;
    pcdarts_sm100.h states the rule exactly).  The defaults keep every word and run the untruncated kernel.  Truncation has
    no stock loop: outside the decode kernel's envelope it raises, even with allow_stock_ops(True).

    seed: None draws one 64-bit seed per call on h0's device from torch's generator (so torch.manual_seed reproduces a run, and
    a call captured in a CUDA graph draws a fresh seed on every replay); a Python int, or a 1-element int64 tensor on h0's
    device read when the kernel runs, fixes the words.  Batches above 64 are decoded in slices of 64 with one seed: the noise
    of a row depends on its index in the whole batch, so the words do not depend on the slicing.  end_token / pad_token as
    decode_greedy: the same words up to the first end_token.  Not differentiable."""
    t32 = C.c_float(float(temperature)).value           # what the kernel divides by
    if not math.isfinite(t32) or t32 <= 0.0:
        raise ValueError(f"decode_sample: temperature must be finite and > 0, got {temperature}")
    stop = _decode_stop(proj.out_features, end_token, pad_token)
    truncation = _decode_truncation(proj.out_features, top_k, top_p)
    if stop is not None or truncation is not None:
        _check_envelope("decode_sample", h0, lstm, word2vec, proj)
    if seed is None:
        seed = torch.empty(1, dtype=torch.int64, device=h0.device).random_(-2 ** 63, None)
    elif not torch.is_tensor(seed):
        s = int(seed) & (2 ** 64 - 1)                   # the uint64 the kernel reads, stored as int64
        seed = torch.tensor([s - 2 ** 64 if s >= 2 ** 63 else s], dtype=torch.int64, device=h0.device)
    elif seed.dtype != torch.int64 or seed.numel() != 1 or seed.device != h0.device:
        raise ValueError("decode_sample: seed must be an int or a 1-element int64 tensor on the device of h0")
    return _decode(N.DECODE_SAMPLED, h0, lstm, word2vec, proj, max_length, start_token, temperature=t32, seed=seed,
                   stop=stop, truncation=truncation)[0]


_MAX_BEAM = 8


def decode_beam(h0, lstm, word2vec, proj, max_length, beam_size, start_token=2, end_token=None, pad_token=0,
                length_penalty=0.0):
    """Beam search over exactly `max_length` words from `start_token` with h0 = c0 = `h0` (B, H) (pcd_decode in beam mode): at
    every step each item keeps the `beam_size` = K paths of highest cumulative log-probability.  Returns (tokens (B, K,
    max_length) int64, scores (B, K) float32), beams best first; beam_size = 1 is the greedy decode scored by its
    log-probability.
    end_token: a beam whose last word is end_token is finished and continues with `pad_token` at no cost; beams are ranked
    by score / length^length_penalty (length counting end_token), scores are the log-probabilities of the paths up to
    end_token, and the kernel stops once every beam of a launch has finished.  Without end_token every hypothesis has
    max_length words and length_penalty is not used.
    Batches are decoded in slices of floor(64 / K) items (the kernel takes 64 rows); items are independent, so the result does
    not depend on the slicing.  Not differentiable: parameters are read detached."""
    V = proj.out_features
    if isinstance(beam_size, bool) or int(beam_size) != beam_size or not 1 <= beam_size <= _MAX_BEAM or beam_size > V:
        raise ValueError(f"decode_beam: beam_size must be an integer in [1, min({_MAX_BEAM}, vocabulary size {V})], "
                         f"got {beam_size}")
    stop = _decode_stop(V, end_token, pad_token, length_penalty)
    _check_envelope("decode_beam", h0, lstm, word2vec, proj)
    return _decode(N.DECODE_BEAM, h0, lstm, word2vec, proj, max_length, start_token, K=int(beam_size), stop=stop)


def decode_question(h0, lstm, word2vec, proj, max_length, deterministic, temperature, beam_size, end_token, length_penalty,
                    top_k=0, top_p=1.0):
    """QstEncoder.generate's decode policy: tokens (B, max_length) of the best beam (beam_size > 1), of the greedy decode
    (`deterministic` truthy) or of the sampled one (`deterministic is False`, truncated by top_k / top_p), all on the decode
    kernel.  None when the caller's stock loop decodes: sampled decoding outside the kernel's envelope, any other falsy
    `deterministic` (an overridden sample()), and greedy decoding outside the envelope once allow_stock_ops(True) lets it.
    Beam search, end-of-sequence decoding and top-k / nucleus truncation have no stock loop: outside the envelope they raise,
    even with allow_stock_ops(True)."""
    truncated = top_k != 0 or top_p != 1.0
    if truncated and deterministic is not False:
        raise ValueError(f"top_k = {top_k!r} / top_p = {top_p!r} need deterministic=False (they truncate sampling)")
    if beam_size > 1:
        if not deterministic:
            raise ValueError(f"beam_size = {beam_size} needs deterministic=True (beam search is not sampled)")
        return decode_beam(h0, lstm, word2vec, proj, max_length, beam_size, end_token=end_token,
                           length_penalty=length_penalty)[0][:, 0].contiguous()
    # end-of-sequence decoding: decode_greedy / decode_sample raise outside the envelope
    stop = end_token is not None
    if deterministic and (stop or decode_supported(h0, lstm, word2vec, proj)):
        return decode_greedy(h0, lstm, word2vec, proj, max_length, end_token=end_token)
    if deterministic is False and (stop or truncated or decode_supported(h0, lstm, word2vec, proj)):
        # words drawn from softmax(logits / temperature) by Gumbel-max on a seed from torch's generator
        return decode_sample(h0, lstm, word2vec, proj, max_length, temperature, end_token=end_token, top_k=top_k,
                             top_p=top_p)
    if deterministic:            # greedy decode outside the kernel's envelope: loud unless stock ops were opted in
        _stock(f"greedy decode with hidden size {h0.shape[1]}")
    return None
