"""ctypes binding of libpcdarts_sm100.so (C ABI: include/pcdarts_sm100.h).

The product path is CUDA only: `lib_for(tensor)` raises if the sm_100a library is missing or if a
tensor is not on a CUDA device.  There is no CPU fallback.  The single exception is the test-only
CPU *emulation* of the very same kernel sources (tests/emu, built with -DPCD_EMU): it is used by the
`-m "not gpu"` tests to check kernel index arithmetic against the oracle, and must be switched on
explicitly with `enable_emulation(path)` — nothing in the package ever does that.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libpcdarts_sm100.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)

i32, i64, f32, vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p


class CellShape(C.Structure):
    _fields_ = [("batch", i32), ("c_prev_prev", i32), ("c_prev", i32), ("channels", i32), ("height", i32),
                ("width", i32), ("reduction", i32), ("reduction_prev", i32), ("steps", i32), ("bn_eps", f32),
                ("bn_momentum", f32)]


class CellSizes(C.Structure):
    _fields_ = [(n, i64) for n in ("param_floats", "running_floats", "nbt_int64", "out_floats", "saved_floats",
                                   "stats_doubles", "bwd_work_floats", "bwd_stats_doubles")] + \
               [("out_height", i32), ("out_width", i32)]


class CellFwdArgs(C.Structure):
    _fields_ = [("shape", CellShape)] + [(n, vp) for n in ("s0", "s1", "weights", "weights2", "params", "running",
                                                           "nbt", "out", "saved", "stats")] + \
        [("skip_dw_outputs", i32)]


class CellBwdArgs(C.Structure):
    _fields_ = [("shape", CellShape)] + [(n, vp) for n in (
        "s0", "s1", "weights", "weights2", "params", "out", "saved", "stats", "grad_out", "grad_s0", "grad_s1",
        "grad_weights", "grad_weights2", "grad_params", "work", "bstats")] + \
        [("need_param_grads", i32), ("need_input_grads", i32)]


class MixedShape(C.Structure):
    _fields_ = [("batch", i32), ("channels", i32), ("height", i32), ("width", i32), ("stride", i32),
                ("bn_eps", f32), ("bn_momentum", f32)]


class MixedSizes(CellSizes):
    pass


class MixedFwdArgs(C.Structure):
    _fields_ = [("shape", MixedShape)] + [(n, vp) for n in ("x", "weights", "params", "running", "nbt", "out",
                                                            "saved", "stats")]


class MixedBwdArgs(C.Structure):
    _fields_ = [("shape", MixedShape)] + [(n, vp) for n in (
        "x", "weights", "params", "saved", "stats", "grad_out", "grad_x", "grad_weights", "grad_params", "work",
        "bstats")] + [("need_param_grads", i32)]


class StemArgs(C.Structure):
    _fields_ = [("batch", i32), ("c_out", i32), ("height", i32), ("width", i32), ("bn_eps", f32),
                ("bn_momentum", f32)] + [(n, vp) for n in ("x", "params", "running", "nbt", "out", "saved_z", "stats",
                                                           "grad_out", "grad_x", "grad_params", "bstats")]


class PreArgs(C.Structure):
    _fields_ = [("batch", i32), ("c_in", i32), ("c_out", i32), ("height", i32), ("width", i32), ("factorized", i32),
                ("bn_eps", f32), ("bn_momentum", f32)] + [(n, vp) for n in (
                    "x", "weight", "running", "nbt", "y", "stats", "grad_y", "grad_x", "grad_weight", "bstats")]


class CellEvalArgs(C.Structure):
    _fields_ = [("shape", CellShape)] + [(n, vp) for n in ("s0", "s1", "weights", "weights2", "params", "running", "out",
                                                           "work")]


class MixedEvalArgs(C.Structure):
    _fields_ = [("shape", MixedShape)] + [(n, vp) for n in ("x", "weights", "params", "running", "out")]


class PreEvalArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "c_in", "c_out", "height", "width", "factorized")] + [("bn_eps", f32)] + \
        [(n, vp) for n in ("x", "weight", "running", "gamma", "beta", "y")]


class StemEvalArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "c_out", "height", "width")] + [("bn_eps", f32)] + \
        [(n, vp) for n in ("x", "params", "running", "out")]


class DropPathArgs(C.Structure):
    _fields_ = [("batch", i32), ("sample_numel", i64)] + [(n, i32) for n in ("drop1", "drop2", "cell", "node", "sample_offset")] + \
        [(n, vp) for n in ("seed", "keep", "h1", "h2", "out", "grad_out", "grad_h1", "grad_h2")]


DECODE_GREEDY, DECODE_SAMPLED, DECODE_BEAM = 0, 1, 2         # pcd_decode_args.mode


class DecodeArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("mode", "T", "B", "K", "H", "E", "V", "start_token", "stop", "end_token", "pad_token")] + \
        [("length_penalty", f32), ("temperature", f32), ("row_offset", i32)] + \
        [(n, vp) for n in ("seed", "emb", "w_ih", "w_hh", "b_ih", "b_hh", "h0", "c0", "w_out", "b_out", "tokens", "scores",
                           "work")]


class DwConvArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "channels", "height", "width", "kernel", "stride", "padding", "dilation",
                                   "relu_input")] + [(n, vp) for n in ("x", "weight", "out", "grad_out", "grad_x", "grad_weight")]


class PwConvArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "c_in", "c_out", "hw")] + [("bn_eps", f32)] + \
        [(n, vp) for n in ("x", "weight", "z", "stats", "grad_y", "gamma", "bstats", "grad_x", "grad_weight")]


class BnArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "channels", "hw")] + [("bn_eps", f32), ("bn_momentum", f32)] + \
        [(n, vp) for n in ("z", "stats", "gamma", "beta", "running", "nbt", "y", "grad_y", "bstats")]


class PoolArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("batch", "channels", "height", "width", "stride", "is_max")] + \
        [(n, vp) for n in ("x", "y", "grad_y", "grad_x")]


EXPORTS = ("pcd_launch_count", "pcd_profile_enable", "pcd_profile_num_kernels", "pcd_profile_kernel_name",
           "pcd_profile_collect", "pcd_version", "pcd_strerror", "pcd_is_cuda_build", "pcd_last_cuda_error", "pcd_channel_shuffle",
           "pcd_cell_sizes_of", "pcd_cell_forward", "pcd_cell_backward", "pcd_mixedop_sizes_of",
           "pcd_mixedop_forward", "pcd_mixedop_backward", "pcd_stem_forward", "pcd_stem_backward",
           "pcd_preprocess_forward", "pcd_preprocess_backward", "pcd_adaptive_avgpool_forward", "pcd_adaptive_avgpool_backward",
           "pcd_gemm_tn_3xtf32", "pcd_set_overlap", "pcd_overlap_join", "pcd_ce_forward", "pcd_ce_backward",
           "pcd_transpose_pad", "pcd_lstm_pbuf_floats", "pcd_lstm_forward", "pcd_lstm_backward",
           "pcd_decode_work_floats", "pcd_decode", "pcd_flat_max_runs", "pcd_flat_axpy", "pcd_flat_scale",
           "pcd_flat_sumsq", "pcd_flat_sumsq_work", "pcd_flat_adam", "pcd_gemm_small_f32",
           "pcd_dwconv_forward", "pcd_dwconv_backward", "pcd_pwconv_forward", "pcd_pwconv_backward", "pcd_bn_apply",
           "pcd_bn_backward_stats", "pcd_pool3x3_forward", "pcd_pool3x3_backward", "pcd_channel_affine",
           "pcd_cell_eval_work_floats", "pcd_cell_forward_eval", "pcd_mixedop_forward_eval", "pcd_preprocess_forward_eval",
           "pcd_stem_forward_eval", "pcd_droppath_sum_forward", "pcd_droppath_sum_backward")


def _declare(lib):
    for name in EXPORTS:
        getattr(lib, name)          # AttributeError if a declared symbol is missing
    lib.pcd_strerror.restype = C.c_char_p
    lib.pcd_strerror.argtypes = [C.c_int]
    lib.pcd_last_cuda_error.restype = C.c_char_p
    lib.pcd_launch_count.restype = C.c_longlong
    lib.pcd_profile_kernel_name.restype = C.c_char_p
    lib.pcd_profile_kernel_name.argtypes = [C.c_int]
    lib.pcd_profile_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]
    lib.pcd_channel_shuffle.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.pcd_cell_sizes_of.argtypes = [C.POINTER(CellShape), C.POINTER(CellSizes)]
    lib.pcd_cell_forward.argtypes = [C.POINTER(CellFwdArgs), vp]
    lib.pcd_cell_backward.argtypes = [C.POINTER(CellBwdArgs), vp]
    lib.pcd_mixedop_sizes_of.argtypes = [C.POINTER(MixedShape), C.POINTER(MixedSizes)]
    lib.pcd_mixedop_forward.argtypes = [C.POINTER(MixedFwdArgs), vp]
    lib.pcd_mixedop_backward.argtypes = [C.POINTER(MixedBwdArgs), vp]
    lib.pcd_stem_forward.argtypes = [C.POINTER(StemArgs), vp]
    lib.pcd_stem_backward.argtypes = [C.POINTER(StemArgs), vp]
    lib.pcd_preprocess_forward.argtypes = [C.POINTER(PreArgs), vp]
    lib.pcd_preprocess_backward.argtypes = [C.POINTER(PreArgs), vp]
    lib.pcd_adaptive_avgpool_forward.argtypes = [vp, vp] + [C.c_int] * 6 + [vp]
    lib.pcd_adaptive_avgpool_backward.argtypes = [vp, vp] + [C.c_int] * 6 + [vp]
    lib.pcd_overlap_join.argtypes = [vp]
    lib.pcd_ce_forward.argtypes = [vp, C.c_longlong, C.c_int, C.c_int, vp, vp, vp, vp]
    lib.pcd_ce_backward.argtypes = [vp, C.c_longlong, C.c_int, C.c_int, vp, vp, vp, vp, vp]
    lib.pcd_lstm_pbuf_floats.restype = C.c_size_t
    lib.pcd_lstm_pbuf_floats.argtypes = [C.c_int, C.c_int]
    lib.pcd_lstm_forward.argtypes = [C.c_int, C.c_int, C.c_int] + [vp] * 8
    lib.pcd_lstm_backward.argtypes = [C.c_int, C.c_int, C.c_int] + [vp] * 12
    lib.pcd_decode_work_floats.restype = C.c_size_t
    lib.pcd_decode_work_floats.argtypes = [C.POINTER(DecodeArgs)]
    lib.pcd_decode.argtypes = [C.POINTER(DecodeArgs), vp]
    lib.pcd_transpose_pad.argtypes = [vp, C.c_longlong, C.c_int, C.c_int, vp, C.c_longlong, vp]
    lib.pcd_gemm_tn_3xtf32.argtypes = [vp, C.c_longlong, vp, C.c_longlong, vp, C.c_longlong, C.c_int, C.c_int, C.c_int, vp,
                                       C.c_int, vp]
    lib.pcd_gemm_small_f32.argtypes = [vp, C.c_longlong, C.c_longlong, vp, C.c_longlong, C.c_longlong, vp, C.c_longlong,
                                       C.c_int, C.c_int, C.c_int, vp, vp]
    ll_p, pp = C.POINTER(C.c_longlong), C.POINTER(vp)
    lib.pcd_flat_axpy.argtypes = [C.c_int, ll_p, pp, pp, vp, C.c_float, vp]
    lib.pcd_flat_scale.argtypes = [C.c_int, ll_p, pp, vp, vp]
    lib.pcd_flat_sumsq.argtypes = [C.c_int, ll_p, pp, vp, vp, vp]
    lib.pcd_flat_sumsq_work.restype = C.c_longlong
    lib.pcd_flat_sumsq_work.argtypes = [C.c_longlong]
    lib.pcd_flat_adam.argtypes = [C.c_int, ll_p, pp, pp, pp, pp] + [C.c_float] * 5 + [vp, vp]
    for fn, st in (("pcd_dwconv_forward", DwConvArgs), ("pcd_dwconv_backward", DwConvArgs), ("pcd_pwconv_forward", PwConvArgs),
                   ("pcd_pwconv_backward", PwConvArgs), ("pcd_bn_apply", BnArgs), ("pcd_bn_backward_stats", BnArgs),
                   ("pcd_pool3x3_forward", PoolArgs), ("pcd_pool3x3_backward", PoolArgs)):
        getattr(lib, fn).argtypes = [C.POINTER(st), vp]
    lib.pcd_channel_affine.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    lib.pcd_cell_eval_work_floats.argtypes = [C.POINTER(CellShape), C.POINTER(C.c_int64)]
    for fn, st in (("pcd_cell_forward_eval", CellEvalArgs), ("pcd_mixedop_forward_eval", MixedEvalArgs),
                   ("pcd_preprocess_forward_eval", PreEvalArgs), ("pcd_stem_forward_eval", StemEvalArgs)):
        getattr(lib, fn).argtypes = [C.POINTER(st), vp]
    for fn in ("pcd_droppath_sum_forward", "pcd_droppath_sum_backward"):
        getattr(lib, fn).argtypes = [C.POINTER(DropPathArgs), vp]
    return lib


_cuda_lib = None
_emu_lib = None


def load_cuda():
    """Load the sm_100a library (built in-tree by __graft_entry__.build()).  Fails loudly."""
    global _cuda_lib
    if _cuda_lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_NAME} not found at {LIB_PATH}: run `python -c 'import __graft_entry__ as g; "
                               "g.build()'` (nvcc, sm_100a).  There is no CPU fallback.")
        lib = _declare(C.CDLL(LIB_PATH))
        if lib.pcd_is_cuda_build() != 1:
            raise RuntimeError(f"{LIB_PATH} is not a CUDA build")
        _cuda_lib = lib
    return _cuda_lib


def enable_emulation(path):
    """TEST ONLY: load the CPU emulation build of the kernel sources (tests/emu)."""
    global _emu_lib
    lib = _declare(C.CDLL(path))
    if lib.pcd_is_cuda_build() != 0:
        raise RuntimeError("enable_emulation() expects the -DPCD_EMU build")
    _emu_lib = lib
    return lib


def lib_for(t: torch.Tensor):
    if t.is_cuda:
        return load_cuda()
    if _emu_lib is not None:
        return _emu_lib
    raise RuntimeError("pcdarts_sm100 kernels need CUDA tensors (no CPU fallback); got device " + str(t.device))


def stream_for(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream if t.is_cuda else None


def check(lib, rc, what):
    if rc != 0:
        msg = lib.pcd_strerror(rc).decode()
        detail = lib.pcd_last_cuda_error().decode()
        raise RuntimeError(f"{what}: {msg}" + (f" ({detail})" if detail else ""))


def ptr(t):
    return None if t is None else t.data_ptr()


def profile_collect(lib):
    """-> {kernel name: (total ms, launches)} for the launches recorded since pcd_profile_enable(1)."""
    n = 96
    ms = (C.c_double * n)()
    cnt = (C.c_longlong * n)()
    rc = lib.pcd_profile_collect(ms, cnt, n)
    if rc < 0:
        check(lib, rc, "pcd_profile_collect")
    return {lib.pcd_profile_kernel_name(i).decode(): (ms[i], cnt[i]) for i in range(lib.pcd_profile_num_kernels())
            if cnt[i]}
