"""ctypes binding of libfishdiff_b200.so (the C ABI declared in include/fishdiff_b200.h).

There is NO fallback: if the shared library is missing or a call fails this module raises.  PyTorch is used by the
callers only for device memory and streams; raw device pointers are passed down.
"""
from __future__ import annotations

import ctypes
import os
import threading
from ctypes import POINTER, c_char_p, c_float, c_int, c_longlong, c_size_t, c_ubyte, c_ulonglong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# FISHDIFF_B200_LIB: another build of the same C ABI (A/B runs of two kernel versions on one box); there is no non-CUDA fallback
LIB_PATH = os.environ.get("FISHDIFF_B200_LIB") or os.path.join(_HERE, "libfishdiff_b200.so")

PREC_F16, PREC_BF16 = 0, 1
PREC_SINGLE = 0x10   # or-ed into the prec of GEMM calls: one product over the hi planes
BACKEND_TC, BACKEND_SIMT = 0, 1
ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2
ABI_VERSION = 2


class NativeError(RuntimeError):
    pass


class ConvDesc(ctypes.Structure):
    """struct fd_conv_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("in_planes", c_void_p), ("w_planes", c_void_p), ("bias", c_void_p), ("addend", c_void_p),
        ("res_f32", c_void_p), ("res_planes", c_void_p), ("row_mask", c_void_p), ("out_f32", c_void_p),
        ("out_planes", c_void_p),
        ("B", c_int), ("T", c_int), ("Cin", c_int), ("N", c_int), ("ntaps", c_int), ("shifts", c_int * 16),
        ("w_inv_scale", c_float), ("post_scale", c_float), ("planes_scale", c_float), ("act_slope", c_float),
        ("out_accum", c_int), ("act", c_int), ("prec", c_int), ("backend", c_int),
    ]


class GemmDesc(ctypes.Structure):
    """struct fd_gemm_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("src", c_void_p * 2), ("src_C", c_int * 2), ("src_rs", c_longlong * 2), ("src_bs", c_longlong * 2),
        ("src_ps", c_longlong * 2), ("w", c_void_p), ("n_total", c_int), ("k_total", c_int), ("w_kshift", c_int),
        ("w_bstride_k", c_longlong), ("B", c_int), ("T", c_int), ("num_seg", c_int), ("seg_src", c_int * 16),
        ("seg_shift", c_int * 16), ("seg_coff", c_int * 16), ("seg_klen", c_int * 16),
        ("bias", c_void_p), ("addend", c_void_p), ("res_f32", c_void_p), ("res_planes", c_void_p),
        ("row_mask", c_void_p), ("out_f32", c_void_p), ("out_planes", c_void_p),
        ("w_inv_scale", c_float), ("res_scale", c_float), ("post_scale", c_float), ("planes_scale", c_float),
        ("act_slope", c_float), ("out_accum", c_int), ("act", c_int), ("prec", c_int), ("backend", c_int),
        ("bias_bstride", c_int),
        ("gate_y", c_void_p), ("gate_cs", c_void_p), ("gate_cs_edge", c_void_p), ("gate_cs_scale", c_float),
        ("gate_tile", c_int), ("gate_dil", c_int),
    ]


class ResPairDesc(ctypes.Structure):
    """struct fd_respair_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("in_planes", c_void_p), ("w1", c_void_p), ("w2", c_void_p), ("b1", c_void_p), ("b2", c_void_p),
        ("out_planes", c_void_p),
        ("B", c_int), ("T", c_int), ("C", c_int), ("k1", c_int), ("d1", c_int), ("k2", c_int),
        ("w1_inv_scale", c_float), ("w2_inv_scale", c_float), ("in_slope", c_float), ("out_slope", c_float),
        ("planes_scale", c_float), ("prec", c_int), ("kmask1", c_ulonglong), ("kmask2", c_ulonglong),
    ]


class WaveNetFwdDesc(ctypes.Structure):
    """struct fd_wavenet_fwd_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("x_planes", c_void_p), ("cond_planes", c_void_p), ("cond_term", c_void_p), ("steps", c_void_p),
        ("x_mask", c_void_p), ("out", c_void_p),
        ("w_in", c_void_p), ("b_in", c_void_p), ("w_in_inv", c_float),
        ("mlp_w0", c_void_p), ("mlp_b0", c_void_p), ("mlp_w1", c_void_p), ("mlp_b1", c_void_p),
        ("wd", c_void_p), ("bd", c_void_p), ("w1p_f32", c_void_p), ("bias_sum", c_void_p),
        ("w1", c_void_p), ("w1_lstride", c_longlong), ("w2", c_void_p), ("w2_lstride", c_longlong),
        ("b2", c_void_p), ("b2_lstride", c_longlong),
        ("w_skip", c_void_p), ("b_skip", c_void_p), ("w_skip_inv", c_float),
        ("w_out", c_void_p), ("b_out", c_void_p), ("w_out_inv", c_float),
        ("w1_inv", c_float * 64), ("w2_inv", c_float * 64), ("dilation", c_int * 64),
        ("xr", c_void_p), ("z", c_void_p), ("skip_planes", c_void_p), ("skip_f32", c_void_p),
        ("s", c_void_p), ("mlp_ws", c_void_p), ("gb", c_void_p), ("gb_ws", c_void_p),
        ("B", c_int), ("T", c_int), ("M", c_int), ("C", c_int), ("E", c_int), ("L", c_int), ("Bs", c_int),
        ("gate_tile", c_int), ("prec", c_int), ("backend", c_int),
    ]


class WaveNetBwdDesc(ctypes.Structure):
    """struct fd_wavenet_bwd_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("x_planes", c_void_p), ("y_planes", c_void_p), ("z_planes", c_void_p), ("cond_planes", c_void_p),
        ("dx_next", c_void_p), ("dskip", c_void_p), ("w2t", c_void_p), ("w1t", c_void_p), ("wct", c_void_p),
        ("w2t_inv", c_float), ("w1t_inv", c_float), ("wct_inv", c_float),
        ("dx_out", c_void_p), ("dx_f32", c_void_p), ("d_cond", c_void_p), ("gw1", c_void_p), ("gw2", c_void_p),
        ("cs_dy", c_void_p), ("cs_edge", c_void_p), ("cs_dx", c_void_p), ("dz", c_void_p), ("dy", c_void_p),
        ("part1", c_void_p), ("part2", c_void_p), ("splits1", c_int), ("splits2", c_int),
        ("B", c_int), ("T", c_int), ("C", c_int), ("E", c_int), ("dilation", c_int), ("gate_tile", c_int),
        ("inv_S", c_float), ("prec", c_int), ("backend", c_int),
    ]


class WgradDesc(ctypes.Structure):
    """struct fd_wgrad_desc (include/fishdiff_b200.h)."""
    _fields_ = [
        ("row_src", c_void_p * 2), ("row_C", c_int * 2), ("col_src", c_void_p * 2), ("col_C", c_int * 2),
        ("num_row_seg", c_int), ("row_seg_src", c_int * 2), ("row_seg_coff", c_int * 2), ("row_seg_width", c_int * 2),
        ("num_col_seg", c_int), ("col_seg_src", c_int * 8), ("col_seg_shift", c_int * 8), ("col_seg_coff", c_int * 8),
        ("col_seg_width", c_int * 8),
        ("B", c_int), ("T", c_int), ("splits", c_int), ("part", c_void_p), ("acc_scale", c_float), ("prec", c_int),
    ]


_SIGS = {
    "fd_gemm_cl_fwd": (c_int, [POINTER(GemmDesc), c_void_p]),
    "fd_wavenet_pack_layers": (c_int, [c_void_p] * 10 + [c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "fd_wgrad_cl": (c_int, [POINTER(WgradDesc), c_void_p]),
    "fd_wavenet_block_bwd": (c_int, [POINTER(WaveNetBwdDesc), c_void_p]),
    "fd_colsum_edges": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p]),
    "fd_wavenet_block_fwd_train": (c_int, [c_void_p] * 10 + [c_int, c_void_p, c_void_p, c_void_p, c_float] +
                                   [c_int] * 6 + [c_float, c_float, c_int, c_int, c_int, c_void_p]),
    "fd_wavenet_gate_bias_from_d": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, c_int, c_void_p]),
    "fd_fold_transpose": (c_int, [c_void_p] * 4 + [c_int, c_void_p] + [c_int] * 5 + [c_float, c_int, c_int, c_int,
                                                                                   c_int, c_int, c_void_p]),
    "fd_gate_bwd": (c_int, [c_void_p] * 3 + [c_longlong, c_int, c_int, c_int, c_void_p]),
    "fd_relu_bwd": (c_int, [c_void_p] * 3 + [c_longlong, c_float, c_int, c_void_p]),
    "fd_lrelu_bwd": (c_int, [c_void_p] * 5 + [c_longlong, c_float, c_float, c_int, c_void_p]),
    "fd_colsum": (c_int, [c_void_p] * 3 + [c_int, c_int, c_int, c_float, c_int, c_void_p]),
    "fd_reduce_batch": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_float, c_void_p]),
    "fd_abi_version": (c_int, []),
    "fd_last_error": (c_char_p, []),
    "fd_set_device": (None, [c_int]),
    "fd_launch_count": (c_longlong, []),
    "fd_tc_supported_linear": (c_int, [c_int, c_int, c_int]),
    "fd_prof_enable": (None, [c_int]),
    "fd_prof_collect": (c_int, [POINTER(ctypes.c_double), POINTER(c_longlong), c_int]),
    "fd_split_ncw": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fd_split_nwc": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p]),
    "fd_mrf_finish": (c_int, [POINTER(c_void_p), c_int, c_void_p, c_longlong, c_float, c_float, c_float, c_int, c_void_p]),
    "fd_transpose_nwc_to_ncw": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fd_transpose_ncw_to_nwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fd_pack_weight": (c_int, [c_void_p, c_void_p, c_longlong, c_float, c_int, c_void_p]),
    "fd_wavenet_step_mlp": (c_int, [c_void_p] * 7 + [c_int, c_int, c_void_p]),
    "fd_wavenet_gate_bias": (c_int, [c_void_p] * 9 + [c_int, c_int, c_int, c_int, c_void_p]),
    "fd_wavenet_block_fwd": (c_int, [c_void_p] * 8 + [c_int, c_void_p, c_void_p, c_void_p, c_float] + [c_int] * 6 +
                             [c_float, c_float, c_int, c_int, c_int, c_void_p]),
    "fd_wavenet_fwd": (c_int, [POINTER(WaveNetFwdDesc), c_void_p]),
    "fd_wavenet_cond_term": (c_int, [c_void_p, c_void_p, c_longlong, POINTER(c_float), c_void_p] + [c_int] * 7 +
                             [c_void_p]),
    "fd_conv_cl_fwd": (c_int, [POINTER(ConvDesc), c_void_p]),
    "fd_respair_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "fd_respair_fwd": (c_int, [POINTER(ResPairDesc), c_void_p]),
    "fd_ddpm_step": (c_int, [c_void_p] * 5 + [c_longlong] + [c_float] * 7 + [c_ulonglong, c_ulonglong, c_ulonglong, c_int,
                                                                               c_void_p]),
    "fd_lincomb": (c_int, [c_void_p, c_void_p, POINTER(c_void_p), POINTER(c_float), c_int, c_longlong, c_int, c_void_p]),
    "fd_affine_cl": (c_int, [c_void_p] * 4 + [c_int, c_longlong, c_int, c_void_p]),
    "fd_q_sample": (c_int, [c_void_p] * 5 + [c_int, c_longlong, c_void_p]),
    "fd_randn": (c_int, [c_void_p, c_longlong, c_ulonglong, c_ulonglong, c_ulonglong, c_void_p]),
    "fd_sinegen_ws_bytes": (c_size_t, [c_int, c_longlong]),
    "fd_sinegen_fwd": (c_int, [c_void_p] * 7 + [c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_ulonglong,
                                                c_void_p]),
    "fd_source_conv_fwd": (c_int, [c_void_p] * 4 + [c_int, c_longlong, c_int, c_int, c_int, c_int, c_void_p]),
    "fd_conv_post_fwd": (c_int, [c_void_p] * 4 + [c_int, c_longlong, c_int, c_int, c_int, c_void_p]),
    "fd_reflect_pad_split": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_int, c_int, c_void_p]),
    "fd_stft_mag_fwd": (c_int, [c_void_p] * 3 + [c_int, c_longlong, c_int, c_int, c_int, c_int, c_float, c_float, c_int,
                                                 c_int, c_void_p]),
    "fd_stft_mag_eps_fwd": (c_int, [c_void_p] * 3 + [c_int, c_longlong, c_int, c_int, c_int, c_int, c_float, c_float, c_float,
                                                     c_int, c_int, c_void_p]),
    "fd_log_clamp": (c_int, [c_void_p, c_void_p, c_longlong, c_float, c_float, c_void_p]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def lib():
    """Load the shared library (once).  Raises NativeError if it is missing -- there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  fish_diffusion_b200 has no CPU or PyTorch fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if l.fd_abi_version() != ABI_VERSION:
            raise NativeError(f"ABI mismatch: library {l.fd_abi_version()} != binding {ABI_VERSION}")
        _lib = l
    return _lib


def last_error() -> str:
    return (lib().fd_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str):
    if rc != 0:
        raise NativeError(f"{what} failed (rc={rc}): {last_error()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be contiguous."""
    if t is None:
        return None
    assert t.is_contiguous(), "native kernels need contiguous tensors"
    return t.data_ptr()


_tls = threading.local()


def stream_ptr(device=None):
    """Current torch stream of `device` as a raw cudaStream_t.  Also tells the library which device the following
    call targets (fd_set_device, thread-local on both sides), so tensors on a non-current device work."""
    if device is None or getattr(device, "index", None) is None:
        idx = torch.cuda.current_device()
    else:
        idx = device.index
    if getattr(_tls, "dev", None) != idx:
        lib().fd_set_device(idx)
        _tls.dev = idx
    return torch.cuda.current_stream(idx).cuda_stream


def require_cuda(t, name="tensor"):
    if not t.is_cuda:
        raise NativeError(f"{name} is on {t.device}: fish_diffusion_b200 runs on CUDA (sm_100a) only, there is no CPU path")


def launch_count() -> int:
    return int(lib().fd_launch_count())


def prec_code(precision: str) -> int:
    """Storage precision of the split planes: 'f16' / 'bf16' (an 'x1' suffix only changes the GEMM arithmetic)."""
    p = precision.lower()
    if p.endswith("x1"):
        p = p[:-2]
    if p in ("f16", "fp16", "half"):
        return PREC_F16
    if p in ("bf16", "bfloat16"):
        return PREC_BF16
    raise ValueError(f"unknown precision {precision!r} (use 'f16', 'bf16', 'f16x1' or 'bf16x1')")


def mma_code(precision: str) -> int:
    """`prec` argument of the GEMM entry points: 'f16' / 'bf16' multiply the split planes with three tensor-core
    products (22- / 16-bit operand mantissas); 'f16x1' / 'bf16x1' multiply the hi planes only (one product: plain
    half-precision operands, fp32 accumulation -- the arithmetic class of torch autocast / TF32 convolutions)."""
    return prec_code(precision) | (PREC_SINGLE if precision.lower().endswith("x1") else 0)


def backend_code(backend: str) -> int:
    b = backend.lower()
    if b in ("tc", "tcgen05"):
        return BACKEND_TC
    if b in ("simt", "fp32"):
        return BACKEND_SIMT
    raise ValueError(f"unknown backend {backend!r} (use 'tc' or 'simt')")


# ------------------------------------------------------------------------------------------------ helpers
def pow2_scale(w: torch.Tensor, target: float = 64.0) -> float:
    """Power-of-two prescale s such that max|w*s| lies in [target/2, target): keeps the fp16 lo-plane of the
    packed weights out of the subnormal range; undone exactly by the kernel's acc_scale = 1/s."""
    m = float(w.detach().abs().max())
    if m == 0.0 or not (m == m):
        return 1.0
    import math
    return float(2.0 ** math.floor(math.log2(target / m)))


def pack_weight(w2d: torch.Tensor, prec: int, scale: float) -> torch.Tensor:
    """fp32 [N, K] (device) -> split planes uint16 [2, N, K]."""
    w2d = w2d.detach().to(torch.float32).contiguous()
    require_cuda(w2d, "weight")
    out = torch.empty((2,) + tuple(w2d.shape), dtype=torch.int16, device=w2d.device)
    check(lib().fd_pack_weight(ptr(w2d), ptr(out), w2d.numel(), scale, prec, stream_ptr(w2d.device)), "fd_pack_weight")
    return out


def split_nwc(x: torch.Tensor, prec: int, mask=None, scale: float = 1.0, out=None) -> torch.Tensor:
    """fp32 [B,T,C] -> planes [2,B,T,C]."""
    B, T, C = x.shape
    x = x.contiguous()
    if out is None:
        out = torch.empty((2, B, T, C), dtype=torch.int16, device=x.device)
    check(lib().fd_split_nwc(ptr(x), ptr(mask), ptr(out), B, T, C, scale, prec, stream_ptr(x.device)), "fd_split_nwc")
    return out


def split_ncw(x: torch.Tensor, prec: int, mask=None, out=None) -> torch.Tensor:
    """fp32 [B,C,T] -> planes [2,B,T,C]."""
    B, C, T = x.shape
    x = x.contiguous()
    if out is None:
        out = torch.empty((2, B, T, C), dtype=torch.int16, device=x.device)
    check(lib().fd_split_ncw(ptr(x), ptr(mask), ptr(out), B, C, T, prec, stream_ptr(x.device)), "fd_split_ncw")
    return out


def conv_cl(in_planes, w_planes, B, T, Cin, N, shifts, *, bias=None, addend=None, res_f32=None, res_planes=None,
            row_mask=None, out_f32=None, out_planes=None, w_inv_scale=1.0, post_scale=1.0, planes_scale=1.0,
            act=ACT_NONE, act_slope=0.0, out_accum=False, prec=PREC_F16, backend=BACKEND_TC):
    d = ConvDesc()
    d.in_planes, d.w_planes = ptr(in_planes), ptr(w_planes)
    d.bias, d.addend, d.res_f32, d.res_planes = ptr(bias), ptr(addend), ptr(res_f32), ptr(res_planes)
    d.row_mask, d.out_f32, d.out_planes = ptr(row_mask), ptr(out_f32), ptr(out_planes)
    d.B, d.T, d.Cin, d.N, d.ntaps = B, T, Cin, N, len(shifts)
    for i, s in enumerate(shifts):
        d.shifts[i] = int(s)
    d.w_inv_scale, d.post_scale, d.planes_scale, d.act_slope = w_inv_scale, post_scale, planes_scale, act_slope
    d.out_accum, d.act, d.prec, d.backend = int(out_accum), act, prec, backend
    check(lib().fd_conv_cl_fwd(ctypes.byref(d), stream_ptr(in_planes.device)), "fd_conv_cl_fwd")


def respair_supported(C: int, k1: int, d1: int, k2: int) -> bool:
    return bool(lib().fd_respair_supported(C, k1, d1, k2))


def respair(in_planes, w1, w2, b1, b2, B, T, C, k1, d1, k2, *, out_planes, w1_inv_scale=1.0, w2_inv_scale=1.0,
            in_slope=0.1, out_slope=0.1, planes_scale=1.0, prec=PREC_F16, kmask1=0, kmask2=0):
    """Fused ResBlock1 pair x' = x + c2(lrelu(c1(lrelu(x)))) on planes of lrelu(x) -> planes of lrelu(x') (fd_respair_fwd).
    kmask1 / kmask2: block-sparsity hints (bit tap*(C/16)+s <=> input channels [16s,16s+16) of that tap are non-zero)."""
    d = ResPairDesc()
    d.in_planes, d.w1, d.w2, d.b1, d.b2 = ptr(in_planes), ptr(w1), ptr(w2), ptr(b1), ptr(b2)
    d.out_planes = ptr(out_planes)
    d.B, d.T, d.C, d.k1, d.d1, d.k2 = B, T, C, k1, d1, k2
    d.w1_inv_scale, d.w2_inv_scale = w1_inv_scale, w2_inv_scale
    d.in_slope, d.out_slope, d.planes_scale = in_slope, out_slope, planes_scale
    d.prec = prec
    d.kmask1, d.kmask2 = int(kmask1), int(kmask2)
    check(lib().fd_respair_fwd(ctypes.byref(d), stream_ptr(in_planes.device)), "fd_respair_fwd")


def mrf_finish(ins, out, *, in_slope=0.1, scale=1.0, out_slope=0.1, prec=PREC_F16):
    """out planes = split(lrelu(sum_i invlrelu(ins[i]) * scale, out_slope))  (fd_mrf_finish)."""
    arr = (c_void_p * len(ins))(*[ptr(t) for t in ins])
    check(lib().fd_mrf_finish(arr, len(ins), ptr(out), out.numel() // 2, in_slope, scale, out_slope, prec,
                              stream_ptr(out.device)), "fd_mrf_finish")


PROF_KINDS = {0: "linear/tc", 1: "linear/simt", 2: "gate/tc", 3: "gate/simt", 4: "res_skip/tc", 5: "res_skip/simt",
              6: "mag/tc", 7: "mag/simt", 8: "gate_bwd/tc", 12: "respair/128", 13: "respair/64", 14: "respair/32",
              15: "respair/16"}


_prof_on = False


def prof_enable(on: bool):
    """Per-launch CUDA-event timing of the tap-GEMM kernels.  While it is on, CUDA-graph replay of the denoiser is
    disabled (events recorded inside a captured graph cannot be timed)."""
    global _prof_on
    _prof_on = bool(on)
    lib().fd_prof_enable(1 if on else 0)


def prof_is_on() -> bool:
    return _prof_on


def prof_collect():
    """-> {kind name: (total ms, launches)} of every tap-GEMM launch since prof_enable(True)."""
    n = max(PROF_KINDS) + 1
    ms = (ctypes.c_double * n)()
    cnt = (c_longlong * n)()
    rc = lib().fd_prof_collect(ms, cnt, n)
    if rc < 0:
        raise NativeError(f"fd_prof_collect failed: {last_error()}")
    return {PROF_KINDS.get(k, f"kind{k}"): (float(ms[k]), int(cnt[k])) for k in range(n) if cnt[k]}, bool(rc)


def tc_supported_linear(n_total: int, k_seg: int, num_seg: int) -> bool:
    return bool(lib().fd_tc_supported_linear(n_total, k_seg, num_seg))


def gemm_cl(src0, C0, w_planes, n_total, k_total, B, T, segs, *, src1=None, C1=0, strides0=None, strides1=None,
            w_kshift=0, w_bstride_k=0, bias=None, bias_per_item=False, addend=None, res_f32=None, res_planes=None, res_scale=1.0,
            row_mask=None, out_f32=None, out_planes=None, w_inv_scale=1.0, post_scale=1.0, planes_scale=1.0,
            act=ACT_NONE, act_slope=0.0, out_accum=False, prec=PREC_F16, backend=BACKEND_TC):
    """General linear tap-GEMM (fd_gemm_cl_fwd).  segs = [(src_index, shift, c_off, k_len), ...];
    stridesX = (row_stride, batch_stride, plane_stride) in elements or None for the canonical [2][B][T][C]."""
    d = GemmDesc()
    d.src[0], d.src_C[0] = ptr(src0), C0
    d.src[1], d.src_C[1] = ptr(src1), C1
    for i, st in enumerate((strides0, strides1)):
        if st is not None:
            d.src_rs[i], d.src_bs[i], d.src_ps[i] = st
    d.w, d.n_total, d.k_total, d.w_kshift, d.w_bstride_k = ptr(w_planes), n_total, k_total, int(w_kshift), int(w_bstride_k)
    d.B, d.T, d.num_seg = B, T, len(segs)
    for j, (si, sh, co, kl) in enumerate(segs):
        d.seg_src[j], d.seg_shift[j], d.seg_coff[j], d.seg_klen[j] = si, sh, co, kl
    d.bias, d.addend, d.res_f32, d.res_planes = ptr(bias), ptr(addend), ptr(res_f32), ptr(res_planes)
    d.row_mask, d.out_f32, d.out_planes = ptr(row_mask), ptr(out_f32), ptr(out_planes)
    d.w_inv_scale, d.res_scale, d.post_scale = w_inv_scale, res_scale, post_scale
    d.planes_scale, d.act_slope = planes_scale, act_slope
    d.out_accum, d.act, d.prec, d.backend = int(out_accum), act, prec, backend
    d.bias_bstride = n_total if bias_per_item else 0
    check(lib().fd_gemm_cl_fwd(ctypes.byref(d), stream_ptr(src0.device)), "fd_gemm_cl_fwd")


def wgrad_supported(row_segs, col_segs) -> bool:
    """Shapes the direct (MN-major tcgen05) weight-gradient kernel takes: every segment a multiple of 64 channels."""
    return (1 <= len(row_segs) <= 2 and 1 <= len(col_segs) <= 8 and all(w % 64 == 0 and w > 0 for *_, w in row_segs)
            and all(w % 64 == 0 and w > 0 for *_, w in col_segs))


def wgrad_splits(R, Cc, B, T):
    """Item splits of a direct weight-gradient GEMM (see wgrad_cl): enough work units for ~2 waves of the 148 SMs, at
    most one partial per item, and one TMEM accumulation run kept to <= ~2048 time steps."""
    bn = 256 if Cc % 256 == 0 else 128 if Cc % 128 == 0 else 64
    tiles = ((R + 127) // 128) * (Cc // bn)
    splits = max(1, min(B, -(-296 // tiles)))
    splits = max(splits, -(-B // max(1, 2048 // T)))
    ips = -(-B // splits)
    return -(-B // ips)


def wgrad_cl(row_srcs, col_srcs, row_segs, col_segs, B, T, *, scale=1.0, prec=PREC_F16, splits=None, out=None):
    """sum_{b,t} ROW[b,t,r] * COL[b,t+shift,c] * scale -> fp32 [R, Cc]  (fd_wgrad_cl + fd_reduce_batch).
    row_srcs / col_srcs: lists of 1..2 plane tensors [2,B,T,C]; row_segs = [(src, c_off, width)],
    col_segs = [(src, shift, c_off, width)]."""
    import torch
    d = WgradDesc()
    for i, t in enumerate(row_srcs):
        assert t.dim() == 4 and t.shape[0] == 2 and t.shape[1] == B and t.shape[2] == T
        d.row_src[i], d.row_C[i] = ptr(t), t.shape[3]
    for i, t in enumerate(col_srcs):
        assert t.dim() == 4 and t.shape[0] == 2 and t.shape[1] == B and t.shape[2] == T
        d.col_src[i], d.col_C[i] = ptr(t), t.shape[3]
    d.num_row_seg, d.num_col_seg = len(row_segs), len(col_segs)
    R = Cc = 0
    for j, (si, co, w) in enumerate(row_segs):
        d.row_seg_src[j], d.row_seg_coff[j], d.row_seg_width[j] = si, co, w
        R += w
    for j, (si, sh, co, w) in enumerate(col_segs):
        d.col_seg_src[j], d.col_seg_shift[j], d.col_seg_coff[j], d.col_seg_width[j] = si, sh, co, w
        Cc += w
    if splits is None:      # enough work units for ~2 waves of the 148 SMs, at most one partial per item
        bn = 256 if Cc % 256 == 0 else 128 if Cc % 128 == 0 else 64
        tiles = ((R + 127) // 128) * (Cc // bn)
        splits = max(1, min(B, -(-296 // tiles)))
        # tensor-core fp32 accumulation truncates: keep one TMEM accumulation run to <= ~2048 time steps (measured:
        # 7000-step runs put ~2e-4 of relative noise on the conditioner / input-projection weight gradients)
        splits = max(splits, -(-B // max(1, 2048 // T)))
    ips = -(-B // splits)
    splits = -(-B // ips)
    dev = row_srcs[0].device
    part = torch.empty((splits, R, Cc), dtype=torch.float32, device=dev)
    d.B, d.T, d.splits, d.part, d.acc_scale, d.prec = B, T, splits, ptr(part), 1.0, prec
    st = stream_ptr(dev)
    check(lib().fd_wgrad_cl(ctypes.byref(d), st), "fd_wgrad_cl")
    if out is None:
        out = torch.empty((R, Cc), dtype=torch.float32, device=dev)
    assert tuple(out.shape) == (R, Cc) and out.dtype == torch.float32
    check(lib().fd_reduce_batch(ptr(part), ptr(out), splits, R * Cc, float(scale), st), "fd_reduce_batch")
    return out


def lrelu_bwd(grad, act_planes, slope, *, addend=None, out_f32=None, out_planes=None, scale=1.0, prec=PREC_F16):
    """v = grad * (act > 0 ? 1 : slope) * scale + addend -> out_f32 and / or out_planes (fd_lrelu_bwd).
    grad / addend / out_f32: fp32 tensors of n elements, act_planes / out_planes: split planes [2, n]."""
    n = grad.numel()
    assert act_planes.numel() == 2 * n and (out_f32 is not None or out_planes is not None)
    check(lib().fd_lrelu_bwd(ptr(grad), ptr(act_planes), ptr(addend), ptr(out_f32), ptr(out_planes), n, float(slope),
                             float(scale), prec, stream_ptr(grad.device)), "fd_lrelu_bwd")


def colsum(planes, B, T, Nn, *, scale=1.0, prec=PREC_F16):
    """sum over (b, t) of planes [2,B,T,Nn] * scale -> fp32 [Nn]  (fd_colsum per item, then a sum over the items)."""
    out = torch.zeros((B, Nn), dtype=torch.float32, device=planes.device)
    check(lib().fd_colsum(ptr(planes), None, ptr(out), B, T, Nn, float(scale), prec, stream_ptr(planes.device)),
          "fd_colsum")
    return out.sum(0)
